// zk_decode.h -- host-visible interface of the batched decode path (zk_decode.cu).
#pragma once
#include "zk_common.cuh"
#include <string.h>

struct ZkDecodeArgs {                 // kernel parameter block (by value)
    const uint8_t* comp;              // compressed bytes; entry e occupies [c_off[e], c_off[e+1])
    const unsigned long long* c_off;  // device, n_entries + 1
    const unsigned long long* d_off;  // device, n_entries + 1; entry e decodes to dst + d_off[e]
    uint8_t* dst;
    uint32_t n_entries;
    ZkBlock* blocks; ZkEntry* entries; ZkCounters* counters; uint32_t* work_counter;
    uint8_t* lit; uint32_t* seq_lit_end; uint32_t* seq_out_end; uint32_t* seq_off;
    uint32_t* huf_list; uint32_t* seq_list;   // compacted indices of blocks with Huffman literals / with sequences
    unsigned long long cap_blocks, cap_lit, cap_seq;
    unsigned long long* trace;        // debug: per-chunk clock64 stamps of entry 0 (env ZK_EXEC_TRACE), else nullptr
    const uint8_t* prefix; uint32_t prefix_len;   // raw-content prefix of every zstd frame (Decoder::decompress_with_prefix, decode.rs:211-214, 246-255); device pointer or nullptr
    const uint32_t* d_need;           // per entry: only this many leading bytes are wanted (range reads); nullptr = everything
    unsigned long long win_max;       // frames announcing a larger window are refused (window_tooLarge)
};

struct ZkDecodeWs {                   // HBM scratch owned by a zk_ctx, grown on demand, reused across batches
    ZkBlock* blocks = nullptr; size_t cap_blocks = 0;
    ZkEntry* entries = nullptr; size_t cap_entries = 0;
    ZkCounters* counters = nullptr;
    uint8_t* lit = nullptr; size_t cap_lit = 0;
    uint32_t* seq_lit_end = nullptr; uint32_t* seq_out_end = nullptr; uint32_t* seq_off = nullptr; size_t cap_seq = 0;
    uint64_t* c_off = nullptr; uint64_t* d_off = nullptr;
    const uint32_t* need = nullptr;   // host array for the NEXT enqueue (one-shot): leading bytes wanted per entry, see ZkDecodeArgs::d_need
    uint32_t* d_need = nullptr; uint32_t* h_need = nullptr;
    const uint8_t* prefix = nullptr; uint32_t prefix_len = 0;   // device pointer for the NEXT enqueue (one-shot, like `need`)
    uint32_t* huf_list = nullptr; uint32_t* seq_list = nullptr;
    bool attr_set = false; uint32_t ring_override = 0;
    bool seq_v1 = false, attr_set2 = false; uint32_t seq2_ctas = 6;   // ZK_SEQ_V1=1: the first-generation FSE kernel; persistent CTAs per SM of the second
    bool exec_v2 = false;             // ZK_EXEC_V2=1: the in-order exec kernel (zk_exec2_kernel) for every batch, not only in prefix mode
    uint32_t huf_pad = 0;             // extra dynamic smem per Huffman CTA: fewer resident CTAs -> more L1 for the streams (tuning)
    unsigned long long* trace = nullptr;
    int share = 1;                    // how many batches share the GPU concurrently (host pipeline depth)
    int prio = 0;                     // CUDA stream priority of the side stream (matches the slot's stream)
    uint32_t seq_ctas = 4, huf_ctas = 8;   // persistent CTAs per SM of the two entropy kernels (tuning: ZK_SEQ_CTAS / ZK_HUF_CTAS)
    bool no_side = false;             // host pipelines: concurrency comes from the other sub-batches; every extra stream costs a hardware queue
    cudaStream_t up = nullptr, down = nullptr;      // host pipelines: dedicated upload / download streams (not owned); nullptr = everything on `stream`
    cudaEvent_t ev_up = nullptr, ev_done = nullptr, ev_down = nullptr;
    cudaStream_t side = nullptr; cudaEvent_t ev_scan = nullptr, ev_huf = nullptr;   // Huffman kernel runs beside the FSE kernel
    ZkEntry* h_entries = nullptr; ZkCounters* h_counters = nullptr; uint64_t* h_off = nullptr;   // pinned
    size_t want_blocks = 0, want_lit = 0, want_seq = 0;   // exact needs reported by a batch that overflowed
    uint32_t pending_n = 0;
    int sm_count = 0;
    unsigned long long win_max = (1ull << 27) + 1;   // ZK_D_WINDOW_LOG_MAX of the owning context; default: a default ZSTD_DCtx's limit
    unsigned long long launches = 0;  // kernels launched so far (bench.py's gpu_launches)
    ZkProf prof;
};

// Decode n seek-table entries.  d_comp / d_dst are device pointers (16-byte aligned, 16 readable bytes of
// padding after the last byte); c_off / d_off are HOST arrays of n+1 cumulative offsets relative to those
// pointers (seek_table.rs:97-101).  status_out[n] (host, optional) receives 0 or -(zstd code) per entry.
// Returns 0, or the first non-zero entry status, or -(code) for a launch/allocation failure.
// Synchronous with respect to `stream` on return.
int zk_decode_batch(ZkDecodeWs* ws, cudaStream_t stream, const uint8_t* d_comp, const uint64_t* c_off, const uint64_t* d_off,
                    uint32_t n, uint8_t* d_dst, int verify_checksum, int32_t* status_out, int exec_warps);
int zk_decode_enqueue(ZkDecodeWs* ws, cudaStream_t stream, const uint8_t* d_comp, const uint64_t* c_off, const uint64_t* d_off,
                      uint32_t n, uint8_t* d_dst, int verify_checksum, int exec_warps);
int zk_decode_collect(ZkDecodeWs* ws, cudaStream_t stream, int32_t* status_out);
void zk_decode_ws_free(ZkDecodeWs* ws);
