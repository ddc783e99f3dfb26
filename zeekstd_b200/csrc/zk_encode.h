// zk_encode.h -- host-visible interface of the batched compress path (zk_encode.cu).
#pragma once
#include "zk_common.cuh"

struct ZkEncodeWs {                    // HBM scratch owned by a zk_ctx slot, grown on demand
    void* buf = nullptr; size_t cap = 0;
    uint32_t* h_sizes = nullptr; size_t cap_frames = 0;   // pinned: per-frame compressed sizes
    int sm_count = 0;
    unsigned long long launches = 0;
    uint32_t pending_frames = 0;
    bool attr_set = false, attr_set_wide = false, attr_set_wide_ldm = false;
    const uint8_t* prefix = nullptr; uint32_t prefix_len = 0;   // device pointer: raw-content prefix for the NEXT enqueue (one-shot)
    const uint32_t* ldm_tab = nullptr; uint32_t ldm_log = 0;   // index of that prefix (zk_ldm_index_build), one-shot with it
    uint32_t win_log = 0;             // window log the frame headers announce at least (ZK_C_WINDOW_LOG; 0 = the level's own)
    int prio = 0;                     // CUDA stream priority of the side stream (matches the slot's stream)
    bool no_side = false;             // host pipelines: concurrency comes from the other sub-batches; every extra stream costs a hardware queue
    cudaStream_t side = nullptr; cudaEvent_t ev_a = nullptr, ev_b = nullptr, ev_c = nullptr;   // K-C2s runs beside K-C2l
    ZkProf prof;
};

// Compress n bytes at d_src into ceil(n/frame_size) frames written back to back at d_dst.
// c_sizes (host, n_frames entries) receives each frame's compressed size.  Synchronous on `stream`.
int zk_encode_batch(ZkEncodeWs* ws, cudaStream_t stream, const uint8_t* d_src, size_t n, uint32_t frame_size, int level,
                    int checksum, uint8_t* d_dst, size_t dst_cap, uint32_t* c_sizes, uint32_t n_frames, size_t* dst_len);
int zk_encode_enqueue(ZkEncodeWs* ws, cudaStream_t stream, const uint8_t* d_src, size_t n, uint32_t frame_size, int level,
                      int checksum, uint8_t* d_dst, size_t dst_cap, uint32_t n_frames);
int zk_encode_collect(ZkEncodeWs* ws, cudaStream_t stream, uint32_t* c_sizes, size_t* dst_len);
void zk_encode_ws_free(ZkEncodeWs* ws);
size_t zk_encode_bound(size_t n, uint32_t frame_size);
// window log a level's frames announce without ZK_C_WINDOW_LOG (17, or 18 for the wide-history tier)
uint32_t zk_encode_level_window_log(int level);
// long-distance matching: slot count (log2) of the index over `span` bytes of prefix, and the index itself -- every
// ZK_LDM_STRIDE-th position of the last min(win, prefix_len) bytes, hashed on 8 bytes, the highest position per slot (+1; 0 = empty)
#define ZK_LDM_STRIDE 8u
uint32_t zk_ldm_index_log(size_t span);
int zk_ldm_index_build(cudaStream_t stream, const uint8_t* d_prefix, uint32_t prefix_len, uint32_t win, uint32_t* d_tab, uint32_t log);
