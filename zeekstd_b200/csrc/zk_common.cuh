// zk_common.cuh -- shared device/host definitions for the zeekstd_b200 codec kernels.
//
// The codec arithmetic that the reference reaches through zstd-safe -> libzstd
// (lib/src/encode.rs:341-345,444-448; lib/src/decode.rs:243-245) is implemented here from the
// Zstandard format (RFC 8878; restated in SURVEY.md Appendix A) as CUDA for sm_100a.
#pragma once

#ifdef ZK_EMUL
// tests/emul/cuda_emul.h is force-included by the emulation test build (g++), see tests/emul/.
#define ZK_LAUNCH(kernel, grid, block, smem, stream, ...) \
    emu::launch(dim3(grid), dim3(block), (smem), [=]() { kernel(__VA_ARGS__); })
#define ZK_DYN_SMEM(name) uint8_t* name = emu::g_dyn_smem
#define ZK_SPIN() emu::yield()
#else
#include <cuda_runtime.h>
#define ZK_LAUNCH(kernel, grid, block, smem, stream, ...) kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__)
#define ZK_DYN_SMEM(name) extern __shared__ __align__(128) uint8_t name[]
#define ZK_SPIN() __nanosleep(32)
#endif

#include <stdint.h>
#include <stddef.h>

// internal status of a failed CUDA runtime call / kernel (the C ABI's ZK_ERR_CUDA); the text is kept per thread
#define ZK_INT_CUDA (-1007)
void zk_note_cuda_error(const char* what, int code);

// Optional per-kernel timing with CUDA events on the launching stream (bench.py's roofline numbers).
// slots: 0 scan, 1 seq, 2 huf, 3 exec, 4 xxh64(dec), 5 match, 6 entropy-enc, 7 frame assembly
#define ZK_PROF_SLOTS 8
struct ZkProf {
    bool enabled = false;
    cudaEvent_t ev[ZK_PROF_SLOTS][2] = {};
    bool used[ZK_PROF_SLOTS] = {};
    float ms[ZK_PROF_SLOTS] = {};
    unsigned count[ZK_PROF_SLOTS] = {};
    void begin(int slot, cudaStream_t st) {
        if (!enabled) return;
        if (!ev[slot][0]) { cudaEventCreate(&ev[slot][0]); cudaEventCreate(&ev[slot][1]); }
        cudaEventRecord(ev[slot][0], st);
    }
    void end(int slot, cudaStream_t st) { if (!enabled) return; cudaEventRecord(ev[slot][1], st); used[slot] = true; }
    void harvest() {                        // call after the stream(s) were synchronised
        if (!enabled) return;
        for (int i = 0; i < ZK_PROF_SLOTS; i++) if (used[i]) {
            float t = 0.f; cudaEventSynchronize(ev[i][1]); cudaEventElapsedTime(&t, ev[i][0], ev[i][1]);
            ms[i] += t; count[i]++; used[i] = false;
        }
    }
    void destroy() { for (int i = 0; i < ZK_PROF_SLOTS; i++) for (int j = 0; j < 2; j++) if (ev[i][j]) { cudaEventDestroy(ev[i][j]); ev[i][j] = nullptr; } }
};

// libzstd's numeric error codes (ZSTD_ErrorCode); the C ABI reports -(code) so that the
// reference's Error::is_zstd()/get_error_name() semantics carry over (error.rs:40-45, 101-113).
enum ZkZstdCode : int {
    ZKZ_OK = 0,
    ZKZ_GENERIC = 1,
    ZKZ_PREFIX_UNKNOWN = 10,
    ZKZ_VERSION_UNSUPPORTED = 12,
    ZKZ_FRAMEPARAM_UNSUPPORTED = 14,
    ZKZ_WINDOW_TOO_LARGE = 16,
    ZKZ_CORRUPTION = 20,
    ZKZ_CHECKSUM_WRONG = 22,
    ZKZ_DICT_CORRUPTED = 30,         // what libzstd reports for Treeless literals before any Huffman table (litEntropy == 0)
    ZKZ_DICT_WRONG = 32,
    ZKZ_PARAM_UNSUPPORTED = 40,
    ZKZ_PARAM_OUT_OF_BOUND = 42,
    ZKZ_MEMORY_ALLOCATION = 64,
    ZKZ_DST_TOO_SMALL = 70,
    ZKZ_SRC_SIZE_WRONG = 72,
};

#define ZK_BLOCK_MAX (1u << 17)          // Block_Maximum_Size, A.2
#define ZK_MAGIC 0xFD2FB528u
#define ZK_SKIPPABLE_MASK 0xFFFFFFF0u
#define ZK_SKIPPABLE_MAGIC 0x184D2A50u

// -------------------------------------------------------------------------------------------
// Work descriptors living in HBM scratch (one batch = up to 2^31 output bytes).
// -------------------------------------------------------------------------------------------
struct ZkBlock {                 // one zstd block of one seek-table entry
    uint32_t src;                // offset of the block content, relative to the entry's first compressed byte
    uint32_t size;               // Block_Size (content bytes; for RLE the regenerated size)
    uint32_t entry;              // seek-table entry this block belongs to
    uint8_t type;                // 0 Raw, 1 RLE, 2 Compressed
    uint8_t flags;               // ZKB_*
    uint8_t lit_kind;            // (entropy kernel) 0 raw-in-place, 1 rle, 2 scratch
    uint8_t lit_byte;            // rle literal byte
    uint32_t lit_base;           // literal scratch offset (bytes)            [scan kernel]
    uint32_t seq_base;           // sequence scratch offset (entries)         [scan kernel]
    uint32_t nseq;               //                                             [scan kernel]
    uint32_t lit_size;           // regenerated literal bytes                  [scan kernel]
    uint32_t lit_src;            // raw literals: offset rel. to entry start   [entropy kernel]
    uint32_t regen;              // regenerated block size                     [entropy kernel]
    int32_t status;              // sequences: 0 or -(zstd code)               [seq kernel]
    int32_t lit_status;          // literals:  0 or -(zstd code)               [huf kernel]
    int32_t huf_ref;             // block index whose Huffman tree a Treeless block reuses (-1 none)
    int32_t ll_ref, of_ref, ml_ref;   // block index defining the table a Repeat mode reuses (-1 none)
    uint32_t rep_out[3];         // rep-offset state after this block: concrete value, or ZK_SYM|slot<<28|delta
    uint64_t fcs;                // last block of a zstd frame: Frame_Content_Size if ZKB_HAS_FCS
    uint32_t hash_start;         // last block: start (rel. to entry output) and length of the zstd frame's content
    uint32_t hash_len;
    uint32_t bmax;               // Block_Maximum_Size of the block's zstd frame: min(Window_Size, 128 KiB)   [scan kernel]
};
#define ZKB_FIRST 1u             // first block of a zstd frame: resets repeat offsets / entropy tables
#define ZKB_LAST 2u              // Last_Block
#define ZKB_HAS_CSUM 4u          // 4-byte content checksum follows the last block
#define ZKB_HAS_FCS 8u

// symbolic repeat offset: "incoming repeat slot s (0..2) minus delta" (delta in 0..2^20)
#define ZK_SYM 0x80000000u
#define ZK_SYM_MAKE(slot, delta) (ZK_SYM | ((uint32_t)(slot) << 28) | (uint32_t)(delta))
#define ZK_SYM_SLOT(v) (((v) >> 28) & 3u)
#define ZK_SYM_DELTA(v) ((v) & 0x0FFFFFFFu)

struct ZkEntry {                 // one seek-table entry (one "frame" of the seekable format)
    uint32_t first_block;
    uint32_t n_blocks;
    int32_t status;              // 0, -(zstd code), or ZK_ST_RETRY
    uint32_t produced;           // bytes written (exec kernel)
};
#define ZK_ST_RETRY 0x7FFFFFFF   // scratch capacity exceeded: host grows the workspace and re-runs

struct ZkCounters {
    unsigned long long n_blocks, n_lit, n_seq;   // exact needs (accumulated even when over capacity)
    uint32_t overflow;
    uint32_t n_errors;
    uint32_t n_huf_blocks, n_seq_blocks;         // lengths of huf_list / seq_list
};

// -------------------------------------------------------------------------------------------
// helpers
// -------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t zk_ld_u8(const uint8_t* p) { return *p; }
__device__ __forceinline__ uint32_t zk_ld_le16(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }
__device__ __forceinline__ uint32_t zk_ld_le24(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16); }
__device__ __forceinline__ uint32_t zk_ld_le32(const uint8_t* p) {
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}
__device__ __forceinline__ int zk_highbit(uint32_t v) { return 31 - __clz((int)v); }   // v != 0

// -------------------------------------------------------------------------------------------
// Backward bitstream reader (A.7) over global memory.
//
// The stream is consumed from its last byte towards its first; `buf` holds the next unread bits
// left-aligned (MSB = the bit just below the cursor), so reading n bits is one shift.  Memory is
// fetched as aligned 32-bit words in descending order, always one word ahead (`nxt`), and the
// cache line after that is prefetched, so a refill never waits for DRAM even though every lane of
// a warp streams through a different region.  Reads below the first byte return zero bits (legal
// only at the very end of Huffman streams / FSE-compressed weights, A.4) and drive `left` negative,
// which callers test to detect corruption.
// -------------------------------------------------------------------------------------------
__device__ __forceinline__ void zk_prefetch_l1(const void* p) {
#ifndef ZK_EMUL
    asm volatile("prefetch.global.L1 [%0];" :: "l"(p));
#else
    (void)p;
#endif
}

struct ZkBackBits {
    const uint32_t* w;          // 4-byte aligned base (stream address rounded down)
    unsigned long long buf;     // unread bits, left-aligned
    uint32_t nxt;               // prefetched word w[j]
    uint32_t lowmask;           // clears the bits of word 0 that precede the stream
    int j;                      // index of `nxt`
    int cnt;                    // valid bits in buf
    int bp;                     // stream bits not yet consumed (negative after an over-read)

    // The word fetched ahead is kept RAW in `nxt` and only masked when it is merged into buf, so the load
    // has a whole refill interval to complete (masking at load time made every refill wait for memory).
    __device__ __forceinline__ uint32_t fetch(int idx) const { return w[idx < 0 ? 0 : idx]; }
    __device__ __forceinline__ uint32_t cooked(uint32_t raw, int idx) const {
        return idx < 0 ? 0u : (idx == 0 ? (raw & lowmask) : raw);
    }
    // returns false when the stream is malformed (empty or no end marker)
    __device__ __forceinline__ bool init(const uint8_t* p, uint32_t n) {
        if (n == 0) return false;
        uint32_t last = p[n - 1];
        if (last == 0) return false;
        uintptr_t addr = (uintptr_t)p;
        w = (const uint32_t*)(addr & ~(uintptr_t)3);
        int shift = (int)(addr & 3) * 8;
        lowmask = 0xFFFFFFFFu << shift;
        bp = (int)(n - 1) * 8 + zk_highbit(last);
        int A = bp + shift;                         // bits between the aligned base and the cursor
        if (A == 0) { buf = 0; cnt = 0; j = -1; nxt = 0; return true; }
        int t = (A - 1) >> 5, r = A - (t << 5);     // top word and how many of its low bits are payload
        buf = (unsigned long long)cooked(fetch(t), t) << (64 - r);
        cnt = r; j = t - 1; nxt = fetch(j);
        if (j >= 32) zk_prefetch_l1(w + j - 32);
        return true;
    }
    // afterwards at least 33 bits are available in buf (zero bits once the stream is exhausted)
    __device__ __forceinline__ void refill() {
        if (cnt <= 32) {
            buf |= (unsigned long long)cooked(nxt, j) << (32 - cnt);
            cnt += 32; j--;
            nxt = fetch(j);
            if ((j & 31) == 31 && j >= 32) zk_prefetch_l1(w + j - 32);     // one line ahead of the word just fetched
        }
    }
    // n in [0,32], n <= cnt
    __device__ __forceinline__ uint32_t peek(int n) const { return (uint32_t)((buf >> 1) >> (63 - n)); }
    __device__ __forceinline__ void skip(int n) { buf <<= n; cnt -= n; bp -= n; }
    __device__ __forceinline__ uint32_t read(int n) { uint32_t v = peek(n); skip(n); return v; }
};

// Forward little-endian bit reader for FSE table descriptions (A.6); byte-wise, bounds checked.
struct ZkFwdBits {
    const uint8_t* p; uint32_t n; uint32_t bit;
    __device__ __forceinline__ uint32_t peek(int nb) const {
        uint32_t byte = bit >> 3, sh = bit & 7;
        unsigned long long v = 0;
#pragma unroll
        for (int i = 0; i < 4; i++) { uint32_t b = byte + i < n ? p[byte + i] : 0u; v |= (unsigned long long)b << (8 * i); }
        return (uint32_t)(v >> sh) & ((1u << nb) - 1u);
    }
};

// -------------------------------------------------------------------------------------------
// FSE tables (A.6): symbol code -> value baseline / extra bits
// -------------------------------------------------------------------------------------------
__constant__ uint32_t ZK_LL_BASE[36] = {0,1,2,3,4,5,6,7,8,9,10,11,12,13,14,15,16,18,20,22,24,28,32,40,48,64,128,256,512,1024,2048,4096,8192,16384,32768,65536};
__constant__ uint8_t ZK_LL_BITS[36] = {0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,1,1,1,1,2,2,3,3,4,6,7,8,9,10,11,12,13,14,15,16};
__constant__ uint32_t ZK_ML_BASE[53] = {3,4,5,6,7,8,9,10,11,12,13,14,15,16,17,18,19,20,21,22,23,24,25,26,27,28,29,30,31,32,33,34,35,37,39,41,43,47,51,59,67,83,99,131,259,515,1027,2051,4099,8195,16387,32771,65539};
__constant__ uint8_t ZK_ML_BITS[53] = {0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,1,1,1,1,2,2,3,3,4,4,5,7,8,9,10,11,12,13,14,15,16};
__constant__ int16_t ZK_LL_DEFAULT[36] = {4,3,2,2,2,2,2,2,2,2,2,2,2,1,1,1,2,2,2,2,2,2,2,2,2,3,2,1,1,1,1,1,-1,-1,-1,-1};
__constant__ int16_t ZK_ML_DEFAULT[53] = {1,4,3,2,2,2,2,2,2,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,-1,-1,-1,-1,-1,-1,-1};
__constant__ int16_t ZK_OF_DEFAULT[29] = {1,1,1,1,1,1,2,2,2,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,-1,-1,-1,-1,-1};

// Parse an FSE normalized-count header.  Returns bytes consumed (>0) or 0 on corruption.
// counts[] gets nsym entries (-1 = "less than one").
__device__ inline uint32_t zk_fse_read_ncount(const uint8_t* p, uint32_t n, int max_log, int max_sym,
                                              int16_t* counts, int* nsym_out, int* log_out) {
    if (n < 1) return 0;
    ZkFwdBits f = { p, n, 0 };
    int al = 5 + (int)f.peek(4); f.bit += 4;
    if (al > max_log) return 0;
    int remaining = (1 << al) + 1, threshold = 1 << al, nb = al + 1, s = 0;
    while (remaining > 1 && s <= max_sym) {
        int mx = 2 * threshold - 1 - remaining, v;
        int lo = (int)f.peek(nb - 1);
        if (lo < mx) { v = lo; f.bit += nb - 1; }
        else { v = (int)f.peek(nb); if (v >= threshold) v -= mx; f.bit += nb; }
        int c = v - 1;
        remaining -= c < 0 ? -c : c;
        counts[s++] = (int16_t)c;
        if (c == 0) {
            for (;;) {
                int r = (int)f.peek(2); f.bit += 2;
                for (int q = 0; q < r && s <= max_sym; q++) counts[s++] = 0;
                if (r != 3) break;
                if ((f.bit >> 3) > n) return 0;
            }
        }
        if (remaining < 1) return 0;
        while (remaining < threshold) { nb--; threshold >>= 1; }
        if ((f.bit >> 3) > n) return 0;
    }
    if (remaining != 1 || s > max_sym + 1) return 0;
    uint32_t used = (f.bit + 7) >> 3;
    if (used > n) return 0;
    *nsym_out = s; *log_out = al;
    return used;
}

// -------------------------------------------------------------------------------------------
// Event = an mbarrier with an arrival count of one: every arrive completes a phase, so "something changed" wakes
// whoever sleeps in try_wait on it (hardware sleep: a waiting warp issues nothing, and wakes ~60 cycles after the
// arrive -- B300_MICROARCH.md, mbarrier).  A waiter re-checks its own condition after every wake-up; it first learns the
// parity of the running phase (test_wait), THEN checks the condition, then sleeps on that parity, so a change between the
// check and the sleep ends the sleep at once.  Two changes in that window would be missed; the time hint bounds that.
// -------------------------------------------------------------------------------------------
#ifndef ZK_EMUL
__device__ __forceinline__ uint32_t zk_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void zk_event_init(unsigned long long* bar) { asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(zk_smem_u32(bar)) : "memory"); }
__device__ __forceinline__ void zk_event_signal(unsigned long long* bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(zk_smem_u32(bar)) : "memory"); }
__device__ __forceinline__ uint32_t zk_event_parity(unsigned long long* bar) {      // parity of the phase that is running now
    uint32_t done0;
    asm volatile("{ .reg .pred p; mbarrier.test_wait.parity.shared::cta.b64 p, [%1], 0; selp.u32 %0, 1, 0, p; }" : "=r"(done0) : "r"(zk_smem_u32(bar)) : "memory");
    return done0;                                                                     // phase of parity 0 complete <=> parity 1 is running
}
__device__ __forceinline__ bool zk_event_sleep(unsigned long long* bar, uint32_t parity, uint32_t hint_ns) {   // true: that phase has completed
    uint32_t ok;
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3; selp.u32 %0, 1, 0, p; }"
                 : "=r"(ok) : "r"(zk_smem_u32(bar)), "r"(parity), "r"(hint_ns) : "memory");
    return ok != 0;
}
#else
__device__ __forceinline__ void zk_event_init(unsigned long long* bar) { *bar = 0; }
__device__ __forceinline__ void zk_event_signal(unsigned long long* bar) { *(volatile unsigned long long*)bar = *bar + 1; }
__device__ __forceinline__ uint32_t zk_event_parity(unsigned long long* bar) { return (uint32_t)(*(volatile unsigned long long*)bar & 1); }
__device__ __forceinline__ bool zk_event_sleep(unsigned long long* bar, uint32_t parity, uint32_t) { emu::yield(); return (uint32_t)(*(volatile unsigned long long*)bar & 1) != parity; }
#endif

// -------------------------------------------------------------------------------------------
// TMA bulk copy global -> shared (cp.async.bulk, SASS UBLKCP) completing on an mbarrier: one thread arms the barrier with
// the byte count and issues the copy; the data lands without passing through registers and whoever needs it waits on the
// barrier's phase.  Addresses and sizes are multiples of 16 bytes.
// -------------------------------------------------------------------------------------------
#ifndef ZK_EMUL
__device__ __forceinline__ void zk_mbar_init(unsigned long long* bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(zk_smem_u32(bar)), "r"(count) : "memory"); }
__device__ __forceinline__ void zk_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, unsigned long long* bar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(zk_smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(zk_smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(zk_smem_u32(bar)) : "memory");
}
// returns false if the phase did not complete within ~2^22 polls (seconds): a lost copy must become an error, not a hung GPU
__device__ __forceinline__ bool zk_mbar_wait(unsigned long long* bar, uint32_t parity) {
    uint32_t ok = 0;
    for (uint32_t spin = 0; !ok && spin < (1u << 22); spin++)
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }" : "=r"(ok) : "r"(zk_smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
#else
// emulation: the barrier word counts completed phases; a copy completes at once
__device__ __forceinline__ void zk_mbar_init(unsigned long long* bar, uint32_t) { *bar = 0; }
__device__ __forceinline__ void zk_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, unsigned long long* bar) { memcpy(dst_smem, src_gmem, bytes); *(volatile unsigned long long*)bar = *bar + 1; }
__device__ __forceinline__ bool zk_mbar_wait(unsigned long long* bar, uint32_t parity) { while ((uint32_t)(*(volatile unsigned long long*)bar & 1) == parity) emu::yield(); return true; }
#endif

// -------------------------------------------------------------------------------------------
// XXH64 (A.8), seed 0, of p[0..len) by one warp; the result is valid in every lane.
//
// The four accumulators are four serial chains (acc = rotl(acc + in * P2, 31) * P1 per 32-byte stripe), so one frame
// cannot go faster than about 40 cycles per stripe whatever the width of the machine.  What CAN be taken off that chain
// is everything else: the warp loads 256 bytes (8 stripes) with one coalesced 8-byte load per lane, four iterations
// ahead, every lane multiplies its own word by P2, and the chain (replicated in all lanes: lane L carries accumulator
// L & 3) picks the products up by shuffle.  The first version (lanes 0..3 each loading their own words, unaligned, one
// stripe at a time) ran at 330 cycles per stripe: 21.7 ms per GiB of 2 MiB frames against 28 ms for the whole LZ77
// execution -- it was the most expensive kernel of a checksummed decode.
// -------------------------------------------------------------------------------------------
#define ZK_P1 0x9E3779B185EBCA87ull
#define ZK_P2 0xC2B2AE3D27D4EB4Full
#define ZK_P3 0x165667B19E3779F9ull
#define ZK_P4 0x85EBCA77C2B2AE63ull
#define ZK_P5 0x27D4EB2F165667C5ull
__device__ __forceinline__ unsigned long long zk_rotl64(unsigned long long x, int r) { return (x << r) | (x >> (64 - r)); }
__device__ __forceinline__ unsigned long long zk_xx_round(unsigned long long acc, unsigned long long in) { return zk_rotl64(acc + in * ZK_P2, 31) * ZK_P1; }
__device__ __forceinline__ unsigned long long zk_xx_merge(unsigned long long h, unsigned long long v) { return (h ^ zk_xx_round(0, v)) * ZK_P1 + ZK_P4; }
__device__ __forceinline__ unsigned long long zk_ld_u64_unaligned(const uint8_t* p) {
    uintptr_t a = (uintptr_t)p; uint32_t mis = (uint32_t)(a & 7);
    const unsigned long long* q = (const unsigned long long*)(a - mis);
    if (mis == 0) return q[0];
    return (q[0] >> (mis * 8)) | (q[1] << (64 - mis * 8));
}

static __device__ __noinline__ unsigned long long zk_warp_xxh64(const uint8_t* p, uint32_t len, int lane) {
    unsigned long long h;
    uint32_t done = 0;
    if (len >= 32) {
        const int al = lane & 3;
        unsigned long long acc = al == 0 ? ZK_P1 + ZK_P2 : (al == 1 ? ZK_P2 : (al == 2 ? 0ull : 0ull - ZK_P1));
        const uint32_t iters = len >> 8;                                 // 256 bytes = 8 stripes per iteration
        if (iters) {
            const uint32_t mis = (uint32_t)((uintptr_t)p & 7), sh = mis * 8;
            const unsigned long long* qa = (const unsigned long long*)(p - mis);       // aligned view; word i covers bytes [8i - mis, 8i + 8 - mis)
            // with mis != 0 the last word read lies up to 7 bytes past p + 256 * iters: inside the buffer whenever len has a tail,
            // inside the 16 bytes of padding every codec buffer carries otherwise
            unsigned long long w0 = qa[lane], w1 = 0, w2 = 0, w3 = 0;
            if (iters > 1) w1 = qa[32 + lane];
            if (iters > 2) w2 = qa[64 + lane];
            if (iters > 3) w3 = qa[96 + lane];
            for (uint32_t it = 0; it < iters; it++) {
                unsigned long long wn = 0;                                // four iterations ahead
                if (it + 4 < iters) wn = qa[(size_t)(it + 4) * 32 + lane];
                unsigned long long v = w0;
                if (mis) {
                    unsigned long long up = __shfl_down_sync(0xFFFFFFFFu, w0, 1);
                    unsigned long long nx = it + 1 < iters ? __shfl_sync(0xFFFFFFFFu, w1, 0) : qa[(size_t)(it + 1) * 32];
                    if (lane == 31) up = nx;
                    v = (w0 >> sh) | (up << (64 - sh));
                }
                const unsigned long long prod = v * ZK_P2;
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const unsigned long long x = __shfl_sync(0xFFFFFFFFu, prod, k * 4 + al);
                    acc = zk_rotl64(acc + x, 31) * ZK_P1;
                }
                w0 = w1; w1 = w2; w2 = w3; w3 = wn;
            }
            done = iters << 8;
        }
        for (uint32_t i = done; i + 32 <= len; i += 32) acc = zk_xx_round(acc, zk_ld_u64_unaligned(p + i + al * 8));   // < 8 stripes
        done += ((len - done) >> 5) << 5;
        const unsigned long long v1 = __shfl_sync(0xFFFFFFFFu, acc, 0), v2 = __shfl_sync(0xFFFFFFFFu, acc, 1),
                                 v3 = __shfl_sync(0xFFFFFFFFu, acc, 2), v4 = __shfl_sync(0xFFFFFFFFu, acc, 3);
        h = zk_rotl64(v1, 1) + zk_rotl64(v2, 7) + zk_rotl64(v3, 12) + zk_rotl64(v4, 18);
        h = zk_xx_merge(h, v1); h = zk_xx_merge(h, v2); h = zk_xx_merge(h, v3); h = zk_xx_merge(h, v4);
    } else h = ZK_P5;
    h += (unsigned long long)len;
    const uint8_t* q = p + done; uint32_t rem = len - done;
    while (rem >= 8) { h ^= zk_xx_round(0, zk_ld_u64_unaligned(q)); h = zk_rotl64(h, 27) * ZK_P1 + ZK_P4; q += 8; rem -= 8; }
    if (rem >= 4) { h ^= (unsigned long long)zk_ld_le32(q) * ZK_P1; h = zk_rotl64(h, 23) * ZK_P2 + ZK_P3; q += 4; rem -= 4; }
    while (rem) { h ^= (unsigned long long)(*q) * ZK_P5; h = zk_rotl64(h, 11) * ZK_P1; q++; rem--; }
    h ^= h >> 33; h *= ZK_P2; h ^= h >> 29; h *= ZK_P3; h ^= h >> 32;
    return h;
}
