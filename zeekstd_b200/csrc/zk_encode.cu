// zk_encode.cu -- batched Zstandard frame compression for sm_100a.
//
// Replaces the reference's compression calls into libzstd,
//   lib/src/encode.rs:341-345   cctx.compress_stream2(out, in, ZSTD_e_continue)
//   lib/src/encode.rs:444-448   cctx.compress_stream2(out, empty, ZSTD_e_end)
// with kernels over a whole batch of independent frames (seekable_format.md:23-29); every frame is cut
// into zstd blocks of ZKC_BLOCK bytes and every block is one unit of work:
//
//   K-C1 zk_match_kernel<HLOG> one warp / block : LZ77 match finding (hash table in shared memory), greedy parse resolved
//                                               with ballots, repeat-offset codes, sequences + literals written per window
//   K-C2s zk_seq_enc_kernel  one warp / block : FSE sequences (three lanes run the state chains, 32 lanes pack the bits)
//   K-C2l zk_lit_enc_kernel  one warp / block : Huffman literals (tree build, FSE-coded weights, 4 streams packed by warp scan)
//   K-C2f zk_block_finish_kernel              : joins the two sections of a block (coded on two streams), Raw fallback, header
//   K-C3 zk_frame_{hash,size,scan,gather}_kernel : optional XXH64, frame sizes, offsets, frame headers + block gather
//
// Output is a standard Zstandard frame per seek-table entry (RFC 8878; SURVEY.md Appendix A), decodable
// by libzstd; the compressed bytes are NOT meant to equal libzstd's.
#include "zk_encode.h"
#include <string.h>

#define ZKC_BLOCK 32768u                 // zstd block size used by this encoder (<= Block_Maximum_Size)
#define ZKC_HLOG_FAST 11                 // hash table per warp: 2048 x u16 at level 1 (40 warps / SM hide the two dependent loads per window),
#define ZKC_HLOG 12                      // 4096 x u16 from level 2 on (24 warps / SM, 0.3-3 % better ratio)
#define ZKC_MINMATCH 5
#define ZKC_MAXSEQ (ZKC_BLOCK / 4 + 8)   // every sequence covers at least 4 bytes (repeat matches may be 4 long); multiple of 8 for 16-byte chunked loads
#define ZKC_SLOT (ZKC_BLOCK + 64u)       // per-block staging slot for the compressed block
#define ZKC_FRAME_HDR 10u                // magic + FHD + window descriptor + 4-byte FCS

struct ZkcBlock {                        // per-block record in HBM
    uint32_t nseq, nlit;                 // K-C1
    uint32_t seq_hdr, seq_bits;          // K-C2s: bytes of the sequence-section header / bitstream (seq_hdr == 0: not encodable)
    uint32_t lit_bytes, last_flag;       // K-C2l: bytes staged so far (3-byte header gap + literals section; 0 = send the block Raw)
    uint32_t csize;                      // K-C2f: size of the staged block incl. its 3-byte header
    uint32_t out_off;                    // K-C3: offset of the block inside its frame
};
#define ZKC_SEQSEC 16384u                // per-block scratch for the sequence section: [0,256) header, [256,..) bitstream
#define ZKC_SEQHDR 256u

struct ZkEncodeArgs {
    const uint8_t* src; size_t n; uint32_t frame_size; uint32_t n_frames; uint32_t blocks_per_frame; uint32_t n_blocks;
    int level, checksum;
    ZkcBlock* blocks;
    uint16_t* seq_ll; uint16_t* seq_ml; uint32_t* seq_off;      // ZKC_MAXSEQ per block
    uint8_t* lits;                                              // ZKC_BLOCK per block
    uint8_t* stage;                                             // ZKC_SLOT per block
    uint8_t* seqsec;                                            // ZKC_SEQSEC per block
    uint32_t* frame_csize; unsigned long long* frame_off; uint32_t* frame_hash;
    uint8_t* dst; size_t dst_cap; unsigned long long* total; uint32_t* error;
    // raw-content prefix (RawEncoder::compress_with_prefix, encode.rs:311-338: re-applied at the start of EVERY frame): the last
    // ptail <= ZKC_BLOCK bytes of it are staged in front of a copy of each frame's first block, so that block's match finder sees
    // one contiguous history and needs no second pointer
    const uint8_t* prefix; uint32_t prefix_len, ptail; uint8_t* pstage;
    // long-distance matching (the LDM flavour of K-C1 only): index of the prefix (zk_ldm_index_kernel) with 2^ldm_log slots, and the
    // announced window -- no offset may exceed it
    const uint32_t* ldm_tab; uint32_t ldm_log, ldm_win;
};
#define ZKC_PSLOT (2u * ZKC_BLOCK + 64u)   // per-frame staging slot: [prefix tail | first block]

__device__ __forceinline__ void zkc_block_range(const ZkEncodeArgs& a, uint32_t b, size_t& lo, size_t& hi, size_t& fstart) {
    uint32_t f = b / a.blocks_per_frame, k = b % a.blocks_per_frame;
    fstart = (size_t)f * a.frame_size;
    size_t fend = fstart + a.frame_size < a.n ? fstart + a.frame_size : a.n;
    lo = fstart + (size_t)k * ZKC_BLOCK; if (lo > fend) lo = fend;
    hi = lo + ZKC_BLOCK < fend ? lo + ZKC_BLOCK : fend;
}

// unaligned 8-byte little-endian load from global memory
__device__ __forceinline__ unsigned long long zkc_ld8(const uint8_t* p) {
    uintptr_t a = (uintptr_t)p; uint32_t mis = (uint32_t)(a & 3);
    const uint32_t* q = (const uint32_t*)(a - mis);
    uint32_t w0 = q[0], w1 = q[1];
    if (mis == 0) return (unsigned long long)w0 | ((unsigned long long)w1 << 32);
    uint32_t w2 = q[2], sh = mis * 8;
    return (unsigned long long)__funnelshift_r(w0, w1, sh) | ((unsigned long long)__funnelshift_r(w1, w2, sh) << 32);
}
template <int HLOG>
__device__ __forceinline__ uint32_t zkc_hash5(unsigned long long v) {
    return (uint32_t)(((v << 24) * 889523592379ull) >> (64 - HLOG));
}
template <int HLOG>
__device__ __forceinline__ uint32_t zkc_hash8(unsigned long long v) {
    return (uint32_t)((v * 0xCF1BBCDCB7A56463ull) >> (64 - HLOG));
}
__device__ __forceinline__ uint32_t zkc_ldm_hash(unsigned long long v, uint32_t log) {
    return (uint32_t)((v * 0x9E3779B97F4A7C15ull) >> (64 - log));
}

// =============================================================================================
// K-C1: match finding.  One warp per block; lane i examines position ip + i * stride.
//
// Every position is a 32-bit offset from `base` (the start of the searchable history, < 64 KiB before the end of the
// block), so the u16 hash table stores positions directly.  A window is always full (32 valid lanes): the last < 40
// bytes of a block are left as literals.  Matches are only taken from stride-1 windows -- when a wider window (used
// after runs of misses on incompressible data) sees a candidate, the window is simply redone at stride 1.  That makes
// literal emission a per-window register operation: a byte that no selected match covers is written from the lane that
// already holds it (ballot + popc rank), and sequences are staged one per lane and stored 32 at a time.
// =============================================================================================
#define ZKC_C1_WARPS 4

// prefix mode: [tail of the prefix | first block of frame f] -> pstage slot f (one CTA per frame)
__global__ void __launch_bounds__(256) zk_prefix_stage_kernel(ZkEncodeArgs a) {
    const uint32_t f = blockIdx.x;
    const size_t fstart = (size_t)f * a.frame_size;
    const size_t fend = fstart + a.frame_size < a.n ? fstart + a.frame_size : a.n;
    const uint32_t len = (uint32_t)(fend - fstart < ZKC_BLOCK ? fend - fstart : ZKC_BLOCK);
    uint8_t* d = a.pstage + (size_t)f * ZKC_PSLOT;
    const uint8_t* pt = a.prefix + (a.prefix_len - a.ptail);
    for (uint32_t i = threadIdx.x; i < a.ptail; i += blockDim.x) d[i] = pt[i];
    for (uint32_t i = threadIdx.x; i < len; i += blockDim.x) d[a.ptail + i] = a.src[fstart + i];
    for (uint32_t i = threadIdx.x; i < 64; i += blockDim.x) d[a.ptail + len + i] = 0;
}

// DFAST (level >= 4): a second table indexed by a hash of EIGHT bytes is probed first -- its candidates are long matches by
// construction, the 5-byte table catches the rest (the idea of zstd's double-fast strategy); two tables of 2^HLOG entries per warp.
// LDM (long-distance matching, prefix calls with ZK_C_ENABLE_LONG_DISTANCE_MATCHING): every lane also probes the HBM index of the prefix
// with the 8 bytes it holds; a verified hit becomes a match whose source lies anywhere in the prefix the window reaches.
template <int HLOG, int NW, bool DFAST, bool LDM = false>
__global__ void __launch_bounds__(NW * 32) zk_match_kernel(ZkEncodeArgs a) {
    __shared__ uint16_t tables[NW][(DFAST ? 2 : 1) << HLOG];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t b = blockIdx.x * NW + warp;
    if (b >= a.n_blocks) return;
    uint16_t* table = tables[warp];
    uint16_t* tableL = table + (1 << HLOG);                // only touched when DFAST
#define ZKM_POS_T uint16_t
#define ZKM_HIST_BYTES ZKC_BLOCK
#include "zk_match_body.inc"
#undef ZKM_POS_T
#undef ZKM_HIST_BYTES
}

// Wide-history tier (level >= ZKC_WIDE_LEVEL): the same body with a history of ZKC_WIDE_HIST blocks of the frame instead of one -- the frame
// header then announces a 256 KiB window (zk_frame_window_kernel) --, 32-bit positions, and one table of 2^HLOG entries in DYNAMIC shared memory
// (128 KiB at HLOG 15: one warp-CTA per SM).  Every block still finds its matches alone and pre-inserts its whole history first, so a block costs
// several times a level-3 block: a tier for ratio (2.50 on the reference's corpus against 2.40 in a 64 KiB window), not for speed.
#define ZKC_WIDE_LEVEL 13
#define ZKC_WIDE_HIST 7
#define ZKC_WIDE_HLOG 15
template <int HLOG, bool LDM = false>
__global__ void __launch_bounds__(32) zk_match_wide_kernel(ZkEncodeArgs a) {
    ZK_DYN_SMEM(wide_tab);
    constexpr bool DFAST = false;
    const int warp = 0, lane = threadIdx.x & 31;
    const uint32_t b = blockIdx.x;
    if (b >= a.n_blocks) return;
    uint32_t* table = (uint32_t*)wide_tab;
    uint32_t* tableL = table;                               // never touched (DFAST is false)
    (void)warp; (void)tableL;
#define ZKM_POS_T uint32_t
#define ZKM_HIST_BYTES ((size_t)ZKC_WIDE_HIST * ZKC_BLOCK)
#include "zk_match_body.inc"
#undef ZKM_POS_T
#undef ZKM_HIST_BYTES
}

// =============================================================================================
// K-C2: entropy coding.  One warp per block.
// =============================================================================================
__constant__ uint8_t ZKC_LL_CODE[64] = {0,1,2,3,4,5,6,7,8,9,10,11,12,13,14,15,16,16,17,17,18,18,19,19,20,20,20,20,21,21,21,21,
                                        22,22,22,22,22,22,22,22,23,23,23,23,23,23,23,23,24,24,24,24,24,24,24,24,24,24,24,24,24,24,24,24};
__constant__ uint8_t ZKC_ML_CODE[128] = {0,1,2,3,4,5,6,7,8,9,10,11,12,13,14,15,16,17,18,19,20,21,22,23,24,25,26,27,28,29,30,31,
                                         32,32,33,33,34,34,35,35,36,36,36,36,37,37,37,37,38,38,38,38,38,38,38,38,39,39,39,39,39,39,39,39,
                                         40,40,40,40,40,40,40,40,40,40,40,40,40,40,40,40,41,41,41,41,41,41,41,41,41,41,41,41,41,41,41,41,
                                         42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42};
__device__ __forceinline__ uint32_t zkc_ll_code(uint32_t ll) { return ll < 64 ? ZKC_LL_CODE[ll] : (uint32_t)zk_highbit(ll) + 19; }
__device__ __forceinline__ uint32_t zkc_ml_code(uint32_t mlb) { return mlb < 128 ? ZKC_ML_CODE[mlb] : (uint32_t)zk_highbit(mlb) + 36; }

// forward bit writer (A.7 streams are written forward, read backward).  WORDS: the base is 4-byte aligned and full
// 32-bit words are stored at once (used when a lane streams straight into HBM).
template <bool WORDS>
struct ZkcBitWT {
    uint8_t* p; uint32_t cap, pos; unsigned long long acc; int nb; bool ovf;
    __device__ __forceinline__ void init(uint8_t* buf, uint32_t capacity) { p = buf; cap = capacity; pos = 0; acc = 0; nb = 0; ovf = false; }
    __device__ __forceinline__ void add(uint32_t v, int n) {          // n <= 32
        acc |= (unsigned long long)(v & (n == 32 ? 0xFFFFFFFFu : ((1u << n) - 1u))) << nb; nb += n;
        if (nb >= 32) {
            if (pos + 4 <= cap) {
                if (WORDS) *(uint32_t*)(p + pos) = (uint32_t)acc;
                else { p[pos] = (uint8_t)acc; p[pos + 1] = (uint8_t)(acc >> 8); p[pos + 2] = (uint8_t)(acc >> 16); p[pos + 3] = (uint8_t)(acc >> 24); }
            } else ovf = true;
            pos += 4; acc >>= 32; nb -= 32;
        }
    }
    // end mark + flush; returns total bytes or 0 on overflow
    __device__ __forceinline__ uint32_t finish() { add(1, 1); return finish_raw(); }
    // flush without end mark (FSE table descriptions, A.6)
    __device__ __forceinline__ uint32_t finish_raw() {
        while (nb > 0) { if (pos < cap) p[pos] = (uint8_t)acc; else ovf = true; pos++; acc >>= 8; nb -= 8; }
        return ovf ? 0 : pos;
    }
};
typedef ZkcBitWT<false> ZkcBitW;
typedef ZkcBitWT<true> ZkcBitWW;

// FSE compression table for one symbol alphabet (state values in [S, 2S))
// (table logs are capped at 8 by this encoder: 1 KiB per table lets twice as many block chains share an SM's shared memory)
struct ZkcFse {
    uint16_t state_tbl[256];
    uint32_t delta_nb[64];
    int16_t delta_find[64];
    int16_t norm[64];
    int8_t log, mode;                    // mode: 0 predefined, 1 RLE, 2 FSE-compressed
    uint8_t nsym, rle_sym;
};

// normalise counts to a sum of 2^log with every present symbol >= 1 (any such distribution is a valid header)
template <class CT>
__device__ void zkc_fse_normalize(ZkcFse& t, const CT* cnt, int nsym, uint32_t total, int log) {
    const uint32_t S = 1u << log;
    uint32_t sum = 0, best = 0; int besti = 0;
    for (int s = 0; s < nsym; s++) {
        uint32_t c = cnt[s], v = 0;
        if (c) { v = (uint32_t)(((unsigned long long)c * S + total / 2) / total); if (v == 0) v = 1; }
        t.norm[s] = (int16_t)v; sum += v;
        if (c > best) { best = c; besti = s; }
    }
    // give / take the rounding error to the largest symbols
    while (sum != S) {
        if (sum < S) { t.norm[besti] = (int16_t)(t.norm[besti] + (S - sum)); sum = S; }
        else {
            uint32_t over = sum - S;
            // take from the symbol with the largest normalised count that can afford it
            int bi = -1; int16_t bv = 1;
            for (int s = 0; s < nsym; s++) if (t.norm[s] > bv) { bv = t.norm[s]; bi = s; }
            if (bi < 0) break;
            uint32_t take = (uint32_t)(bv - 1) < over ? (uint32_t)(bv - 1) : over;
            t.norm[bi] = (int16_t)(bv - take); sum -= take;
        }
    }
    t.log = (int8_t)log; t.nsym = (uint8_t)nsym;
}

// build the encoding tables from t.norm (mirror of A.6 table build)
__device__ void zkc_fse_build(ZkcFse& t, uint8_t* symof /* >= 512 bytes scratch */) {
    const int log = t.log, S = 1 << log, nsym = t.nsym;
    uint16_t cumul[65];
    int high = S - 1;
    cumul[0] = 0;
    for (int s = 0; s < nsym; s++) {
        if (t.norm[s] == -1) { cumul[s + 1] = cumul[s] + 1; symof[high--] = (uint8_t)s; }
        else cumul[s + 1] = (uint16_t)(cumul[s] + t.norm[s]);
    }
    const int step = (S >> 1) + (S >> 3) + 3; int pos = 0;
    for (int s = 0; s < nsym; s++)
        for (int q = 0; q < t.norm[s]; q++) { symof[pos] = (uint8_t)s; do { pos = (pos + step) & (S - 1); } while (pos > high); }
    for (int u = 0; u < S; u++) { int s = symof[u]; t.state_tbl[cumul[s]++] = (uint16_t)(S + u); }
    int total = 0;
    for (int s = 0; s < nsym; s++) {
        int n = t.norm[s];
        if (n == 0) { t.delta_nb[s] = ((uint32_t)(log + 1) << 16) - (1u << log); t.delta_find[s] = 0; }
        else if (n == 1 || n == -1) { t.delta_nb[s] = ((uint32_t)log << 16) - (1u << log); t.delta_find[s] = (int16_t)(total - 1); total++; }
        else {
            uint32_t max_bits_out = (uint32_t)log - (uint32_t)zk_highbit((uint32_t)n - 1);
            uint32_t min_state_plus = (uint32_t)n << max_bits_out;
            t.delta_nb[s] = (max_bits_out << 16) - min_state_plus;
            t.delta_find[s] = (int16_t)(total - n); total += n;
        }
    }
}

// write the normalised-count header (A.6); returns bytes written (0 on overflow)
__device__ uint32_t zkc_fse_write_ncount(const ZkcFse& t, uint8_t* out, uint32_t cap) {
    ZkcBitW w; w.init(out, cap);
    const int log = t.log; const int S = 1 << log;
    w.add((uint32_t)(log - 5), 4);
    int remaining = S + 1, threshold = S, nb = log + 1, s = 0; bool prev0 = false;
    while (s < t.nsym && remaining > 1) {
        if (prev0) {
            int start = s;
            while (s < t.nsym && t.norm[s] == 0) s++;
            if (s == t.nsym) break;
            while (s >= start + 3) { start += 3; w.add(3, 2); }
            w.add((uint32_t)(s - start), 2);
        }
        int count = t.norm[s++];
        const int mx = 2 * threshold - 1 - remaining;
        remaining -= count < 0 ? -count : count;
        count++;
        if (count >= threshold) count += mx;
        w.add((uint32_t)count, nb - (count < mx ? 1 : 0));
        prev0 = count == 1;
        if (remaining < 1) return 0;
        while (remaining < threshold) { nb--; threshold >>= 1; }
    }
    if (remaining != 1) return 0;
    return w.finish_raw();
}

__device__ __forceinline__ void zkc_fse_init_state(const ZkcFse& t, uint32_t sym, uint32_t& state) {
    if (t.mode == 1) { state = 0; return; }
    const uint32_t dnb = t.delta_nb[sym];
    const uint32_t nb_out = (dnb + (1u << 15)) >> 16;
    const uint32_t value = (nb_out << 16) - dnb;
    state = t.state_tbl[(value >> nb_out) + t.delta_find[sym]];
}
template <class W>
__device__ __forceinline__ void zkc_fse_encode(const ZkcFse& t, W& w, uint32_t sym, uint32_t& state) {
    if (t.mode == 1) return;
    const uint32_t nb_out = (state + t.delta_nb[sym]) >> 16;
    w.add(state, (int)nb_out);
    state = t.state_tbl[(state >> nb_out) + t.delta_find[sym]];
}
template <class W>
__device__ __forceinline__ void zkc_fse_flush(const ZkcFse& t, W& w, uint32_t state) {
    if (t.mode == 1) return;
    w.add(state, t.log);
}

__device__ void zkc_fse_set_predefined(ZkcFse& t, int which) {
    if (which == 0) { for (int i = 0; i < 36; i++) t.norm[i] = ZK_LL_DEFAULT[i]; t.nsym = 36; t.log = 6; }
    else if (which == 1) { for (int i = 0; i < 29; i++) t.norm[i] = ZK_OF_DEFAULT[i]; t.nsym = 29; t.log = 5; }
    else { for (int i = 0; i < 53; i++) t.norm[i] = ZK_ML_DEFAULT[i]; t.nsym = 53; t.log = 6; }
    t.mode = 0;
}

// =============================================================================================
// K-C2s: sequence section -- one WARP per block.
// The only serial part of coding a block's sequences is the FSE state chain (state -> bits out -> next state, A.6): four
// integer operations and one shared-memory load per symbol.  Three lanes run the three chains (LL, OF, ML) over a tile of
// 32 sequences; everything else is done by all 32 lanes, one sequence each: codes and histograms (pass A), the per-step
// (deltaNbBits, deltaFindState) operands of the chains, extra bits, a warp scan of the bit counts and the packing of each
// sequence's <= 87 bits into a shared-memory staging window that is flushed to HBM as whole words.  (The first version
// ran one LANE per block with all of that on the serial chain: ~400 dependent instructions per sequence.)
// The section is written to a per-block scratch ([0,256) header + table descriptions, [256,..) bitstream) and moved
// into place by the assembly kernel.  Offsets arrive as Offset_Values (repeat codes resolved by K-C1).
// =============================================================================================
#define ZKC_SW 8                   // warps per CTA = blocks in flight per CTA
struct ZkcTabs { uint32_t ll_base[36], ml_base[53]; uint8_t ll_bits[36], ml_bits[53], ll_code[64], ml_code[128]; };
__device__ __forceinline__ uint32_t zkc_llc(const ZkcTabs& tb, uint32_t ll) { return ll < 64 ? tb.ll_code[ll] : (uint32_t)zk_highbit(ll) + 19; }
__device__ __forceinline__ uint32_t zkc_mlc(const ZkcTabs& tb, uint32_t mlb) { return mlb < 128 ? tb.ml_code[mlb] : (uint32_t)zk_highbit(mlb) + 36; }

struct ZkcSeqWarp {
    ZkcFse fse[3];                                   // 0 LL, 1 OF, 2 ML
    uint32_t cnt[3][64];
    union {
        uint8_t symof[3][256];                       // table build scratch (lanes 0..2 build one table each)
        struct {
            uint2 tin[3][33];                        // per step: (deltaNbBits, deltaFindState) of the step's symbol (padded: the three chains hit different banks)
            uint16_t tout[3][34];                    // per step: (bits << 4) | nbBits written by the chain
            uint32_t stage[96];                      // bit staging: [0] carries the partial word of the previous tile
        } b;
    } u;
    uint8_t hdr[3][84];                              // table descriptions before they are concatenated
};

// one table (lane t of the warp): choose the mode, build the coding table, write its description.  -> false: not encodable
__device__ bool zkc_seq_table(ZkcFse& ft, const uint32_t* cnt, int t, uint32_t nseq, uint8_t* symof, uint8_t* hdr, uint32_t* mode, uint32_t* nbytes) {
    const int max_log = 8, nsym_all = t == 0 ? 36 : (t == 1 ? 32 : 53);
    int last = nsym_all - 1; while (last > 0 && cnt[last] == 0) last--;
    uint32_t distinct = 0; for (int q = 0; q <= last; q++) distinct += cnt[q] != 0;
    if (distinct == 1) {
        ft.mode = 1; ft.rle_sym = (uint8_t)last; ft.log = 0;
        ft.state_tbl[0] = 0; ft.delta_nb[last] = 0; ft.delta_find[last] = 0;             // the chain then idles at state 0, emitting no bits
        hdr[0] = (uint8_t)last; *mode = 1; *nbytes = 1;
        return true;
    }
    if (nseq < 48 && (t != 1 || last <= 28)) { zkc_fse_set_predefined(ft, t); zkc_fse_build(ft, symof); *mode = 0; *nbytes = 0; return true; }
    int lg = zk_highbit(nseq) - 1; if (lg < 5) lg = 5; if (lg > max_log) lg = max_log;
    int need = zk_highbit(distinct) + 1; if (lg < need) lg = need; if (lg > max_log) return false;
    zkc_fse_normalize(ft, cnt, last + 1, nseq, lg);
    ft.mode = 2;
    zkc_fse_build(ft, symof);
    const uint32_t hb = zkc_fse_write_ncount(ft, hdr, 84);
    if (!hb) return false;
    *mode = 2; *nbytes = hb;
    return true;
}

// whole warp; returns false if the section cannot be encoded within the scratch (the block then becomes a Raw block)
__device__ bool zkc_encode_sequences(ZkcSeqWarp& sw, const ZkcTabs& tb, const uint16_t* s_ll, const uint16_t* s_ml, const uint32_t* s_ov, uint32_t nseq,
                                     uint8_t* out, uint32_t* hdr_bytes, uint32_t* bits_bytes, int lane) {
    // ---- pass A: code histograms, one sequence per lane
    for (int i = lane; i < 3 * 64; i += 32) (&sw.cnt[0][0])[i] = 0;
    __syncwarp();
    for (uint32_t i = lane; i < nseq; i += 32) {
        atomicAdd(&sw.cnt[0][zkc_llc(tb, s_ll[i])], 1u); atomicAdd(&sw.cnt[1][zk_highbit(s_ov[i])], 1u); atomicAdd(&sw.cnt[2][zkc_mlc(tb, s_ml[i])], 1u);
    }
    __syncwarp();
    // ---- tables: lanes 0..2 build one each
    uint32_t mode = 0, nb_t = 0; bool ok = true;
    if (lane < 3) ok = zkc_seq_table(sw.fse[lane], sw.cnt[lane], lane, nseq, sw.u.symof[lane], sw.hdr[lane], &mode, &nb_t);
    if (!__all_sync(0xFFFFFFFFu, ok)) return false;
    uint32_t hp = 0;
    if (lane == 0) {
        if (nseq < 128) out[hp++] = (uint8_t)nseq;
        else if (nseq < 0x7F00) { out[hp++] = (uint8_t)((nseq >> 8) + 128); out[hp++] = (uint8_t)nseq; }
        else { out[hp++] = 255; out[hp++] = (uint8_t)(nseq - 0x7F00); out[hp++] = (uint8_t)((nseq - 0x7F00) >> 8); }
    }
    hp = __shfl_sync(0xFFFFFFFFu, hp, 0);
    {
        const uint32_t m0 = __shfl_sync(0xFFFFFFFFu, mode, 0), m1 = __shfl_sync(0xFFFFFFFFu, mode, 1), m2 = __shfl_sync(0xFFFFFFFFu, mode, 2);
        const uint32_t n0 = __shfl_sync(0xFFFFFFFFu, nb_t, 0), n1 = __shfl_sync(0xFFFFFFFFu, nb_t, 1), n2 = __shfl_sync(0xFFFFFFFFu, nb_t, 2);
        if (lane == 0) out[hp] = (uint8_t)((m0 << 6) | (m1 << 4) | (m2 << 2));
        hp++;
        if (hp + n0 + n1 + n2 > ZKC_SEQHDR - 6) return false;
        for (uint32_t i = lane; i < n0; i += 32) out[hp + i] = sw.hdr[0][i];
        for (uint32_t i = lane; i < n1; i += 32) out[hp + n0 + i] = sw.hdr[1][i];
        for (uint32_t i = lane; i < n2; i += 32) out[hp + n0 + n1 + i] = sw.hdr[2][i];
        hp += n0 + n1 + n2;
    }
    __syncwarp();                                    // the build scratch (union) is dead from here on
    // ---- pass B (backward): the bitstream, last sequence first (mirror of the decoder's order, A.5)
    uint32_t* const gw = (uint32_t*)(out + ZKC_SEQHDR);
    const uint32_t cap_words = (ZKC_SEQSEC - ZKC_SEQHDR) / 4;
    for (int i = lane; i < 96; i += 32) sw.u.b.stage[i] = 0;
    uint32_t st = 0;                                 // lanes 0..2: state of chain `lane`
    uint32_t bitpos = 0;                             // bits emitted so far
    bool first = true, ovf = false;
    const uint32_t lt_mask = (1u << lane) - 1u; (void)lt_mask;
    for (uint32_t hi_i = nseq; hi_i > 0;) {
        const uint32_t cntT = hi_i < 32u ? hi_i : 32u;
        const bool act = (uint32_t)lane < cntT;
        const uint32_t idx = act ? hi_i - 1u - (uint32_t)lane : 0u;       // step `lane` of this tile codes sequence idx
        const uint32_t llv = s_ll[idx], mlb = s_ml[idx], ov = s_ov[idx];
        const uint32_t llc = zkc_llc(tb, llv), mlc = zkc_mlc(tb, mlb), ofc = (uint32_t)zk_highbit(ov);
        if (act) {
            sw.u.b.tin[0][lane] = make_uint2(sw.fse[0].delta_nb[llc], (uint32_t)(int)sw.fse[0].delta_find[llc]);
            sw.u.b.tin[1][lane] = make_uint2(sw.fse[1].delta_nb[ofc], (uint32_t)(int)sw.fse[1].delta_find[ofc]);
            sw.u.b.tin[2][lane] = make_uint2(sw.fse[2].delta_nb[mlc], (uint32_t)(int)sw.fse[2].delta_find[mlc]);
        }
        __syncwarp();
        if (lane < 3) {                              // the three chains
            const uint16_t* stt = sw.fse[lane].state_tbl;
            const uint2* ti = sw.u.b.tin[lane]; uint16_t* to = sw.u.b.tout[lane];
            uint32_t j = 0;
            if (first) {
                if (sw.fse[lane].mode == 1) st = 0;
                else {
                    const uint2 d = ti[0];
                    const uint32_t nb_out = (d.x + (1u << 15)) >> 16, value = (nb_out << 16) - d.x;
                    st = stt[(value >> nb_out) + (int)d.y];
                }
                to[0] = 0; j = 1;
            }
#pragma unroll 4
            for (; j < cntT; j++) {
                const uint2 d = ti[j];
                const uint32_t nb_out = (st + d.x) >> 16;
                to[j] = (uint16_t)(((st & ((1u << nb_out) - 1u)) << 4) | nb_out);
                st = stt[(st >> nb_out) + (int)d.y];
            }
        }
        first = false;
        __syncwarp();
        // this lane's sequence: state bits (OF, ML, LL), then extra bits (LL, ML, OF)
        unsigned long long v = 0; uint32_t n1 = 0, v2 = 0, n2 = 0;
        if (act) {
            const uint32_t o = sw.u.b.tout[1][lane], m = sw.u.b.tout[2][lane], l = sw.u.b.tout[0][lane];
            v = o >> 4; n1 = o & 15u;
            v |= (unsigned long long)(m >> 4) << n1; n1 += m & 15u;
            v |= (unsigned long long)(l >> 4) << n1; n1 += l & 15u;
            v |= (unsigned long long)(llv - tb.ll_base[llc]) << n1; n1 += tb.ll_bits[llc];
            v |= (unsigned long long)(mlb + 3u - tb.ml_base[mlc]) << n1; n1 += tb.ml_bits[mlc];
            v2 = ov - (1u << ofc); n2 = ofc;
        }
        uint32_t incl = n1 + n2;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d); if (lane >= d) incl += t; }
        const uint32_t tile_bits = __shfl_sync(0xFFFFFFFFu, incl, 31);
        const uint32_t base_bit = bitpos & 31u;
        if (act) {
            uint32_t pos = base_bit + incl - (n1 + n2);
            if (n1) {
                const uint32_t w = pos >> 5, sh = pos & 31u;
                const unsigned long long lo = v << sh;
                atomicOr(&sw.u.b.stage[w], (uint32_t)lo);
                if (lo >> 32) atomicOr(&sw.u.b.stage[w + 1], (uint32_t)(lo >> 32));
                if (sh) { const uint32_t hi = (uint32_t)(v >> (64u - sh)); if (hi) atomicOr(&sw.u.b.stage[w + 2], hi); }
            }
            pos += n1;
            if (n2) {
                const uint32_t w = pos >> 5, sh = pos & 31u;
                const unsigned long long lo = (unsigned long long)v2 << sh;
                atomicOr(&sw.u.b.stage[w], (uint32_t)lo);
                if (lo >> 32) atomicOr(&sw.u.b.stage[w + 1], (uint32_t)(lo >> 32));
            }
        }
        __syncwarp();
        // flush the full words, keep the partial one as word 0 of the next tile
        const uint32_t nwords = (base_bit + tile_bits) >> 5, word0 = bitpos >> 5;
        if (word0 + nwords > cap_words) ovf = true;
        else for (uint32_t w = lane; w < nwords; w += 32) gw[word0 + w] = sw.u.b.stage[w];
        const uint32_t carry = sw.u.b.stage[nwords];
        __syncwarp();
        for (uint32_t w = lane; w <= nwords + 2; w += 32) sw.u.b.stage[w] = w == 0 ? carry : 0u;
        __syncwarp();
        bitpos += tile_bits;
        hi_i -= cntT;
    }
    // final states (ML, OF, LL), then the end mark
    const uint32_t s_l = __shfl_sync(0xFFFFFFFFu, st, 0), s_o = __shfl_sync(0xFFFFFFFFu, st, 1), s_m = __shfl_sync(0xFFFFFFFFu, st, 2);
    const uint32_t lg_l = (uint32_t)sw.fse[0].log, lg_o = (uint32_t)sw.fse[1].log, lg_m = (uint32_t)sw.fse[2].log;
    unsigned long long fin = s_m & ((1u << lg_m) - 1u); uint32_t nf = lg_m;
    fin |= (unsigned long long)(s_o & ((1u << lg_o) - 1u)) << nf; nf += lg_o;
    fin |= (unsigned long long)(s_l & ((1u << lg_l) - 1u)) << nf; nf += lg_l;
    fin |= 1ull << nf; nf += 1;
    const uint32_t base_bit = bitpos & 31u, word0 = bitpos >> 5;
    const unsigned long long tail = ((unsigned long long)sw.u.b.stage[0]) | (fin << base_bit);      // <= 31 + 25 bits
    const uint32_t total_bits = bitpos + nf;
    const uint32_t sb = (total_bits + 7u) >> 3;
    if (ovf || word0 + 2 > cap_words) return false;
    if (lane == 0) { gw[word0] = (uint32_t)tail; gw[word0 + 1] = (uint32_t)(tail >> 32); }
    *hdr_bytes = hp; *bits_bytes = sb;
    return true;
}

__global__ void __launch_bounds__(32 * ZKC_SW) zk_seq_enc_kernel(ZkEncodeArgs a) {
    ZK_DYN_SMEM(smem);
    ZkcTabs* tb = (ZkcTabs*)smem;
    ZkcSeqWarp* sws = (ZkcSeqWarp*)(smem + ((sizeof(ZkcTabs) + 15) & ~(size_t)15));
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, tid = threadIdx.x, nt = 32 * ZKC_SW;
    for (int i = tid; i < 36; i += nt) { tb->ll_base[i] = ZK_LL_BASE[i]; tb->ll_bits[i] = ZK_LL_BITS[i]; }
    for (int i = tid; i < 53; i += nt) { tb->ml_base[i] = ZK_ML_BASE[i]; tb->ml_bits[i] = ZK_ML_BITS[i]; }
    for (int i = tid; i < 64; i += nt) tb->ll_code[i] = ZKC_LL_CODE[i];
    for (int i = tid; i < 128; i += nt) tb->ml_code[i] = ZKC_ML_CODE[i];
    __syncthreads();
    const uint32_t b = blockIdx.x * ZKC_SW + warp;
    if (b >= a.n_blocks) return;
    const uint32_t nseq = a.blocks[b].nseq;
    uint32_t hb = 0, sb = 0;
    if (nseq) {
        const bool ok = zkc_encode_sequences(sws[warp], *tb, a.seq_ll + (size_t)b * ZKC_MAXSEQ, a.seq_ml + (size_t)b * ZKC_MAXSEQ,
                                             a.seq_off + (size_t)b * ZKC_MAXSEQ, nseq, a.seqsec + (size_t)b * ZKC_SEQSEC, &hb, &sb, lane);
        if (!ok) { hb = 0; sb = 0; }
    }
    if (lane == 0) { a.blocks[b].seq_hdr = hb; a.blocks[b].seq_bits = sb; }
}

#define ZKC_BITBUF 6144u                // shared-memory scratch: Huffman build arrays, then one Huffman stream (longer streams are packed in tiles)

// per-warp shared state of K-C2l.  The three phases (tree build, tree description, stream packing) never overlap, so
// their scratch shares one union: 10 KiB per warp instead of 18 -- the kernel is latency-bound and shared memory was
// what limited the warps per SM.
struct ZkcC2Smem {
    uint32_t hist[256];
    uint32_t hist4[2][256];             // per-stream counts, two 16-bit fields per word (streams 0|1, 2|3): stream sizes without a second pass over the literals
    uint16_t hcode[256]; uint8_t hlen[256];      // hcode: (length << 11) | code
    union {
        uint8_t bitbuf[ZKC_BITBUF];
        struct { ZkcFse fse; uint8_t symof[512]; uint8_t weights[256]; } w;    // FSE coding of the Huffman weights
    } u;
    uint8_t hdr[256];                   // literal header + tree description
    uint32_t scratch[16];
};

// Huffman code lengths limited to 11 bits.  Whole warp: the symbols are ranked by count with an all-pairs comparison
// in shared memory (each lane ranks 8 symbols), then lane 0 runs the two-queue tree build on shared-memory arrays
// (aliasing the bit buffer, which is not in use yet).  Returns max code length (0 = fewer than two symbols).
__device__ int zkc_huf_build(ZkcC2Smem& sm, int lane) {
    uint16_t* order = (uint16_t*)sm.u.bitbuf;                 // 256 x u16   symbols sorted by count ascending
    uint32_t* weight = (uint32_t*)(sm.u.bitbuf + 512);        // 511 x u32
    uint16_t* parent = (uint16_t*)(sm.u.bitbuf + 512 + 2048); // 511 x u16
    uint8_t* depth = sm.u.bitbuf + 512 + 2048 + 1024;         // 511 x u8
    int n = 0;
    for (int s0 = 0; s0 < 256; s0 += 32) n += __popc(__ballot_sync(0xFFFFFFFFu, sm.hist[s0 + lane] != 0));
    if (n < 2) return 0;
    // compact the present symbols (ascending), then rank them among themselves: n^2 / 32 comparisons per lane instead of 256 * 8
    uint32_t* pcnt = (uint32_t*)(sm.u.bitbuf + 4608);         // n x u32
    uint8_t* psym = sm.u.bitbuf + 4608 + 1024;                // n x u8
    {
        int basep = 0;
        for (int s0 = 0; s0 < 256; s0 += 32) {
            const uint32_t c = sm.hist[s0 + lane];
            const uint32_t m = __ballot_sync(0xFFFFFFFFu, c != 0);
            if (c) { const int k = basep + __popc(m & ((1u << lane) - 1u)); pcnt[k] = c; psym[k] = (uint8_t)(s0 + lane); }
            basep += __popc(m);
        }
    }
    __syncwarp();
    for (int k = lane; k < n; k += 32) {
        const uint32_t c = pcnt[k];
        int rank = 0;
        for (int j = 0; j < n; j++) { const uint32_t cj = pcnt[j]; rank += (cj < c || (cj == c && j < k)); }
        order[rank] = (uint16_t)psym[k];
    }
    __syncwarp();
    if (lane == 0) {
        for (int i = 0; i < n; i++) weight[i] = sm.hist[order[i]];
        int leaf = 0, inode = n, next = n;
        for (int k = 0; k < n - 1; k++) {       // two-queue Huffman: leaves 0..n-1 (sorted), internal nodes n..2n-2
            int a, b;
            if (leaf < n && (inode >= next || weight[leaf] <= weight[inode])) a = leaf++; else a = inode++;
            if (leaf < n && (inode >= next || weight[leaf] <= weight[inode])) b = leaf++; else b = inode++;
            weight[next] = weight[a] + weight[b]; parent[a] = (uint16_t)next; parent[b] = (uint16_t)next; next++;
        }
        depth[next - 1] = 0;
        for (int i = next - 2; i >= 0; i--) depth[i] = (uint8_t)(depth[parent[i]] + 1);
        // histogram of code lengths, limited to 11 (miniz-style redistribution keeps the code complete)
        const int L = 11;
        int num[33]; for (int i = 0; i <= 32; i++) num[i] = 0;
        for (int i = 0; i < n; i++) num[depth[i] > 32 ? 32 : depth[i]]++;
        for (int i = L + 1; i <= 32; i++) { num[L] += num[i]; num[i] = 0; }
        unsigned total = 0;
        for (int i = L; i > 0; i--) total += (unsigned)num[i] << (L - i);
        while (total != (1u << L)) {
            num[L]--;
            for (int i = L - 1; i > 0; i--) if (num[i]) { num[i]--; num[i + 1] += 2; break; }
            total--;
        }
        // most frequent symbols (end of `order`) get the shortest codes
        int idx = n - 1, maxlen = 0;
        for (int l = 1; l <= L; l++) for (int k = 0; k < num[l]; k++) { sm.hlen[order[idx--]] = (uint8_t)l; maxlen = l; }
        sm.scratch[2] = (uint32_t)maxlen;
    }
    __syncwarp();
    return (int)sm.scratch[2];
}

__global__ void __launch_bounds__(32) zk_lit_enc_kernel(ZkEncodeArgs a) {
    __shared__ ZkcC2Smem sm;
    const int lane = threadIdx.x;
    const uint32_t b = blockIdx.x;
    size_t lo, hi, fstart;
    zkc_block_range(a, b, lo, hi, fstart);
    const uint32_t len = (uint32_t)(hi - lo);
    const uint32_t k_in_frame = b % a.blocks_per_frame;
    // blocks past the end of a short last frame carry nothing
    {
        uint32_t f = b / a.blocks_per_frame;
        size_t fend = fstart + a.frame_size < a.n ? fstart + a.frame_size : a.n;
        uint32_t nb_frame = (uint32_t)((fend - fstart + ZKC_BLOCK - 1) / ZKC_BLOCK); if (nb_frame == 0) nb_frame = 1;
        (void)f;
        if (k_in_frame >= nb_frame) { if (lane == 0) { a.blocks[b].csize = 0; a.blocks[b].lit_bytes = 0xFFFFFFFFu; } return; }
        // Last_Block flag
        sm.scratch[0] = (k_in_frame == nb_frame - 1) ? 1u : 0u;
    }
    __syncwarp();
    const uint32_t last_flag = sm.scratch[0];
    const uint32_t nseq = a.blocks[b].nseq, nlit = a.blocks[b].nlit;
    const uint8_t* lits = a.lits + (size_t)b * ZKC_BLOCK;
    uint8_t* out = a.stage + (size_t)b * ZKC_SLOT;
    uint32_t opos = 3;                                   // block header written last
    bool raw_block = len < 32;                           // tiny blocks: not worth entropy coding

    // ------------------------------------------------------------------ literals section (A.3)
    if (!raw_block) {
        for (int i = lane; i < 256; i += 32) { sm.hist4[0][i] = 0; sm.hist4[1][i] = 0; sm.hlen[i] = 0; }
        __syncwarp();
        {   // four literals per lane and load (the buffer is 32 KiB aligned); the stream a literal belongs to follows from its index
            const uint32_t seg = (nlit + 3) / 4, n4 = nlit & ~3u;
            for (uint32_t i = 4u * (uint32_t)lane; i < n4; i += 128) {
                const uint32_t w = *(const uint32_t*)(lits + i);
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const uint32_t idx = i + q, st = (idx >= seg) + (idx >= 2 * seg) + (idx >= 3 * seg);
                    atomicAdd(&sm.hist4[st >> 1][(w >> (8 * q)) & 255u], 1u << ((st & 1u) * 16u));
                }
            }
            if ((uint32_t)lane < nlit - n4) {
                const uint32_t idx = n4 + lane, st = (idx >= seg) + (idx >= 2 * seg) + (idx >= 3 * seg);
                atomicAdd(&sm.hist4[st >> 1][lits[idx]], 1u << ((st & 1u) * 16u));
            }
        }
        __syncwarp();
        for (int i = lane; i < 256; i += 32) { const uint32_t a0 = sm.hist4[0][i], a1 = sm.hist4[1][i]; sm.hist[i] = (a0 & 0xFFFFu) + (a0 >> 16) + (a1 & 0xFFFFu) + (a1 >> 16); }
        __syncwarp();
        // decide: Raw / RLE / Huffman
        int maxlen = 0; uint32_t lit_mode = 0;           // 0 raw, 1 rle, 2 huffman
        uint32_t mx = 0;
        for (int s = lane; s < 256; s += 32) mx = max(mx, sm.hist[s]);
        for (int d = 16; d; d >>= 1) mx = max(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, d));
        if (nlit > 0 && mx == nlit && nlit >= 2) lit_mode = 1;
        else if (nlit >= 64) {
            maxlen = zkc_huf_build(sm, lane);
            if (maxlen) {
                uint32_t bits = 0;
                for (int s = lane; s < 256; s += 32) bits += sm.hist[s] * sm.hlen[s];
                for (int d = 16; d; d >>= 1) bits += __shfl_xor_sync(0xFFFFFFFFu, bits, d);
                uint32_t est = (bits + 7) / 8 + 8 + 130;
                if (est < nlit) lit_mode = 2;
            }
        }

        uint32_t tree_bytes = 0;
        if (lit_mode == 2) {
            // canonical codes exactly as the decoder lays out its table: weight ascending, symbol ascending (A.4)
            if (lane == 0) {
                int last_sym = 255; while (last_sym > 0 && sm.hlen[last_sym] == 0) last_sym--;
                // start cell of every symbol in two linear passes: cells per weight class, then a running cursor per class
                uint32_t cls[13];
                for (int w = 0; w < 13; w++) cls[w] = 0;
                for (int s = 0; s <= last_sym; s++) if (sm.hlen[s]) cls[maxlen + 1 - sm.hlen[s]] += 1;
                { uint32_t acc = 0; for (int w = 1; w <= maxlen; w++) { uint32_t n = cls[w]; cls[w] = acc; acc += n << (w - 1); } }
                for (int s = 0; s <= last_sym; s++)
                    if (sm.hlen[s]) { const int w = maxlen + 1 - sm.hlen[s]; sm.hcode[s] = (uint16_t)((cls[w] >> (w - 1)) | ((uint32_t)sm.hlen[s] << 11)); cls[w] += 1u << (w - 1); }
                // tree description: weights of symbols 0..last_sym-1 (the last one is implied)
                int nw = last_sym;
                for (int s = 0; s < nw; s++) sm.u.w.weights[s] = sm.hlen[s] ? (uint8_t)(maxlen + 1 - sm.hlen[s]) : 0;
                uint32_t tb = 0;
                // FSE-compressed weights (two interleaved states), A.4
                if (nw > 1) {
                    uint32_t wc[16]; for (int i = 0; i < 16; i++) wc[i] = 0;
                    int maxw = 0;
                    for (int s = 0; s < nw; s++) { wc[sm.u.w.weights[s]]++; if (sm.u.w.weights[s] > maxw) maxw = sm.u.w.weights[s]; }
                    uint32_t distinct = 0; for (int i = 0; i <= maxw; i++) distinct += wc[i] != 0;
                    if (distinct > 1) {
                        ZkcFse& t = sm.u.w.fse;
                        int lg = 6; while (lg > 5 && (1 << lg) > nw) lg--;        // table log 5..6
                        zkc_fse_normalize(t, wc, maxw + 1, (uint32_t)nw, lg);
                        t.mode = 2;
                        zkc_fse_build(t, sm.u.w.symof);
                        uint32_t hb = zkc_fse_write_ncount(t, sm.hdr + 1, 120);
                        if (hb) {
                            ZkcBitW w; w.init(sm.hdr + 1 + hb, 127 - hb);
                            // encode from the last weight to the first, alternating two states
                            uint32_t s1, s2; int n = nw;
                            if (n & 1) { zkc_fse_init_state(t, sm.u.w.weights[n - 1], s1); zkc_fse_init_state(t, sm.u.w.weights[n - 2], s2); n -= 2;
                                         zkc_fse_encode(t, w, sm.u.w.weights[n - 1], s1); n--; }
                            else { zkc_fse_init_state(t, sm.u.w.weights[n - 1], s2); zkc_fse_init_state(t, sm.u.w.weights[n - 2], s1); n -= 2; }
                            while (n >= 2) { zkc_fse_encode(t, w, sm.u.w.weights[n - 1], s2); zkc_fse_encode(t, w, sm.u.w.weights[n - 2], s1); n -= 2; }
                            zkc_fse_flush(t, w, s2); zkc_fse_flush(t, w, s1);
                            uint32_t sb = w.finish();
                            if (sb && hb + sb < 128 && hb + sb < (uint32_t)(nw + 1) / 2) { sm.hdr[0] = (uint8_t)(hb + sb); tb = 1 + hb + sb; }
                        }
                    }
                }
                if (!tb) {
                    if (nw <= 128) {
                        sm.hdr[0] = (uint8_t)(127 + nw);
                        for (int s = 0; s < nw; s += 2) sm.hdr[1 + s / 2] = (uint8_t)((sm.u.w.weights[s] << 4) | (s + 1 < nw ? sm.u.w.weights[s + 1] : 0));
                        tb = 1 + (uint32_t)(nw + 1) / 2;
                    }
                }
                sm.scratch[3] = tb;
            }
            __syncwarp();
            tree_bytes = sm.scratch[3];
            if (!tree_bytes) lit_mode = 0;               // cannot describe the tree: raw literals
        }

        if (lit_mode == 2) {
            // stream sizes first (so the section header, which precedes the streams, can be sized)
            const uint32_t seg = (nlit + 3) / 4;
            uint32_t ssz[4];
            {
                uint32_t b0 = 0, b1 = 0, b2 = 0, b3 = 0;
                for (int sy = lane; sy < 256; sy += 32) {
                    const uint32_t l = sm.hlen[sy], a0 = sm.hist4[0][sy], a1 = sm.hist4[1][sy];
                    b0 += (a0 & 0xFFFFu) * l; b1 += (a0 >> 16) * l; b2 += (a1 & 0xFFFFu) * l; b3 += (a1 >> 16) * l;
                }
                for (int d = 16; d; d >>= 1) {
                    b0 += __shfl_xor_sync(0xFFFFFFFFu, b0, d); b1 += __shfl_xor_sync(0xFFFFFFFFu, b1, d);
                    b2 += __shfl_xor_sync(0xFFFFFFFFu, b2, d); b3 += __shfl_xor_sync(0xFFFFFFFFu, b3, d);
                }
                ssz[0] = (b0 + 1 + 7) / 8; ssz[1] = (b1 + 1 + 7) / 8; ssz[2] = (b2 + 1 + 7) / 8; ssz[3] = (b3 + 1 + 7) / 8;   // + end mark
            }
            const uint32_t comp = tree_bytes + 6 + ssz[0] + ssz[1] + ssz[2] + ssz[3];
            if (comp >= nlit || ssz[0] > 0xFFFF || ssz[1] > 0xFFFF || ssz[2] > 0xFFFF) lit_mode = 0;
            else {
                // header: 4 streams, size format by magnitude
                uint32_t hsz;
                if (nlit < 1024 && comp < 1024) { hsz = 3; unsigned long long v = 2u | (1u << 2) | ((unsigned long long)nlit << 4) | ((unsigned long long)comp << 14);
                    if (lane == 0) { out[opos] = (uint8_t)v; out[opos + 1] = (uint8_t)(v >> 8); out[opos + 2] = (uint8_t)(v >> 16); } }
                else if (nlit < 16384 && comp < 16384) { hsz = 4; unsigned long long v = 2u | (2u << 2) | ((unsigned long long)nlit << 4) | ((unsigned long long)comp << 18);
                    if (lane == 0) { out[opos] = (uint8_t)v; out[opos + 1] = (uint8_t)(v >> 8); out[opos + 2] = (uint8_t)(v >> 16); out[opos + 3] = (uint8_t)(v >> 24); } }
                else { hsz = 5; unsigned long long v = 2u | (3u << 2) | ((unsigned long long)nlit << 4) | ((unsigned long long)comp << 22);
                    if (lane == 0) { out[opos] = (uint8_t)v; out[opos + 1] = (uint8_t)(v >> 8); out[opos + 2] = (uint8_t)(v >> 16); out[opos + 3] = (uint8_t)(v >> 24); out[opos + 4] = (uint8_t)(v >> 32); } }
                opos += hsz;
                for (uint32_t i = lane; i < tree_bytes; i += 32) out[opos + i] = sm.hdr[i];
                opos += tree_bytes;
                if (lane == 0) { out[opos] = (uint8_t)ssz[0]; out[opos + 1] = (uint8_t)(ssz[0] >> 8); out[opos + 2] = (uint8_t)ssz[1]; out[opos + 3] = (uint8_t)(ssz[1] >> 8);
                                 out[opos + 4] = (uint8_t)ssz[2]; out[opos + 5] = (uint8_t)(ssz[2] >> 8); }
                opos += 6;
                // encode each stream: symbol i of the stream sits above all later symbols (the decoder reads backward),
                // so its bit position is the sum of the code lengths of the symbols after it -> warp scan over reversed order
                __syncwarp();                                         // the tree description has left the union
                for (int st = 0; st < 4; st++) {
                    const uint32_t s0 = st * seg, s1 = st < 3 ? s0 + seg : nlit, m = s1 - s0;
                    uint32_t* wbuf = (uint32_t*)sm.u.bitbuf;
                    // a stream that fits the buffer is packed there and copied out once; a longer one goes through a 48-word
                    // window whose full words are flushed after every 128 symbols
                    const bool whole = ssz[st] + 8 <= ZKC_BITBUF;
                    const uint32_t words = whole ? (ssz[st] + 3) / 4 : 64u;
                    for (uint32_t i = lane; i < words; i += 32) wbuf[i] = 0;
                    __syncwarp();
                    uint32_t base = 0;                                // bits of the stream emitted so far
                    for (uint32_t g = 0; g < m; g += 128) {
                        // four symbols per lane (reversed indices r .. r+3, r lowest in the stream): one scan and at most
                        // three atomics serve 128 symbols
                        const uint32_t r = g + 4u * (uint32_t)lane;
                        unsigned long long v = 0; uint32_t l = 0;
                        if (r + 4 <= m) {
                            // the four symbols are the bytes [s1-4-r, s1-r): one unaligned 4-byte load (two aligned ones)
                            const uint32_t ad = s1 - 4u - r, mis = ad & 3u;
                            const uint32_t* wp = (const uint32_t*)(lits + (ad - mis));
                            const uint32_t w4 = mis ? __funnelshift_r(wp[0], wp[1], mis * 8u) : wp[0];
#pragma unroll
                            for (int q = 0; q < 4; q++) {
                                const uint32_t cl = sm.hcode[(w4 >> (8 * (3 - q))) & 255u]; v |= (unsigned long long)(cl & 2047u) << l; l += cl >> 11;
                            }
                        } else {
#pragma unroll
                            for (int q = 0; q < 4; q++) {
                                if (r + q < m) { const uint32_t cl = sm.hcode[lits[s1 - 1 - r - q]]; v |= (unsigned long long)(cl & 2047u) << l; l += cl >> 11; }
                            }
                        }
                        uint32_t incl = l;
                        for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d); if (lane >= d) incl += t; }
                        const uint32_t org = whole ? base : (base & 31u);     // bit position of the tile inside wbuf
                        const uint32_t bitpos = org + incl - l;
                        if (l) {
                            const uint32_t sh = bitpos & 31u, w = bitpos >> 5;
                            const unsigned long long lo2 = v << sh;
                            atomicOr(&wbuf[w], (uint32_t)lo2);
                            if (lo2 >> 32) atomicOr(&wbuf[w + 1], (uint32_t)(lo2 >> 32));
                            if (sh) { const uint32_t hi2 = (uint32_t)(v >> (64u - sh)); if (hi2) atomicOr(&wbuf[w + 2], hi2); }
                        }
                        const uint32_t tile_bits = __shfl_sync(0xFFFFFFFFu, incl, 31);
                        if (!whole) {
                            __syncwarp();
                            const uint32_t nwords = (org + tile_bits) >> 5, byte0 = (base >> 5) * 4u;
                            for (uint32_t i = lane; i < nwords * 4u; i += 32) out[opos + byte0 + i] = sm.u.bitbuf[i];
                            const uint32_t carry = wbuf[nwords];
                            __syncwarp();
                            for (uint32_t i = lane; i <= nwords + 2; i += 32) wbuf[i] = i == 0 ? carry : 0u;
                            __syncwarp();
                        }
                        base += tile_bits;
                    }
                    __syncwarp();
                    if (whole) {
                        if (lane == 0) atomicOr(&wbuf[base >> 5], 1u << (base & 31));   // end mark
                        __syncwarp();
                        for (uint32_t i = lane; i < ssz[st]; i += 32) out[opos + i] = sm.u.bitbuf[i];
                    } else if (lane == 0) {
                        const unsigned long long tail = (unsigned long long)wbuf[0] | (1ull << (base & 31u));
                        const uint32_t byte0 = (base >> 5) * 4u;
                        for (uint32_t i = 0; byte0 + i < ssz[st]; i++) out[opos + byte0 + i] = (uint8_t)(tail >> (8u * i));
                    }
                    opos += ssz[st];
                    __syncwarp();
                }
            }
        }
        if (lit_mode == 1) {
            // RLE literals
            uint32_t hsz = nlit < 32 ? 1 : (nlit < 4096 ? 2 : 3);
            if (lane == 0) {
                if (hsz == 1) out[opos] = (uint8_t)(1u | (nlit << 3));
                else if (hsz == 2) { uint32_t v = 1u | (1u << 2) | (nlit << 4); out[opos] = (uint8_t)v; out[opos + 1] = (uint8_t)(v >> 8); }
                else { uint32_t v = 1u | (3u << 2) | (nlit << 4); out[opos] = (uint8_t)v; out[opos + 1] = (uint8_t)(v >> 8); out[opos + 2] = (uint8_t)(v >> 16); }
                out[opos + hsz] = lits[0];
            }
            opos += hsz + 1;
        } else if (lit_mode == 0) {
            uint32_t hsz = nlit < 32 ? 1 : (nlit < 4096 ? 2 : 3);
            if (lane == 0) {
                if (hsz == 1) out[opos] = (uint8_t)(0u | (nlit << 3));
                else if (hsz == 2) { uint32_t v = 0u | (1u << 2) | (nlit << 4); out[opos] = (uint8_t)v; out[opos + 1] = (uint8_t)(v >> 8); }
                else { uint32_t v = 0u | (3u << 2) | (nlit << 4); out[opos] = (uint8_t)v; out[opos + 1] = (uint8_t)(v >> 8); out[opos + 2] = (uint8_t)(v >> 16); }
            }
            opos += hsz;
            if (opos + nlit + 4 >= len + 3) raw_block = true;       // cannot win any more
            else { for (uint32_t i = lane; i < nlit; i += 32) out[opos + i] = lits[i]; opos += nlit; }
        }
    }

    // the sequences section is coded concurrently by K-C2s on another stream; zk_block_finish_kernel joins the two
    if (lane == 0) { a.blocks[b].lit_bytes = raw_block ? 0u : opos; a.blocks[b].last_flag = last_flag; }
}

// K-C2f: join literals + sequences, fall back to a Raw block when that is not smaller, write the block header (A.2)
__global__ void __launch_bounds__(128) zk_block_finish_kernel(ZkEncodeArgs a) {
    const int lane = threadIdx.x & 31;
    const uint32_t b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= a.n_blocks) return;
    const ZkcBlock bl = a.blocks[b];
    if (bl.csize == 0 && bl.lit_bytes == 0xFFFFFFFFu) return;           // slot beyond the end of a short frame
    size_t lo, hi, fstart;
    zkc_block_range(a, b, lo, hi, fstart);
    const uint32_t len = (uint32_t)(hi - lo);
    uint8_t* out = a.stage + (size_t)b * ZKC_SLOT;
    uint32_t opos = bl.lit_bytes;
    bool raw_block = opos == 0;
    if (!raw_block) {
        if (bl.nseq == 0) { if (lane == 0) out[opos] = 0; opos += 1; }
        else {
            const uint32_t hp = bl.seq_hdr, sb = bl.seq_bits;
            if (!hp || opos + hp + sb >= len + 3) raw_block = true;
            else {
                const uint8_t* sec = a.seqsec + (size_t)b * ZKC_SEQSEC;
                for (uint32_t i = lane; i < hp; i += 32) out[opos + i] = sec[i];
                opos += hp;
                for (uint32_t i = lane; i < sb; i += 32) out[opos + i] = sec[ZKC_SEQHDR + i];
                opos += sb;
            }
        }
    }
    if (!raw_block && opos >= len + 3) raw_block = true;
    if (raw_block) {
        for (uint32_t i = lane; i < len; i += 32) out[3 + i] = a.src[lo + i];
        opos = 3 + len;
    }
    if (lane == 0) {
        uint32_t bh = bl.last_flag | ((raw_block ? 0u : 2u) << 1) | ((raw_block ? len : opos - 3) << 3);
        out[0] = (uint8_t)bh; out[1] = (uint8_t)(bh >> 8); out[2] = (uint8_t)(bh >> 16);
        a.blocks[b].csize = opos;
    }
}

// =============================================================================================
// K-C3: frame layout + gather
// =============================================================================================
// XXH64 (A.8) of each frame's input, one warp per frame (zk_warp_xxh64: coalesced loads, products off the chain)
__global__ void __launch_bounds__(128) zk_frame_hash_kernel(ZkEncodeArgs a) {
    const int lane = threadIdx.x & 31;
    const uint32_t f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (f >= a.n_frames) return;
    const size_t fstart = (size_t)f * a.frame_size;
    const size_t fend = fstart + a.frame_size < a.n ? fstart + a.frame_size : a.n;
    const uint8_t* p = a.src + fstart; const uint32_t len = (uint32_t)(fend - fstart);
    const unsigned long long h = zk_warp_xxh64(p, len, lane);
    if (lane == 0) a.frame_hash[f] = (uint32_t)h;
}

// per-frame sizes and per-block offsets (one thread per frame), then a single-CTA scan for the frame offsets
__global__ void __launch_bounds__(256) zk_frame_size_kernel(ZkEncodeArgs a) {
    const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= a.n_frames) return;
    uint32_t off = ZKC_FRAME_HDR;
    for (uint32_t k = 0; k < a.blocks_per_frame; k++) {
        ZkcBlock& bl = a.blocks[(size_t)f * a.blocks_per_frame + k];
        bl.out_off = off; off += bl.csize;
    }
    if (a.checksum) off += 4;
    a.frame_csize[f] = off;
}

__global__ void __launch_bounds__(1024) zk_frame_scan_kernel(ZkEncodeArgs a) {
    __shared__ unsigned long long part[1024];
    __shared__ unsigned long long carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < a.n_frames; base += 1024) {
        const uint32_t f = base + threadIdx.x;
        unsigned long long v = f < a.n_frames ? a.frame_csize[f] : 0;
        part[threadIdx.x] = v;
        __syncthreads();
        for (uint32_t d = 1; d < 1024; d <<= 1) {
            unsigned long long t = threadIdx.x >= d ? part[threadIdx.x - d] : 0;
            __syncthreads();
            part[threadIdx.x] += t;
            __syncthreads();
        }
        if (f < a.n_frames) a.frame_off[f] = carry + part[threadIdx.x] - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry += part[1023];
        __syncthreads();
    }
    if (threadIdx.x == 0) { *a.total = carry; if (carry > a.dst_cap) *a.error = ZKZ_DST_TOO_SMALL; }
}

// wide-history tier only: the frame headers written by zk_frame_gather_kernel announce a 128 KiB window; offsets of this tier reach
// (ZKC_WIDE_HIST + 1) blocks back, so the Window_Descriptor becomes 256 KiB (exponent 8, mantissa 0)
__global__ void __launch_bounds__(128) zk_frame_window_kernel(ZkEncodeArgs a, uint32_t n_frames) {
    const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_frames || *a.error) return;
    a.dst[a.frame_off[f] + 5] = 0x40;
}

// ZK_C_WINDOW_LOG / long-distance matching: the Window_Descriptor of every frame becomes 2^log (exponent log - 10, mantissa 0)
__global__ void __launch_bounds__(128) zk_frame_wlog_kernel(ZkEncodeArgs a, uint32_t n_frames, uint32_t log) {
    const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_frames || *a.error) return;
    a.dst[a.frame_off[f] + 5] = (uint8_t)((log - 10u) << 3);
}

// long-distance matching: the index of the prefix.  One thread per sampled position q (every ZK_LDM_STRIDE-th position from q0 on);
// atomicMax keeps the highest position per slot whatever the schedule, so the table -- and the compressed bytes -- are deterministic
__global__ void __launch_bounds__(256) zk_ldm_index_kernel(const uint8_t* prefix, uint32_t q0, uint32_t count, uint32_t* tab, uint32_t log) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const uint32_t q = q0 + i * ZK_LDM_STRIDE;
    atomicMax(&tab[zkc_ldm_hash(zkc_ld8(prefix + q), log)], q + 1u);
}

// gather: one warp per block copies its staged bytes to the final position; block 0 of a frame also writes the
// frame header, the last block the checksum
__global__ void __launch_bounds__(128) zk_frame_gather_kernel(ZkEncodeArgs a) {
    const int lane = threadIdx.x & 31;
    const uint32_t b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= a.n_blocks || *a.error) return;
    const uint32_t f = b / a.blocks_per_frame, k = b % a.blocks_per_frame;
    const ZkcBlock bl = a.blocks[b];
    uint8_t* fo = a.dst + a.frame_off[f];
    if (k == 0 && lane == 0) {
        const size_t fstart = (size_t)f * a.frame_size;
        const size_t fend = fstart + a.frame_size < a.n ? fstart + a.frame_size : a.n;
        const uint32_t fcs = (uint32_t)(fend - fstart);
        fo[0] = 0x28; fo[1] = 0xB5; fo[2] = 0x2F; fo[3] = 0xFD;
        fo[4] = (uint8_t)(0x80 | (a.checksum ? 0x04 : 0));       // FCS 4 bytes, no single segment, no dict
        fo[5] = 0x38;                                             // window 128 KiB (log 17): offsets stay below 64 KiB
        fo[6] = (uint8_t)fcs; fo[7] = (uint8_t)(fcs >> 8); fo[8] = (uint8_t)(fcs >> 16); fo[9] = (uint8_t)(fcs >> 24);
        if (a.checksum) {
            const uint32_t h = a.frame_hash[f]; uint8_t* c = fo + a.frame_csize[f] - 4;
            c[0] = (uint8_t)h; c[1] = (uint8_t)(h >> 8); c[2] = (uint8_t)(h >> 16); c[3] = (uint8_t)(h >> 24);
        }
    }
    const uint8_t* s = a.stage + (size_t)b * ZKC_SLOT; uint8_t* d = fo + bl.out_off;
    const uint32_t n = bl.csize;
    // staged slots are 16-byte aligned; destinations are arbitrary -> byte-granular head, 16-byte body when co-aligned
    uint32_t head = (uint32_t)((16 - ((uintptr_t)d & 15)) & 15); if (head > n) head = n;
    if (lane < (int)head) d[lane] = s[lane];
    const uint8_t* s2 = s + head; uint8_t* d2 = d + head; const uint32_t n2 = n - head, nvec = n2 >> 4;
    const uint32_t mis = (uint32_t)((uintptr_t)s2 & 3);
    const uint32_t* sa = (const uint32_t*)(s2 - mis); const uint32_t sh = mis * 8;
    for (uint32_t i = lane; i < nvec; i += 32) {
        const uint32_t* q = sa + 4 * i;
        uint32_t w0 = q[0], w1 = q[1], w2 = q[2], w3 = q[3], w4 = mis ? q[4] : 0;
        ((uint4*)d2)[i] = mis ? make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh), __funnelshift_r(w3, w4, sh))
                              : make_uint4(w0, w1, w2, w3);
    }
    for (uint32_t i = (nvec << 4) + lane; i < n2; i += 32) d2[i] = s2[i];
}

// =============================================================================================
// host-side launcher
// =============================================================================================
#ifndef ZK_EMUL
#define ZKC_CUDA_OK(x) do { cudaError_t err__ = (x); if (err__ != cudaSuccess) { zk_note_cuda_error(#x, (int)err__); return ZK_INT_CUDA; } } while (0)
#else
#define ZKC_CUDA_OK(x) do { (void)(x); } while (0)
#endif

uint32_t zk_encode_level_window_log(int level) { return (level <= 0 ? 3 : level) >= ZKC_WIDE_LEVEL ? 18u : 17u; }

// about one slot per sampled position, at least 2^12 and at most 2^26 slots (256 MiB, a 1 GiB window)
uint32_t zk_ldm_index_log(size_t span) {
    const size_t samples = span / ZK_LDM_STRIDE + 1;
    uint32_t log = 12;
    while (log < 26 && ((size_t)1 << log) < samples) log++;
    return log;
}

int zk_ldm_index_build(cudaStream_t stream, const uint8_t* d_prefix, uint32_t prefix_len, uint32_t win, uint32_t* d_tab, uint32_t log) {
    ZKC_CUDA_OK(cudaMemsetAsync(d_tab, 0, sizeof(uint32_t) << log, stream));
    if (prefix_len < 8) return 0;
    const uint32_t lo = prefix_len > win ? prefix_len - win : 0u;
    const uint32_t q0 = (lo + ZK_LDM_STRIDE - 1) / ZK_LDM_STRIDE * ZK_LDM_STRIDE;
    if (q0 > prefix_len - 8) return 0;
    const uint32_t count = (prefix_len - 8 - q0) / ZK_LDM_STRIDE + 1;
    ZK_LAUNCH(zk_ldm_index_kernel, (count + 255) / 256, 256, 0, stream, d_prefix, q0, count, d_tab, log);
    return 0;
}

size_t zk_encode_bound(size_t n, uint32_t frame_size) {
    if (frame_size == 0) frame_size = 1;
    size_t frames = n / frame_size + 1;
    size_t blocks = n / ZKC_BLOCK + frames + 1;
    return n + frames * (ZKC_FRAME_HDR + 4) + blocks * 3 + 64;
}

void zk_encode_ws_free(ZkEncodeWs* ws) {
    if (ws->buf) cudaFree(ws->buf);
    if (ws->h_sizes) cudaFreeHost(ws->h_sizes);
    if (ws->side) cudaStreamDestroy(ws->side);
    if (ws->ev_a) cudaEventDestroy(ws->ev_a);
    if (ws->ev_b) cudaEventDestroy(ws->ev_b);
    if (ws->ev_c) cudaEventDestroy(ws->ev_c);
    ws->prof.destroy();
    *ws = ZkEncodeWs();
}

static size_t zkc_align(size_t v) { return (v + 255) & ~(size_t)255; }

int zk_encode_enqueue(ZkEncodeWs* ws, cudaStream_t stream, const uint8_t* d_src, size_t n, uint32_t frame_size, int level,
                      int checksum, uint8_t* d_dst, size_t dst_cap, uint32_t n_frames) {
    const uint8_t* d_prefix = ws->prefix; const uint32_t prefix_len = ws->prefix_len;     // one-shot (set by the caller for THIS batch)
    const uint32_t* ldm_tab = ws->ldm_tab; const uint32_t ldm_log = ws->ldm_log;
    ws->prefix = nullptr; ws->prefix_len = 0; ws->ldm_tab = nullptr; ws->ldm_log = 0;
    ws->pending_frames = 0;
    if (n_frames == 0) return 0;
    if (frame_size == 0 || frame_size > 0x40000000u) return -(int)ZKZ_PARAM_OUT_OF_BOUND;
    const size_t eff = n < frame_size ? n : frame_size;          // a lone short frame needs fewer block slots
    uint32_t bpf = (uint32_t)((eff + ZKC_BLOCK - 1) / ZKC_BLOCK); if (bpf == 0) bpf = 1;
    const size_t n_blocks = (size_t)n_frames * bpf;
    if (n_blocks > 0x7FFFFFFFull) return -(int)ZKZ_PARAM_OUT_OF_BOUND;
    // carve the workspace
    size_t off = 0;
    const size_t o_blocks = off; off = zkc_align(off + n_blocks * sizeof(ZkcBlock));
    const size_t o_ll = off; off = zkc_align(off + n_blocks * ZKC_MAXSEQ * 2);
    const size_t o_ml = off; off = zkc_align(off + n_blocks * ZKC_MAXSEQ * 2);
    const size_t o_off = off; off = zkc_align(off + n_blocks * ZKC_MAXSEQ * 4);
    const size_t o_lits = off; off = zkc_align(off + n_blocks * ZKC_BLOCK);
    const size_t o_stage = off; off = zkc_align(off + n_blocks * ZKC_SLOT + 64);
    const size_t o_seqsec = off; off = zkc_align(off + n_blocks * ZKC_SEQSEC);
    const size_t o_fcs = off; off = zkc_align(off + (size_t)n_frames * 4);
    const size_t o_foff = off; off = zkc_align(off + (size_t)n_frames * 8);
    const size_t o_fh = off; off = zkc_align(off + (size_t)n_frames * 4);
    const size_t o_tot = off; off = zkc_align(off + 16);
    const size_t o_pst = off; if (d_prefix && prefix_len && n) off = zkc_align(off + (size_t)n_frames * ZKC_PSLOT);
    if (ws->cap < off) {
        if (ws->buf) cudaFree(ws->buf);
        ws->buf = nullptr; ws->cap = 0;
        size_t want = off + off / 8;
        if (cudaMalloc(&ws->buf, want) != cudaSuccess) return -(int)ZKZ_MEMORY_ALLOCATION;
        ws->cap = want;
    }
    if (ws->cap_frames < n_frames) {
        if (ws->h_sizes) cudaFreeHost(ws->h_sizes);
        ws->h_sizes = nullptr;
        size_t want = (size_t)n_frames + n_frames / 8 + 16;
        if (cudaMallocHost((void**)&ws->h_sizes, want * 4 + 32) != cudaSuccess) return -(int)ZKZ_MEMORY_ALLOCATION;
        ws->cap_frames = want;
    }
    uint8_t* base = (uint8_t*)ws->buf;
    ZkEncodeArgs a;
    a.src = d_src; a.n = n; a.frame_size = frame_size; a.n_frames = n_frames; a.blocks_per_frame = bpf; a.n_blocks = (uint32_t)n_blocks;
    a.level = level <= 0 ? 3 : level; a.checksum = checksum ? 1 : 0;
    a.blocks = (ZkcBlock*)(base + o_blocks);
    a.seq_ll = (uint16_t*)(base + o_ll); a.seq_ml = (uint16_t*)(base + o_ml); a.seq_off = (uint32_t*)(base + o_off);
    a.lits = base + o_lits; a.stage = base + o_stage; a.seqsec = base + o_seqsec;
    a.frame_csize = (uint32_t*)(base + o_fcs); a.frame_off = (unsigned long long*)(base + o_foff); a.frame_hash = (uint32_t*)(base + o_fh);
    a.dst = d_dst; a.dst_cap = dst_cap; a.total = (unsigned long long*)(base + o_tot); a.error = (uint32_t*)(base + o_tot + 8);
    a.prefix = d_prefix; a.prefix_len = 0; a.ptail = 0; a.pstage = base + o_pst;
    // announced window: the level's own, raised to 2^win_log; the LDM flavour of K-C1 keeps every offset within it
    const uint32_t tier_log = zk_encode_level_window_log(a.level);
    const uint32_t win_log = ws->win_log > tier_log ? ws->win_log : tier_log;
    const bool ldm = ldm_tab && d_prefix && prefix_len && n;
    a.ldm_tab = ldm ? ldm_tab : nullptr; a.ldm_log = ldm ? ldm_log : 0; a.ldm_win = 1u << win_log;
    if (d_prefix && prefix_len && n) {
        a.prefix_len = prefix_len; a.ptail = prefix_len < ZKC_BLOCK ? prefix_len : ZKC_BLOCK;
        ZK_LAUNCH(zk_prefix_stage_kernel, n_frames, 256, 0, stream, a);
        ws->launches += 1;
    }
    ZKC_CUDA_OK(cudaMemsetAsync(base + o_tot, 0, 16, stream));
    // the content checksum only needs the input: it runs beside the match finder on the side stream (one warp per frame, bound
    // by the latency of its four serial chains, so it leaves the machine to K-C1)
    cudaStream_t ss = stream;
    if (!ws->no_side) {
        if (!ws->side) {
            ZKC_CUDA_OK(cudaStreamCreateWithPriority(&ws->side, cudaStreamNonBlocking, ws->prio));
            ZKC_CUDA_OK(cudaEventCreateWithFlags(&ws->ev_a, cudaEventDisableTiming));
            ZKC_CUDA_OK(cudaEventCreateWithFlags(&ws->ev_b, cudaEventDisableTiming));
            ZKC_CUDA_OK(cudaEventCreateWithFlags(&ws->ev_c, cudaEventDisableTiming));
        }
        ss = ws->side;
    }
    if (checksum && ss != stream) {
        ZKC_CUDA_OK(cudaEventRecord(ws->ev_c, stream)); ZKC_CUDA_OK(cudaStreamWaitEvent(ss, ws->ev_c, 0));     // after whatever produced the input
        ZK_LAUNCH(zk_frame_hash_kernel, (n_frames + 3) / 4, 128, 0, ss, a);
    }
    ws->prof.begin(5, stream);
    // six tiers (EncodeOptions::compression_level, encode.rs:176): 1 = 2048-entry table, no history, no lazy step; 2-3 = 4096 entries,
    // previous-block history, one lazy step; 4-6 = double table (8-byte + 5-byte hashes, 4096 entries each), two warps per CTA; 7-9 = double
    // table of 8192 entries each, one warp per CTA; 10-12 = one table of 16384 entries, one warp per CTA; >= 13 = 256 KiB history, 32768 x u32
    // entries in dynamic shared memory.  Ratio on the reference's corpus: 2.12 / 2.24 / 2.28 / 2.38 / 2.40 / 2.50 (profiles/ratio_dickens_r2.json)
    if (ldm) {
        if (a.level <= 1) ZK_LAUNCH((zk_match_kernel<ZKC_HLOG_FAST, ZKC_C1_WARPS, false, true>), (uint32_t)((n_blocks + ZKC_C1_WARPS - 1) / ZKC_C1_WARPS), ZKC_C1_WARPS * 32, 0, stream, a);
        else if (a.level <= 3) ZK_LAUNCH((zk_match_kernel<ZKC_HLOG, ZKC_C1_WARPS, false, true>), (uint32_t)((n_blocks + ZKC_C1_WARPS - 1) / ZKC_C1_WARPS), ZKC_C1_WARPS * 32, 0, stream, a);
        else if (a.level <= 6) ZK_LAUNCH((zk_match_kernel<ZKC_HLOG, 2, true, true>), (uint32_t)((n_blocks + 1) / 2), 64, 0, stream, a);
        else if (a.level <= 9) ZK_LAUNCH((zk_match_kernel<13, 1, true, true>), (uint32_t)n_blocks, 32, 0, stream, a);
        else if (a.level < ZKC_WIDE_LEVEL) ZK_LAUNCH((zk_match_kernel<14, 1, false, true>), (uint32_t)n_blocks, 32, 0, stream, a);
        else {
            const int wide_smem = (int)sizeof(uint32_t) << ZKC_WIDE_HLOG;
            if (!ws->attr_set_wide_ldm) { ZKC_CUDA_OK(cudaFuncSetAttribute(zk_match_wide_kernel<ZKC_WIDE_HLOG, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, wide_smem)); ws->attr_set_wide_ldm = true; }
            ZK_LAUNCH((zk_match_wide_kernel<ZKC_WIDE_HLOG, true>), (uint32_t)n_blocks, 32, wide_smem, stream, a);
        }
    }
    else if (a.level <= 1) ZK_LAUNCH((zk_match_kernel<ZKC_HLOG_FAST, ZKC_C1_WARPS, false>), (uint32_t)((n_blocks + ZKC_C1_WARPS - 1) / ZKC_C1_WARPS), ZKC_C1_WARPS * 32, 0, stream, a);
    else if (a.level <= 3) ZK_LAUNCH((zk_match_kernel<ZKC_HLOG, ZKC_C1_WARPS, false>), (uint32_t)((n_blocks + ZKC_C1_WARPS - 1) / ZKC_C1_WARPS), ZKC_C1_WARPS * 32, 0, stream, a);
    else if (a.level <= 6) ZK_LAUNCH((zk_match_kernel<ZKC_HLOG, 2, true>), (uint32_t)((n_blocks + 1) / 2), 64, 0, stream, a);
    else if (a.level <= 9) ZK_LAUNCH((zk_match_kernel<13, 1, true>), (uint32_t)n_blocks, 32, 0, stream, a);
    else if (a.level < ZKC_WIDE_LEVEL) ZK_LAUNCH((zk_match_kernel<14, 1, false>), (uint32_t)n_blocks, 32, 0, stream, a);
    else {
        const int wide_smem = (int)sizeof(uint32_t) << ZKC_WIDE_HLOG;
        if (!ws->attr_set_wide) { ZKC_CUDA_OK(cudaFuncSetAttribute(zk_match_wide_kernel<ZKC_WIDE_HLOG>, cudaFuncAttributeMaxDynamicSharedMemorySize, wide_smem)); ws->attr_set_wide = true; }
        ZK_LAUNCH((zk_match_wide_kernel<ZKC_WIDE_HLOG>), (uint32_t)n_blocks, 32, wide_smem, stream, a);
    }
    ws->prof.end(5, stream);
    const size_t seq_smem = ((sizeof(ZkcTabs) + 15) & ~(size_t)15) + sizeof(ZkcSeqWarp) * ZKC_SW;
    if (!ws->attr_set) { ZKC_CUDA_OK(cudaFuncSetAttribute(zk_seq_enc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)seq_smem)); ws->attr_set = true; }
    // the two entropy kernels are independent and both latency-bound: run them side by side, join in zk_block_finish_kernel
    ws->prof.begin(6, stream);
    if (ss != stream) { ZKC_CUDA_OK(cudaEventRecord(ws->ev_a, stream)); ZKC_CUDA_OK(cudaStreamWaitEvent(ss, ws->ev_a, 0)); }
    ZK_LAUNCH(zk_seq_enc_kernel, (uint32_t)((n_blocks + ZKC_SW - 1) / ZKC_SW), 32 * ZKC_SW, seq_smem, ss, a);
    if (ss != stream) ZKC_CUDA_OK(cudaEventRecord(ws->ev_b, ss));
    ZK_LAUNCH(zk_lit_enc_kernel, (uint32_t)n_blocks, 32, 0, stream, a);
    if (ss != stream) ZKC_CUDA_OK(cudaStreamWaitEvent(stream, ws->ev_b, 0));
    ZK_LAUNCH(zk_block_finish_kernel, (uint32_t)((n_blocks + 3) / 4), 128, 0, stream, a);
    ws->prof.end(6, stream);
    ws->prof.begin(7, stream);
    if (checksum && ss == stream) ZK_LAUNCH(zk_frame_hash_kernel, (n_frames + 3) / 4, 128, 0, stream, a);   // else: already done on the side stream (joined by ev_b)
    ZK_LAUNCH(zk_frame_size_kernel, (n_frames + 255) / 256, 256, 0, stream, a);
    ZK_LAUNCH(zk_frame_scan_kernel, 1, 1024, 0, stream, a);
    ZK_LAUNCH(zk_frame_gather_kernel, (uint32_t)((n_blocks + 3) / 4), 128, 0, stream, a);
    if (a.level >= ZKC_WIDE_LEVEL) { ZK_LAUNCH(zk_frame_window_kernel, (n_frames + 127) / 128, 128, 0, stream, a, n_frames); ws->launches++; }
    if (win_log > tier_log) { ZK_LAUNCH(zk_frame_wlog_kernel, (n_frames + 127) / 128, 128, 0, stream, a, n_frames, win_log); ws->launches++; }
    ws->prof.end(7, stream);
    ZKC_CUDA_OK(cudaMemcpyAsync(ws->h_sizes, a.frame_csize, (size_t)n_frames * 4, cudaMemcpyDeviceToHost, stream));
    ZKC_CUDA_OK(cudaMemcpyAsync(ws->h_sizes + ws->cap_frames, a.total, 16, cudaMemcpyDeviceToHost, stream));
    ws->launches += 7 + (checksum ? 1 : 0);
    ws->pending_frames = n_frames;
    return 0;
}

int zk_encode_collect(ZkEncodeWs* ws, cudaStream_t stream, uint32_t* c_sizes, size_t* dst_len) {
    const uint32_t nf = ws->pending_frames;
    if (nf == 0) { if (dst_len) *dst_len = 0; return 0; }
    ZKC_CUDA_OK(cudaStreamSynchronize(stream));
#ifndef ZK_EMUL
    { cudaError_t le__ = cudaGetLastError(); if (le__ != cudaSuccess) { zk_note_cuda_error("kernel launch / execution", (int)le__); return ZK_INT_CUDA; } }
#endif
    ws->pending_frames = 0;
    ws->prof.harvest();
    unsigned long long total; uint32_t err;
    memcpy(&total, ws->h_sizes + ws->cap_frames, 8);
    memcpy(&err, (uint8_t*)(ws->h_sizes + ws->cap_frames) + 8, 4);
    if (err) return -(int)err;
    if (c_sizes) memcpy(c_sizes, ws->h_sizes, (size_t)nf * 4);
    if (dst_len) *dst_len = (size_t)total;
    return 0;
}

int zk_encode_batch(ZkEncodeWs* ws, cudaStream_t stream, const uint8_t* d_src, size_t n, uint32_t frame_size, int level,
                    int checksum, uint8_t* d_dst, size_t dst_cap, uint32_t* c_sizes, uint32_t n_frames, size_t* dst_len) {
    int rc = zk_encode_enqueue(ws, stream, d_src, n, frame_size, level, checksum, d_dst, dst_cap, n_frames);
    if (rc) return rc;
    return zk_encode_collect(ws, stream, c_sizes, dst_len);
}
