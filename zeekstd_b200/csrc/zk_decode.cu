// zk_decode.cu -- batched Zstandard frame decode for sm_100a.
//
// Replaces the reference's only decompression call into libzstd,
//   lib/src/decode.rs:243-245   self.dctx.decompress_stream(&mut out_buffer, &mut in_buffer)
// with four kernels over a whole batch of independent seek-table entries ("frames" of the
// seekable format, seekable_format.md:23-29):
//
//   K-D0 zk_scan_kernel     one thread / entry : walk frame + block headers, carve scratch
//   K-D1s zk_seq_kernel     one LANE  / block  : FSE sequence decode (4-byte cells + state machine in smem)
//   K-D1h zk_huf_kernel     one LANE  / stream : Huffman literal decode (4 lanes per 4-stream block, two-level table)
//   K-D2 zk_exec_kernel[_w5] one CTA  / entry  : ordered sequence execution through a shared-memory window
//   K-D3 zk_xxh64_kernel    one warp  / entry  : content checksum (only if requested & present)
//
// Format rules: RFC 8878 as restated in SURVEY.md Appendix A (the arithmetic is not in the
// reference tree).  All integer/byte work; no tensor cores.
#include "zk_common.cuh"
#include "zk_decode.h"
#include <stdio.h>
#include <stdlib.h>

// =============================================================================================
// K-D0: header scan
// =============================================================================================
struct ZkBlkInfo {
    uint32_t src, size; uint8_t type, flags;
    uint32_t lit_size, nseq, bmax; uint8_t lit_type, modes, lit_hdr; uint64_t fcs;
};

struct ZkLitHdr { uint32_t type, hdr, regen, comp, streams; };

// Literals_Section_Header (A.3).  n = bytes available. Returns false if truncated.
__device__ __forceinline__ bool zk_parse_lit_hdr(const uint8_t* p, uint32_t n, ZkLitHdr& h) {
    if (n < 1) return false;
    uint32_t b0 = p[0];
    h.type = b0 & 3; uint32_t sf = (b0 >> 2) & 3;
    h.comp = 0; h.streams = 1;
    if (h.type < 2) {
        if (sf == 0 || sf == 2) { h.hdr = 1; h.regen = b0 >> 3; }
        else if (sf == 1) { if (n < 2) return false; h.hdr = 2; h.regen = (b0 >> 4) | ((uint32_t)p[1] << 4); }
        else { if (n < 3) return false; h.hdr = 3; h.regen = (b0 >> 4) | ((uint32_t)p[1] << 4) | ((uint32_t)p[2] << 12); }
    } else {
        if (n < 5) return false;
        unsigned long long v = (unsigned long long)zk_ld_le32(p) | ((unsigned long long)p[4] << 32);
        if (sf == 0) { h.hdr = 3; h.streams = 1; h.regen = (uint32_t)(v >> 4) & 0x3FF; h.comp = (uint32_t)(v >> 14) & 0x3FF; }
        else if (sf == 1) { h.hdr = 3; h.streams = 4; h.regen = (uint32_t)(v >> 4) & 0x3FF; h.comp = (uint32_t)(v >> 14) & 0x3FF; }
        else if (sf == 2) { h.hdr = 4; h.streams = 4; h.regen = (uint32_t)(v >> 4) & 0x3FFF; h.comp = (uint32_t)(v >> 18) & 0x3FFF; }
        else { h.hdr = 5; h.streams = 4; h.regen = (uint32_t)(v >> 4) & 0x3FFFF; h.comp = (uint32_t)(v >> 22) & 0x3FFFF; }
    }
    return true;
}
__device__ __forceinline__ uint32_t zk_lit_section_size(const ZkLitHdr& h) {
    return h.hdr + (h.type == 0 ? h.regen : h.type == 1 ? 1u : h.comp);
}

// Sequences_Section_Header (A.5): number of sequences.  Returns header bytes (1..3) or 0 if truncated.
__device__ __forceinline__ uint32_t zk_parse_nseq(const uint8_t* s, uint32_t n, uint32_t& nseq) {
    if (n < 1) return 0;
    uint32_t b0 = s[0];
    if (b0 < 128) { nseq = b0; return 1; }
    if (b0 < 255) { if (n < 2) return 0; nseq = ((b0 - 128) << 8) + s[1]; return 2; }
    if (n < 3) return 0;
    nseq = (uint32_t)s[1] + ((uint32_t)s[2] << 8) + 0x7F00u; return 3;
}

// Walks every zstd / skippable frame inside one seek-table entry.  emit(info) is called per block.
template <class Emit>
__device__ int zk_walk_entry(const uint8_t* p, uint32_t n, Emit& emit, unsigned long long win_max) {
    uint32_t pos = 0;
    while (pos < n) {
        if (n - pos < 4) return ZKZ_SRC_SIZE_WRONG;
        uint32_t magic = zk_ld_le32(p + pos);
        if ((magic & ZK_SKIPPABLE_MASK) == ZK_SKIPPABLE_MAGIC) {
            if (n - pos < 8) return ZKZ_SRC_SIZE_WRONG;
            uint32_t sz = zk_ld_le32(p + pos + 4);
            if ((unsigned long long)sz + 8ull > (unsigned long long)(n - pos)) return ZKZ_SRC_SIZE_WRONG;
            pos += 8 + sz;
            continue;
        }
        if (magic != ZK_MAGIC) return ZKZ_PREFIX_UNKNOWN;
        if (n - pos < 5) return ZKZ_SRC_SIZE_WRONG;
        uint32_t fhd = p[pos + 4];
        uint32_t fcs_flag = fhd >> 6, single = (fhd >> 5) & 1, csum = (fhd >> 2) & 1, did = fhd & 3;
        if (fhd & 0x08) return ZKZ_FRAMEPARAM_UNSUPPORTED;
        uint32_t did_sz = did == 3 ? 4u : did;
        uint32_t fcs_sz = fcs_flag == 0 ? single : (fcs_flag == 1 ? 2u : (fcs_flag == 2 ? 4u : 8u));
        uint32_t hsz = 5 + (single ? 0 : 1) + did_sz + fcs_sz;
        if (n - pos < hsz) return ZKZ_SRC_SIZE_WRONG;
        uint32_t q = pos + 5;
        unsigned long long window = 0;
        if (!single) {
            const uint32_t wd = p[q++], wlog = 10 + (wd >> 3);
            if (wlog > 31) return ZKZ_WINDOW_TOO_LARGE;                  // ZSTD_WINDOWLOG_MAX, refused while the header is parsed
            window = (1ull << wlog) + ((1ull << wlog) >> 3) * (wd & 7);
        }
        uint32_t dict = 0;
        for (uint32_t i = 0; i < did_sz; i++) dict |= (uint32_t)p[q + i] << (8 * i);
        q += did_sz;
        if (dict != 0) return ZKZ_DICT_WRONG;
        unsigned long long fcs = 0;
        for (uint32_t i = 0; i < fcs_sz; i++) fcs |= (unsigned long long)p[q + i] << (8 * i);
        if (fcs_sz == 2) fcs += 256;
        // the reference decodes with a default DCtx (decode.rs:130-133): streaming decompression refuses windows above
        // 2^ZSTD_WINDOWLOG_LIMIT_DEFAULT (+1), after the dictionary check -- a Single_Segment frame's window is its content size.
        // ZK_D_WINDOW_LOG_MAX moves the limit to 2^value, as ZSTD_d_windowLogMax does
        if (single) window = fcs;
        if (window > win_max) return ZKZ_WINDOW_TOO_LARGE;
        // Block_Maximum_Size = min(Window_Size, 128 KiB) (RFC 8878 3.1.1.2.3): libzstd refuses a block whose content or
        // regenerated size exceeds it (ZSTD_decompressContinue: "Block Size Exceeds Maximum", "Decompressed Block Size Exceeds Maximum")
        const uint32_t bsmax = window < ZK_BLOCK_MAX ? (uint32_t)window : ZK_BLOCK_MAX;
        pos += hsz;
        bool first = true;
        for (;;) {
            if (n - pos < 3) return ZKZ_SRC_SIZE_WRONG;
            uint32_t bh = zk_ld_le24(p + pos);
            uint32_t last = bh & 1, type = (bh >> 1) & 3, bsize = bh >> 3;
            if (type == 3) return ZKZ_CORRUPTION;
            if (bsize > bsmax) return ZKZ_CORRUPTION;
            uint32_t content = type == 1 ? 1u : bsize;
            if (n - pos - 3 < content) return ZKZ_SRC_SIZE_WRONG;
            ZkBlkInfo bi;
            bi.src = pos + 3; bi.size = bsize; bi.type = (uint8_t)type;
            bi.flags = (uint8_t)((first ? ZKB_FIRST : 0) | (last ? ZKB_LAST : 0) | ((last && csum) ? ZKB_HAS_CSUM : 0) |
                                 ((last && fcs_sz) ? ZKB_HAS_FCS : 0));
            bi.fcs = fcs; bi.bmax = bsmax; bi.lit_size = 0; bi.nseq = 0; bi.lit_type = 0; bi.modes = 0; bi.lit_hdr = 0;
            if (type == 2) {
                const uint8_t* b = p + pos + 3;
                if (bsize < 2) return ZKZ_CORRUPTION;
                ZkLitHdr lh;
                if (!zk_parse_lit_hdr(b, bsize, lh)) return ZKZ_CORRUPTION;
                if (lh.regen > bsmax) return ZKZ_CORRUPTION;
                uint32_t lsec = zk_lit_section_size(lh);
                if (lsec >= bsize) return ZKZ_CORRUPTION;          // at least the nseq byte must follow
                uint32_t nseq;
                uint32_t sh = zk_parse_nseq(b + lsec, bsize - lsec, nseq);
                if (sh == 0) return ZKZ_CORRUPTION;
                if (nseq == 0) { if (lsec + sh != bsize) return ZKZ_CORRUPTION; }
                else {
                    if (lsec + sh >= bsize) return ZKZ_CORRUPTION;
                    bi.modes = b[lsec + sh];
                    if (bi.modes & 3) return ZKZ_CORRUPTION;
                }
                bi.lit_size = lh.regen; bi.nseq = nseq; bi.lit_type = (uint8_t)lh.type; bi.lit_hdr = (uint8_t)lh.hdr;
            }
            int rc = emit(bi);
            if (rc) return rc;
            pos += 3 + content;
            first = false;
            if (last) break;
        }
        if (csum) { if (n - pos < 4) return ZKZ_SRC_SIZE_WRONG; pos += 4; }
    }
    return 0;
}

struct ZkCountEmit {
    uint32_t nb = 0, nlit = 0, nseq = 0, nhuf = 0, nsqb = 0;
    // Treeless literals / Repeat_Mode tables must refer to something defined earlier in the same zstd frame.  This is
    // checked HERE so that the fill pass (which reserves slots of huf_list / seq_list from these counts) cannot fail
    // after the count pass succeeded: every reserved work-list slot is always written.
    uint32_t have = 0;            // bit 0 Huffman tree, bits 1..3 LL / OF / ML table
    __device__ int operator()(const ZkBlkInfo& bi) {
        nb++;
        if (bi.flags & ZKB_FIRST) have = 0;
        if (bi.type == 2) {
            if (bi.lit_type == 3 && !(have & 1u)) return ZKZ_DICT_CORRUPTED;
            if (bi.lit_type == 2) have |= 1u;
            if (bi.lit_type >= 2) { nlit += (bi.lit_size + 15u) & ~15u; nhuf++; }
            if (bi.nseq) {
                const uint32_t ml_m = (bi.modes >> 2) & 3, of_m = (bi.modes >> 4) & 3, ll_m = (bi.modes >> 6) & 3;
                if (ll_m == 3) { if (!(have & 2u)) return ZKZ_CORRUPTION; } else have |= 2u;
                if (of_m == 3) { if (!(have & 4u)) return ZKZ_CORRUPTION; } else have |= 4u;
                if (ml_m == 3) { if (!(have & 8u)) return ZKZ_CORRUPTION; } else have |= 8u;
            }
            nseq += bi.nseq; nsqb += bi.nseq != 0;
        }
        return 0;
    }
};

struct ZkFillEmit {
    ZkBlock* blocks; const uint8_t* ebase; uint32_t* huf_list; uint32_t* seq_list; uint32_t entry, bidx, lit, seq, hufi, sqbi;
    int32_t huf_ref = -1, ll_ref = -1, of_ref = -1, ml_ref = -1;
    __device__ int operator()(const ZkBlkInfo& bi) {
        ZkBlock b;
        b.src = bi.src; b.size = bi.size; b.entry = entry; b.type = bi.type; b.flags = bi.flags;
        b.lit_kind = 0; b.lit_byte = 0; b.lit_base = lit; b.seq_base = seq; b.nseq = bi.nseq; b.lit_size = bi.lit_size;
        b.lit_src = 0; b.regen = bi.type == 2 ? 0 : bi.size; b.status = 0; b.lit_status = 0;
        b.rep_out[0] = ZK_SYM_MAKE(0, 0); b.rep_out[1] = ZK_SYM_MAKE(1, 0); b.rep_out[2] = ZK_SYM_MAKE(2, 0);
        b.fcs = bi.fcs; b.hash_start = 0; b.hash_len = 0; b.bmax = bi.bmax;
        if (bi.flags & ZKB_FIRST) { huf_ref = ll_ref = of_ref = ml_ref = -1; }
        b.huf_ref = -1; b.ll_ref = -1; b.of_ref = -1; b.ml_ref = -1;
        if (bi.type == 2) {
            if (bi.lit_type == 3) { if (huf_ref < 0) return ZKZ_DICT_CORRUPTED; b.huf_ref = huf_ref; }
            if (bi.lit_type == 2) huf_ref = (int32_t)bidx;
            if (bi.lit_type >= 2) { lit += (bi.lit_size + 15u) & ~15u; b.lit_kind = 2; huf_list[hufi++] = bidx; }
            else if (bi.lit_type == 0) { b.lit_kind = 0; b.lit_src = bi.src + bi.lit_hdr; }
            else { b.lit_kind = 1; b.lit_byte = ebase[bi.src + bi.lit_hdr]; }
            if (bi.nseq == 0) b.regen = bi.lit_size;         // literals-only block
            if (bi.nseq) {
                seq_list[sqbi++] = bidx;
                uint32_t ml_m = (bi.modes >> 2) & 3, of_m = (bi.modes >> 4) & 3, ll_m = (bi.modes >> 6) & 3;
                if (ll_m == 3) { if (ll_ref < 0) return ZKZ_CORRUPTION; b.ll_ref = ll_ref; } else ll_ref = (int32_t)bidx;
                if (of_m == 3) { if (of_ref < 0) return ZKZ_CORRUPTION; b.of_ref = of_ref; } else of_ref = (int32_t)bidx;
                if (ml_m == 3) { if (ml_ref < 0) return ZKZ_CORRUPTION; b.ml_ref = ml_ref; } else ml_ref = (int32_t)bidx;
                seq += bi.nseq;
            }
        }
        blocks[bidx++] = b;
        return 0;
    }
};

__global__ void __launch_bounds__(128) zk_scan_kernel(ZkDecodeArgs a) {
    uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= a.n_entries) return;
    ZkEntry ent; ent.first_block = 0; ent.n_blocks = 0; ent.status = 0; ent.produced = 0;
    unsigned long long c0 = a.c_off[e], c1 = a.c_off[e + 1];
    if (c1 < c0 || c1 - c0 > 0xFFFFFFFFull) { ent.status = -ZKZ_SRC_SIZE_WRONG; a.entries[e] = ent; return; }
    const uint8_t* p = a.comp + c0; uint32_t n = (uint32_t)(c1 - c0);
    ZkCountEmit ce;
    int rc = zk_walk_entry(p, n, ce, a.win_max);
    if (rc) { ent.status = -rc; atomicAdd(&a.counters->n_errors, 1u); a.entries[e] = ent; return; }
    unsigned long long b0 = atomicAdd(&a.counters->n_blocks, (unsigned long long)ce.nb);
    unsigned long long l0 = atomicAdd(&a.counters->n_lit, (unsigned long long)ce.nlit);
    unsigned long long s0 = atomicAdd(&a.counters->n_seq, (unsigned long long)ce.nseq);
    uint32_t h0 = atomicAdd(&a.counters->n_huf_blocks, ce.nhuf), q0 = atomicAdd(&a.counters->n_seq_blocks, ce.nsqb);
    if (b0 + ce.nb > a.cap_blocks || l0 + ce.nlit > a.cap_lit || s0 + ce.nseq > a.cap_seq) {
        atomicOr(&a.counters->overflow, 1u);
        ent.status = ZK_ST_RETRY; a.entries[e] = ent; return;
    }
    ZkFillEmit fe; fe.blocks = a.blocks; fe.entry = e; fe.bidx = (uint32_t)b0; fe.lit = (uint32_t)l0; fe.seq = (uint32_t)s0;
    fe.ebase = p; fe.huf_list = a.huf_list; fe.seq_list = a.seq_list; fe.hufi = h0; fe.sqbi = q0;   // lists have cap_blocks entries
    rc = zk_walk_entry(p, n, fe, a.win_max);
    ent.first_block = (uint32_t)b0; ent.n_blocks = ce.nb;
    if (rc) { ent.status = -rc; ent.n_blocks = 0; atomicAdd(&a.counters->n_errors, 1u); }
    a.entries[e] = ent;
}

// =============================================================================================
// K-D1s: FSE sequence decode -- one LANE per zstd block.
//
// A sequence bitstream is one serial dependency chain (three interleaved FSE states sharing one
// backward bit cursor, A.5), so the only parallelism is across blocks.  Profiling the first version
// (one block per CTA, one active lane per warp) showed the SMs issue-bound at 1/32 SIMT efficiency;
// here every lane of a warp runs the identical decode loop over ITS OWN block with ITS OWN tables
// in shared memory, so one issued instruction advances up to ZK_SEQ_LANES chains.
// =============================================================================================
#define ZK_SEQ_LPW 3              // chains per warp
#define ZK_SEQ_WARPS 3            // warps per CTA: 9 x 5.6 KiB of tables per CTA (4 CTAs / SM) spread over more warps --
#define ZK_SEQ_LANES (ZK_SEQ_LPW * ZK_SEQ_WARPS)   // each chain is ALU-latency bound, so more warps per SM hide more of it

// Thin decoding cell: one 32-bit shared-memory load yields everything on the dependency chain of a sequence (bits to
// skip, bits of the next state, next-state baseline); the value baselines come from small per-CTA tables by symbol code,
// off the chain.  (The first version used libzstd's 8-byte cell: 11.7 KiB of tables per chain, 18 chains per SM.)
//   [0,9) next-state baseline   [9,13) nbBits   [13,18) extra bits   [18,24) symbol code
#define ZK_CELL(code, add, nb, base) ((uint32_t)(base) | ((uint32_t)(nb) << 9) | ((uint32_t)(add) << 13) | ((uint32_t)(code) << 18))
#define ZK_CELL_BASE(c) ((c) & 511u)
#define ZK_CELL_NB(c) (((c) >> 9) & 15u)
#define ZK_CELL_ADD(c) (((c) >> 13) & 31u)
#define ZK_CELL_CODE(c) (((c) >> 18) & 63u)

struct ZkSeqSlot {
    uint32_t ll[512], ml[512], of[256];        // 5 KiB
    int16_t cnt[3][64];
    uint16_t nxt[64];
    int tbl_log[3], tbl_nsym[3], tbl_mode[3];  // mode: 0 = counts in cnt[t], 1 = RLE (cnt[t][0] = symbol)
};
struct ZkSeqTabs { uint32_t ll_base[36], ml_base[53]; };

// Locate the three table descriptions of a block (A.5) and parse those that are wanted into sl.cnt[t]
// (t: 0 LL, 1 OF, 2 ML).  Returns 0 or a zstd code.  *bits_off = start of the sequence bitstream.
__device__ int zk_locate_seq_tables(ZkSeqSlot& sl, const uint8_t* b, uint32_t bsize, bool w0, bool w1, bool w2, uint32_t* bits_off) {
    ZkLitHdr lh;
    if (!zk_parse_lit_hdr(b, bsize, lh)) return ZKZ_CORRUPTION;
    uint32_t lsec = zk_lit_section_size(lh);
    if (lsec >= bsize) return ZKZ_CORRUPTION;
    uint32_t nseq, sh = zk_parse_nseq(b + lsec, bsize - lsec, nseq);
    if (!sh || nseq == 0 || lsec + sh >= bsize) return ZKZ_CORRUPTION;
    uint32_t modes = b[lsec + sh], pos = lsec + sh + 1;
    for (int t = 0; t < 3; t++) {
        const bool want = t == 0 ? w0 : (t == 1 ? w1 : w2);
        const int max_log = t == 1 ? 8 : 9, max_sym = t == 0 ? 35 : (t == 1 ? 31 : 52);
        uint32_t m = (modes >> (6 - 2 * t)) & 3;
        if (m == 0) {
            if (want) {
                sl.tbl_mode[t] = 0;
                if (t == 0) { for (int i = 0; i < 36; i++) sl.cnt[0][i] = ZK_LL_DEFAULT[i]; sl.tbl_nsym[0] = 36; sl.tbl_log[0] = 6; }
                else if (t == 1) { for (int i = 0; i < 29; i++) sl.cnt[1][i] = ZK_OF_DEFAULT[i]; sl.tbl_nsym[1] = 29; sl.tbl_log[1] = 5; }
                else { for (int i = 0; i < 53; i++) sl.cnt[2][i] = ZK_ML_DEFAULT[i]; sl.tbl_nsym[2] = 53; sl.tbl_log[2] = 6; }
            }
        } else if (m == 1) {
            if (pos >= bsize) return ZKZ_CORRUPTION;
            if (want) {
                if (b[pos] > max_sym) return ZKZ_CORRUPTION;
                sl.tbl_mode[t] = 1; sl.cnt[t][0] = b[pos]; sl.tbl_log[t] = 0; sl.tbl_nsym[t] = 1;
            }
            pos += 1;
        } else if (m == 2) {
            int ns, lg;
            // an unwanted table is parsed into the (not yet used) nxt scratch just to learn its length
            uint32_t used = zk_fse_read_ncount(b + pos, bsize - pos, max_log, max_sym, want ? sl.cnt[t] : (int16_t*)sl.nxt, &ns, &lg);
            if (!used) return ZKZ_CORRUPTION;
            if (want) { sl.tbl_mode[t] = 0; sl.tbl_nsym[t] = ns; sl.tbl_log[t] = lg; }
            pos += used;
        } else {
            if (want) return ZKZ_CORRUPTION;   // Repeat is resolved through *_ref by the caller
        }
    }
    if (pos > bsize) return ZKZ_CORRUPTION;
    *bits_off = pos;
    return 0;
}

// Build one sequence decoding table from sl.cnt[t] (A.6).  The symbol spread is written into the cell array itself and
// converted to cells in place.
__device__ int zk_build_seq_table(ZkSeqSlot& sl, int t, uint16_t* nxt_scratch = nullptr) {
    uint32_t* cell = t == 0 ? sl.ll : (t == 1 ? sl.of : sl.ml);
    if (sl.tbl_mode[t] == 1) {
        const uint32_t sy = (uint32_t)sl.cnt[t][0];
        const uint32_t add = t == 0 ? ZK_LL_BITS[sy] : (t == 1 ? sy : ZK_ML_BITS[sy]);
        cell[0] = ZK_CELL(sy, add, 0, 0);
        return 0;
    }
    int log = sl.tbl_log[t], S = 1 << log, nsym = sl.tbl_nsym[t], high = S - 1;
    uint16_t* nxt = nxt_scratch ? nxt_scratch : sl.nxt; const int16_t* cnt = sl.cnt[t];
    for (int s = 0; s < nsym; s++) {
        if (cnt[s] == -1) { cell[high--] = (uint32_t)s; nxt[s] = 1; }
        else nxt[s] = (uint16_t)cnt[s];
    }
    int step = (S >> 1) + (S >> 3) + 3, pos = 0;
    for (int s = 0; s < nsym; s++)
        for (int q = 0; q < cnt[s]; q++) {
            cell[pos] = (uint32_t)s;
            do { pos = (pos + step) & (S - 1); } while (pos > high);
        }
    if (pos != 0) return ZKZ_CORRUPTION;
    for (int u = 0; u < S; u++) {
        const uint32_t sy = cell[u];
        const uint32_t x = nxt[sy]++;
        const int nb = log - zk_highbit(x);
        const uint32_t add = t == 0 ? ZK_LL_BITS[sy] : (t == 1 ? sy : ZK_ML_BITS[sy]);
        cell[u] = ZK_CELL(sy, add, nb, (x << nb) - (uint32_t)S);
    }
    return 0;
}

// Decode all sequences of one block (lane-local).  Returns 0 or a zstd code.
__device__ int zk_decode_block_sequences(ZkSeqSlot& sl, const ZkSeqTabs& tb, const ZkDecodeArgs& a, const ZkBlock& blk, uint32_t bidx, const uint8_t* ebase) {
    const uint8_t* b = ebase + blk.src;
    uint32_t bits_off = 0;
    int st = zk_locate_seq_tables(sl, b, blk.size, blk.ll_ref < 0, blk.of_ref < 0, blk.ml_ref < 0, &bits_off);
    if (st) return st;
    if (blk.ll_ref >= 0) { const ZkBlock& rb = a.blocks[blk.ll_ref]; uint32_t d; if ((st = zk_locate_seq_tables(sl, ebase + rb.src, rb.size, true, false, false, &d))) return st; }
    if (blk.of_ref >= 0) { const ZkBlock& rb = a.blocks[blk.of_ref]; uint32_t d; if ((st = zk_locate_seq_tables(sl, ebase + rb.src, rb.size, false, true, false, &d))) return st; }
    if (blk.ml_ref >= 0) { const ZkBlock& rb = a.blocks[blk.ml_ref]; uint32_t d; if ((st = zk_locate_seq_tables(sl, ebase + rb.src, rb.size, false, false, true, &d))) return st; }
    for (int t = 0; t < 3; t++) if ((st = zk_build_seq_table(sl, t))) return st;

    ZkBackBits br;
    if (!br.init(b + bits_off, blk.size - bits_off)) return ZKZ_CORRUPTION;
    const int ll_log = sl.tbl_log[0], of_log = sl.tbl_log[1], ml_log = sl.tbl_log[2];
    br.refill();
    uint32_t s_l = br.read(ll_log), s_o = br.read(of_log), s_m = br.read(ml_log);
    uint32_t r0 = ZK_SYM_MAKE(0, 0), r1 = ZK_SYM_MAKE(1, 0), r2 = ZK_SYM_MAKE(2, 0);
    uint32_t lit_end = 0, out_end = 0;
    uint32_t* o_lit = a.seq_lit_end + blk.seq_base;
    uint32_t* o_out = a.seq_out_end + blk.seq_base;
    uint32_t* o_off = a.seq_off + blk.seq_base;
    const uint32_t nseq = blk.nseq;
    for (uint32_t i = 0; i < nseq; i++) {
        const uint32_t cl = sl.ll[s_l], co = sl.of[s_o], cm = sl.ml[s_m];
        br.refill();                                                  // <= 31 bits follow
        const uint32_t ofc = ZK_CELL_CODE(co);
        uint32_t ofv = (1u << ofc) + br.read((int)ofc);
        br.refill();                                                  // <= 16 + 16 bits follow
        uint32_t mlv = tb.ml_base[ZK_CELL_CODE(cm)] + br.read((int)ZK_CELL_ADD(cm));
        uint32_t llv = tb.ll_base[ZK_CELL_CODE(cl)] + br.read((int)ZK_CELL_ADD(cl));
        br.refill();                                                  // <= 9 + 9 + 8 bits follow
        if (i + 1 < nseq) {
            s_l = ZK_CELL_BASE(cl) + br.read((int)ZK_CELL_NB(cl));
            s_m = ZK_CELL_BASE(cm) + br.read((int)ZK_CELL_NB(cm));
            s_o = ZK_CELL_BASE(co) + br.read((int)ZK_CELL_NB(co));
        }
        // repeat-offset history, kept symbolic w.r.t. the (unknown) state entering this block
        uint32_t off;
        if (ofv > 3) { off = ofv - 3; r2 = r1; r1 = r0; r0 = off; }
        else {
            uint32_t idx = ofv - 1 + (llv == 0);
            if (idx == 0) off = r0;
            else {
                if (idx == 3) {
                    if (r0 & ZK_SYM) off = r0 + 1;                    // delta + 1
                    else { off = r0 - 1; if (off == 0) st = ZKZ_CORRUPTION; }
                } else off = idx == 1 ? r1 : r2;
                if (idx != 1) r2 = r1;
                r1 = r0; r0 = off;
            }
        }
        lit_end += llv; out_end += llv + mlv;
        // bounded after EVERY sequence (one step adds < 2^18, so neither sum can wrap past 2^32 unnoticed): the exec
        // kernel uses the intermediate sums as literal-source and output positions
        if (lit_end > blk.lit_size || out_end > ZK_BLOCK_MAX) { st = ZKZ_CORRUPTION; break; }
        o_lit[i] = lit_end; o_out[i] = out_end; o_off[i] = off;
    }
    if (!st && br.bp != 0) st = ZKZ_CORRUPTION;
    if (!st && out_end + (blk.lit_size - lit_end) > blk.bmax) st = ZKZ_CORRUPTION;
    a.blocks[bidx].rep_out[0] = r0; a.blocks[bidx].rep_out[1] = r1; a.blocks[bidx].rep_out[2] = r2;
    a.blocks[bidx].regen = out_end + (blk.lit_size - lit_end);
    return st;
}

__global__ void __launch_bounds__(32 * ZK_SEQ_WARPS) zk_seq_kernel(ZkDecodeArgs a) {
    ZK_DYN_SMEM(smem);
    ZkSeqTabs* tb = (ZkSeqTabs*)smem;
    ZkSeqSlot* slots = (ZkSeqSlot*)(smem + ((sizeof(ZkSeqTabs) + 15) & ~(size_t)15));
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < 36; i += 32 * ZK_SEQ_WARPS) tb->ll_base[i] = ZK_LL_BASE[i];
    for (int i = threadIdx.x; i < 53; i += 32 * ZK_SEQ_WARPS) tb->ml_base[i] = ZK_ML_BASE[i];
    __syncthreads();
    if (a.counters->overflow) return;
    const uint32_t n = a.counters->n_seq_blocks;
    for (;;) {                                  // every warp pulls its own groups of ZK_SEQ_LPW blocks
        uint32_t g = 0;
        if (lane == 0) g = atomicAdd(&a.work_counter[0], 1u);
        g = __shfl_sync(0xFFFFFFFFu, g, 0);
        uint32_t first = g * ZK_SEQ_LPW;
        if (first >= n) break;
        uint32_t my = first + lane;
        if (lane < ZK_SEQ_LPW && my < n) {
            uint32_t bidx = a.seq_list[my];
            ZkBlock blk; blk.entry = 0xFFFFFFFFu;
            if (bidx < a.cap_blocks) blk = a.blocks[bidx];          // always: every reserved slot is written by the scan kernel
            if (blk.entry < a.n_entries && a.entries[blk.entry].status == 0) {
                int st = zk_decode_block_sequences(slots[warp * ZK_SEQ_LPW + lane], *tb, a, blk, bidx, a.comp + a.c_off[blk.entry]);
                a.blocks[bidx].status = st ? -st : 0;
            }
        }
        __syncwarp();
    }
}

// =============================================================================================
// K-D1s (second generation): the same decode, cut into what MUST be serial and what need not be.
//
// A sequence bitstream is one serial chain: the next FSE states depend on bits whose position depends on the current
// states' cells.  The first kernel ran the whole per-sequence work (~110 dependent instructions: extra-bit reads, value
// arithmetic, repeat-offset history, three stores, refills from global memory) on that chain -- about 1 000 cycles per
// sequence.  Here
//   * the bitstream is staged in shared memory by TMA bulk copies (cp.async.bulk + mbarrier, four 512-byte tiles per
//     chain, refilled ahead of the cursor), so a bit field anywhere near the cursor is two shared-memory loads and a
//     funnel shift -- no bit buffer, no refill branches, no global latency on the chain;
//   * a CHAIN LANE only walks the states: three cell loads, the sum of the extra-bit counts, one 32-bit window for the
//     three state updates, and one 16-byte record {cells, cursor} per sequence (~40 instructions);
//   * after every 32 steps ALL lanes turn the records into values: extra bits, literal / match lengths, two warp scans for
//     the cumulative ends, bounds checks, coalesced stores; the repeat-offset history -- a serial state machine -- is run
//     warp-uniformly over the FEW sequences that use a repeat code (explicit offsets just shift it).
// Four chains per warp (lanes 0, 8, 16, 24) share every issued instruction of the chain phase.
// =============================================================================================
#define ZK_S2_NCH 4
#define ZK_S2_TILE 512u
#define ZK_S2_RING_BYTES 2048u            // four tiles: the cursor's tile, the two below it, one being refilled
struct ZkSeq2Chain {
    ZkSeqSlot t;                           // thin cells + build scratch (zk_locate_seq_tables / zk_build_seq_table)
    alignas(128) uint32_t ring[ZK_S2_RING_BYTES / 4];   // staged bitstream (bulk copies want 16-byte aligned shared addresses): byte at offset o from gbase lives at ring byte o & 2047
    uint4 rec[32];                         // per step: {LL cell, OF cell, ML cell, bit cursor before the extra bits}
    uint16_t nxt2[2][64];                  // build scratch of the OF / ML tables (LL uses t.nxt): the three tables are built side by side
    alignas(8) unsigned long long bar[4];  // one mbarrier per tile slot
    uint32_t lit_end, out_end, r0, r1, r2; // carries of the helper phase
    int st;
};

// the 32 bits just below bit position cur (MSB = bit cur - 1) of the staged stream
__device__ __forceinline__ uint32_t zk_s2_window(const uint32_t* ring, uint32_t cur) {
    const uint32_t t = cur - 1u, wi = t >> 5, sh = 31u - (t & 31u);
    return __funnelshift_l(ring[(wi - 1u) & (ZK_S2_RING_BYTES / 4 - 1)], ring[wi & (ZK_S2_RING_BYTES / 4 - 1)], sh);
}
__device__ __forceinline__ uint32_t zk_s2_bits(const uint32_t* ring, uint32_t cur, uint32_t n) {       // n in [0, 31]
    return __funnelshift_l(zk_s2_window(ring, cur), 0u, n);
}

__global__ void __launch_bounds__(32) zk_seq2_kernel(ZkDecodeArgs a) {
    ZK_DYN_SMEM(smem);
    ZkSeqTabs* tb = (ZkSeqTabs*)smem;
    ZkSeq2Chain* chains = (ZkSeq2Chain*)(smem + ((sizeof(ZkSeqTabs) + 127) & ~(size_t)127));
    const int lane = threadIdx.x & 31;
    const int myc = lane >> 3;                                     // the chain this lane belongs to ...
    const bool chain_lane = (lane & 7) == 0;                       // ... and whether it walks it
    for (int i = lane; i < 36; i += 32) tb->ll_base[i] = ZK_LL_BASE[i];
    for (int i = lane; i < 53; i += 32) tb->ml_base[i] = ZK_ML_BASE[i];
    if (chain_lane) for (int k = 0; k < 4; k++) zk_mbar_init(&chains[myc].bar[k], 1);
#ifndef ZK_EMUL
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#endif
    __syncwarp();
    if (a.counters->overflow) return;
    const uint32_t n = a.counters->n_seq_blocks;
    uint32_t tile_uses = 0;                                        // tiles this chain lane has issued so far (slot = use & 3, parity = (use >> 2) & 1)
    for (;;) {
        uint32_t g = 0;
        if (lane == 0) g = atomicAdd(&a.work_counter[0], 1u);
        g = __shfl_sync(0xFFFFFFFFu, g, 0);
        const uint32_t first = g * ZK_S2_NCH;
        if (first >= n) break;
        ZkSeq2Chain& ch = chains[myc];
        // ---------------- per chain: tables, stream geometry, first tiles, initial states (chain lanes, side by side)
        uint32_t bidx = 0, remaining = 0, done = 0, cur = 0, sb_bit = 0, s_l = 0, s_o = 0, s_m = 0, seq_base = 0, lit_size = 0;
        const uint8_t* gbase = nullptr;
        int next_issue = -1, next_wait = -1, top_tile = 0; uint32_t stream_end_off = 0, use0 = 0;
        bool live = false, parsed = false;
        if (chain_lane) {
            ch.st = 0; ch.lit_end = 0; ch.out_end = 0; ch.r0 = ZK_SYM_MAKE(0, 0); ch.r1 = ZK_SYM_MAKE(1, 0); ch.r2 = ZK_SYM_MAKE(2, 0);
            const uint32_t my = first + (uint32_t)myc;
            if (my < n) {
                bidx = a.seq_list[my];
                ZkBlock blk; blk.entry = 0xFFFFFFFFu;
                if (bidx < a.cap_blocks) blk = a.blocks[bidx];
                if (blk.entry < a.n_entries && a.entries[blk.entry].status == 0) {
                    live = true;
                    const uint8_t* ebase = a.comp + a.c_off[blk.entry];
                    const uint8_t* b = ebase + blk.src;
                    uint32_t bits_off = 0;
                    int st = zk_locate_seq_tables(ch.t, b, blk.size, blk.ll_ref < 0, blk.of_ref < 0, blk.ml_ref < 0, &bits_off);
                    if (!st && blk.ll_ref >= 0) { const ZkBlock& rb = a.blocks[blk.ll_ref]; uint32_t d; st = zk_locate_seq_tables(ch.t, ebase + rb.src, rb.size, true, false, false, &d); }
                    if (!st && blk.of_ref >= 0) { const ZkBlock& rb = a.blocks[blk.of_ref]; uint32_t d; st = zk_locate_seq_tables(ch.t, ebase + rb.src, rb.size, false, true, false, &d); }
                    if (!st && blk.ml_ref >= 0) { const ZkBlock& rb = a.blocks[blk.ml_ref]; uint32_t d; st = zk_locate_seq_tables(ch.t, ebase + rb.src, rb.size, false, false, true, &d); }
                    ch.st = st; parsed = !st;
                    const uint8_t* sp = b + bits_off; const uint32_t sn = blk.size - bits_off;
                    if (!st && (sn == 0 || sp[sn - 1] == 0)) st = ZKZ_CORRUPTION;
                    if (!st) {
                        gbase = (const uint8_t*)((uintptr_t)sp & ~(uintptr_t)15);
                        sb_bit = (uint32_t)(sp - gbase) * 8u;
                        stream_end_off = (uint32_t)(sp - gbase) + sn;                       // byte offset of the end of the stream from gbase
                        cur = sb_bit + (sn - 1) * 8u + (uint32_t)zk_highbit(sp[sn - 1]);     // the end mark itself is not data
                        // tiles are staged from the CURSOR's tile downwards: when the end mark is the first byte of a tile, that tile holds
                        // no data (the mark was read above), and counting it would put five tiles in flight on four slots
                        top_tile = (int)(((cur ? cur - 1u : 0u) >> 3) / ZK_S2_TILE);
                        next_issue = top_tile; next_wait = top_tile; use0 = tile_uses;
                        remaining = blk.nseq; seq_base = blk.seq_base; lit_size = blk.lit_size;
                    }
                    ch.st = st;
                }
            }
        }
        // ---------------- the three decoding tables of every chain, built side by side by lanes 0..2 of the chain's lane group
        __syncwarp();
        {
            const bool go = __shfl_sync(0xFFFFFFFFu, (uint32_t)(parsed && ch.st == 0), myc * 8) != 0;
            const int t = lane & 7;
            int bst = 0;
            if (go && t < 3) bst = zk_build_seq_table(ch.t, t, t == 0 ? nullptr : ch.nxt2[t - 1]);
            const uint32_t failed = __ballot_sync(0xFFFFFFFFu, bst != 0);
            if (chain_lane && ((failed >> (myc * 8)) & 7u) && ch.st == 0) ch.st = ZKZ_CORRUPTION;
        }
        __syncwarp();
        // ---------------- tiles of 32 steps
        for (;;) {
            uint32_t cnt = 0;
            if (chain_lane && remaining && ch.st == 0) {
                // tiles: the cursor's tile jc and the two below it must have landed; everything above jc is dead (the records of
                // the previous steps were consumed), so the copies may run down to jc - 3
                const int jc = (int)(((cur ? cur - 1u : 0u) >> 3) / ZK_S2_TILE);
                while (next_issue >= 0 && next_issue >= jc - 3) {
                    const uint32_t off = (uint32_t)next_issue * ZK_S2_TILE;
                    uint32_t bytes = stream_end_off - off; bytes = bytes > ZK_S2_TILE ? ZK_S2_TILE : ((bytes + 15u) & ~15u);   // (16 readable bytes follow every buffer)
                    zk_bulk_g2s((uint8_t*)ch.ring + (off & (ZK_S2_RING_BYTES - 1)), gbase + off, bytes, &ch.bar[tile_uses & 3u]);
                    tile_uses++; next_issue--;
                }
                while (next_wait >= 0 && next_wait >= jc - 2) {
                    const uint32_t u = use0 + (uint32_t)(top_tile - next_wait);
                    if (!zk_mbar_wait(&ch.bar[u & 3u], (u >> 2) & 1u)) {
                        printf("zk_seq2: tile wait timed out: block %u tile %d top %d use %u use0 %u jc %d cur %u\n", bidx, next_wait, top_tile, u, use0, jc, cur);
                        ch.st = ZKZ_GENERIC;
                    }
                    next_wait--;
                }
                if (done == 0) {                                                          // initial states (A.5: LL, OF, ML)
                    const int ll_log = ch.t.tbl_log[0], of_log = ch.t.tbl_log[1], ml_log = ch.t.tbl_log[2];
                    if (cur < sb_bit + (uint32_t)(ll_log + of_log + ml_log)) ch.st = ZKZ_CORRUPTION;
                    else {
                        s_l = zk_s2_bits(ch.ring, cur, (uint32_t)ll_log); cur -= (uint32_t)ll_log;
                        s_o = zk_s2_bits(ch.ring, cur, (uint32_t)of_log); cur -= (uint32_t)of_log;
                        s_m = zk_s2_bits(ch.ring, cur, (uint32_t)ml_log); cur -= (uint32_t)ml_log;
                    }
                }
                if (ch.st == 0) {
                    cnt = remaining < 32u ? remaining : 32u;
                    const bool last_tile = cnt == remaining;
                    bool over = false;
                    for (uint32_t k = 0; k < cnt; k++) {
                        const uint32_t cl = ch.t.ll[s_l], co = ch.t.of[s_o], cm = ch.t.ml[s_m];
                        ch.rec[k] = make_uint4(cl, co, cm, cur);
                        const uint32_t eb = ZK_CELL_CODE(co) + ZK_CELL_ADD(cm) + ZK_CELL_ADD(cl);
                        const uint32_t nl = ZK_CELL_NB(cl), nm = ZK_CELL_NB(cm), no = ZK_CELL_NB(co);
                        const bool upd = !(last_tile && k + 1 == cnt);                   // no state update after the block's last sequence
                        const uint32_t need_bits = eb + (upd ? nl + nm + no : 0u);
                        if (cur - sb_bit < need_bits) { over = true; cnt = k; break; }    // the stream is shorter than its sequences need
                        cur -= eb;
                        if (upd) {
                            const uint32_t w = zk_s2_window(ch.ring, cur);
                            s_l = ZK_CELL_BASE(cl) + __funnelshift_l(w, 0u, nl);
                            s_m = ZK_CELL_BASE(cm) + __funnelshift_l(w << nl, 0u, nm);
                            s_o = ZK_CELL_BASE(co) + __funnelshift_l(w << (nl + nm), 0u, no);
                            cur -= nl + nm + no;
                        }
                    }
                    if (over) ch.st = ZKZ_CORRUPTION;
                    remaining -= cnt; 
                    if (over) remaining = 0;
                }
            }
            __syncwarp();
            // ---------------- helper phase: every lane, one chain after the other
            uint32_t any = 0;
#pragma unroll 1
            for (int cc = 0; cc < ZK_S2_NCH; cc++) {
                const uint32_t ncc = __shfl_sync(0xFFFFFFFFu, cnt, cc * 8);
                if (ncc == 0) continue;
                any = 1;
                ZkSeq2Chain& hc = chains[cc];
                const uint32_t sbase = __shfl_sync(0xFFFFFFFFu, seq_base, cc * 8), sdone = __shfl_sync(0xFFFFFFFFu, done, cc * 8);
                const uint32_t lsz = __shfl_sync(0xFFFFFFFFu, lit_size, cc * 8);
                const bool act = (uint32_t)lane < ncc;
                uint32_t llv = 0, mlv = 0, ofv = 4;                                       // inactive lanes: explicit offsets that push nothing (masked below)
                if (act) {
                    const uint4 r = hc.rec[lane];
                    const uint32_t ofc = ZK_CELL_CODE(r.y), mlb = ZK_CELL_ADD(r.z), llb = ZK_CELL_ADD(r.x);
                    uint32_t c = r.w;
                    ofv = (1u << ofc) + zk_s2_bits(hc.ring, c, ofc); c -= ofc;
                    mlv = tb->ml_base[ZK_CELL_CODE(r.z)] + zk_s2_bits(hc.ring, c, mlb); c -= mlb;
                    llv = tb->ll_base[ZK_CELL_CODE(r.x)] + zk_s2_bits(hc.ring, c, llb);
                }
                // cumulative ends: two inclusive warp scans on top of the chain's carries
                uint32_t le = llv, oe = llv + mlv;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t x = __shfl_up_sync(0xFFFFFFFFu, le, d), y = __shfl_up_sync(0xFFFFFFFFu, oe, d);
                    if (lane >= d) { le += x; oe += y; }
                }
                le += hc.lit_end; oe += hc.out_end;
                // bounded after EVERY sequence (a tile adds < 2^23, the carries are <= 2^17: no wrap can hide an overflow)
                const bool badv = act && (le > lsz || oe > ZK_BLOCK_MAX);
                // repeat-offset history (A.5), symbolic with respect to the state entering the block: explicit offsets only shift it,
                // so the serial part runs over the sequences that USE a repeat code
                uint32_t r0 = hc.r0, r1 = hc.r1, r2 = hc.r2, off = ofv - 3u;
                const uint32_t repm = __ballot_sync(0xFFFFFFFFu, act && ofv <= 3u);
                const uint32_t idxv = ofv - 1u + (llv == 0u ? 1u : 0u);                 // meaningful on repeat lanes only
                uint32_t m = repm; int lastpos = 0; bool badr = false;
                for (;;) {
                    const int j = m ? __ffs((int)m) - 1 : (int)ncc;                      // next repeat lane, or the end of the tile
                    const int cnte = j - lastpos;                                        // explicit offsets since the last repeat lane
                    if (cnte > 0) {
                        const uint32_t e1 = __shfl_sync(0xFFFFFFFFu, off, j - 1);
                        const uint32_t e2 = __shfl_sync(0xFFFFFFFFu, off, cnte > 1 ? j - 2 : 0), e3 = __shfl_sync(0xFFFFFFFFu, off, cnte > 2 ? j - 3 : 0);
                        const uint32_t o0 = r0, o1 = r1;
                        r0 = e1; r1 = cnte > 1 ? e2 : o0; r2 = cnte > 2 ? e3 : (cnte == 2 ? o0 : o1);
                    }
                    if (!m) break;
                    const uint32_t idx = __shfl_sync(0xFFFFFFFFu, idxv, j);
                    uint32_t o;
                    if (idx == 0) o = r0;
                    else {
                        if (idx == 3) { if (r0 & ZK_SYM) o = r0 + 1u; else { o = r0 - 1u; if (o == 0) badr = true; } }
                        else o = idx == 1 ? r1 : r2;
                        if (idx != 1) r2 = r1;
                        r1 = r0; r0 = o;
                    }
                    if (lane == j) off = o;
                    lastpos = j + 1; m &= m - 1;
                }
                if (act) {
                    const uint32_t at = sbase + sdone + (uint32_t)lane;
                    a.seq_lit_end[at] = le; a.seq_out_end[at] = oe; a.seq_off[at] = off;
                }
                const bool anybad = __any_sync(0xFFFFFFFFu, badv) || badr;
                if (lane == (int)ncc - 1) { hc.lit_end = le; hc.out_end = oe; }
                if (lane == 0) { hc.r0 = r0; hc.r1 = r1; hc.r2 = r2; if (anybad && hc.st == 0) hc.st = ZKZ_CORRUPTION; }
            }
            __syncwarp();
            if (chain_lane) { done += cnt; if (ch.st != 0) remaining = 0; }
            if (!any) break;
        }
        // ---------------- results of the block
        if (chain_lane) {     // copies issued ahead but never needed must have landed before the next block reuses the ring
            while (next_wait > next_issue) { const uint32_t u = use0 + (uint32_t)(top_tile - next_wait); zk_mbar_wait(&ch.bar[u & 3u], (u >> 2) & 1u); next_wait--; }
        }
        if (chain_lane && live) {
            int st = ch.st;
            if (!st && cur != sb_bit) st = ZKZ_CORRUPTION;                                // every bit of the stream is consumed, no more
            if (!st && ch.out_end + (lit_size - ch.lit_end) > a.blocks[bidx].bmax) st = ZKZ_CORRUPTION;
            a.blocks[bidx].rep_out[0] = ch.r0; a.blocks[bidx].rep_out[1] = ch.r1; a.blocks[bidx].rep_out[2] = ch.r2;
            a.blocks[bidx].regen = ch.out_end + (lit_size - ch.lit_end);
            a.blocks[bidx].status = st ? -st : 0;
        }
        __syncwarp();
    }
}

// =============================================================================================
// K-D1h: Huffman literal decode -- one LANE per Huffman stream (4 lanes per 4-stream block).
// =============================================================================================
#define ZK_HUF_SLOTS 8            // blocks per warp-CTA; 8 x 3.1 KiB -> 9 CTAs / SM

// Two-level decoding table.  Cells are laid out weight ascending (A.4), so the codes of the two longest lengths occupy
// the first L <= 510 cells of the 2^maxBits index space, and everything above is replicated at least four times:
//   idx < L  -> low[idx]        (full resolution)        idx >= L -> l1[idx >> 2]      (2^(maxBits-2) <= 512 entries)
// 2 KiB instead of the flat 4 KiB table: the kernel is bound by memory latency with shared memory capping the streams
// in flight, so the extra compare per symbol buys 1.7x the blocks per SM.
struct ZkHufSlot {
    uint16_t l1[512], low[512];                // (nbBits << 8) | symbol
    uint32_t n_low;                            // L
    uint8_t weights[256];
    uint16_t hpos[256];
    uint8_t wsym[64], wnb[64]; uint16_t wbase[64];   // FSE table for compressed weights (log <= 6)
    int huf_bits, nw, st;
    uint32_t tree_bytes;
};

// Huffman tree description -> sl.weights[0..nw) incl. the implied last weight (A.4).
// Returns bytes consumed or 0 on corruption; sets sl.huf_bits / sl.nw.
__device__ uint32_t zk_read_huf_weights(ZkHufSlot& sl, const uint8_t* p, uint32_t n) {
    if (n < 1) return 0;
    uint32_t hb = p[0], used; int nw = 0;
    if (hb >= 128) {
        nw = (int)hb - 127; used = 1 + (uint32_t)(nw + 1) / 2;
        if (used > n) return 0;
        for (int i = 0; i < nw; i++) { uint32_t b = p[1 + i / 2]; sl.weights[i] = (uint8_t)((i & 1) ? (b & 15) : (b >> 4)); }
    } else {
        used = 1 + hb;
        if (hb == 0 || used > n) return 0;
        int16_t cnt[16]; int ns, lg;
        uint32_t r = zk_fse_read_ncount(p + 1, hb, 6, 12, cnt, &ns, &lg);
        if (!r) return 0;
        int S = 1 << lg, high = S - 1; uint16_t nx[16];
        for (int s = 0; s < ns; s++) { if (cnt[s] == -1) { sl.wsym[high--] = (uint8_t)s; nx[s] = 1; } else nx[s] = (uint16_t)cnt[s]; }
        int step = (S >> 1) + (S >> 3) + 3, pos = 0;
        for (int s = 0; s < ns; s++)
            for (int q = 0; q < cnt[s]; q++) { sl.wsym[pos] = (uint8_t)s; do { pos = (pos + step) & (S - 1); } while (pos > high); }
        if (pos != 0) return 0;
        for (int u = 0; u < S; u++) {
            int s = sl.wsym[u]; uint32_t x = nx[s]++; int nb = lg - zk_highbit(x);
            sl.wnb[u] = (uint8_t)nb; sl.wbase[u] = (uint16_t)((x << nb) - S);
        }
        ZkBackBits br;
        if (!br.init(p + 1 + r, hb - r)) return 0;
        br.refill();
        uint32_t s1 = br.read(lg), s2 = br.read(lg);
        if (br.bp < 0) return 0;
        for (;;) {   // two interleaved states, over-read terminates (A.4)
            if (nw >= 254) return 0;
            br.refill();
            sl.weights[nw++] = sl.wsym[s1];
            s1 = sl.wbase[s1] + br.read(sl.wnb[s1]);
            if (br.bp < 0) { sl.weights[nw++] = sl.wsym[s2]; break; }
            sl.weights[nw++] = sl.wsym[s2];
            s2 = sl.wbase[s2] + br.read(sl.wnb[s2]);
            if (br.bp < 0) { sl.weights[nw++] = sl.wsym[s1]; break; }
        }
        if (nw > 255) return 0;                    // at most 255 explicit weights (+ the implied one = 256 symbols)
    }
    uint32_t total = 0, n_w1 = 0;
    for (int i = 0; i < nw; i++) {
        uint32_t w = sl.weights[i];
        if (w > 11) return 0;
        if (w) total += 1u << (w - 1);
        n_w1 += (w == 1);
    }
    if (total == 0) return 0;
    int max_bits = zk_highbit(total) + 1;
    if (max_bits > 11) return 0;
    uint32_t left = (1u << max_bits) - total;
    if (left & (left - 1)) return 0;               // must be a power of two (left >= 1 by construction)
    uint32_t lw = (uint32_t)zk_highbit(left) + 1;
    sl.weights[nw++] = (uint8_t)lw;
    n_w1 += (lw == 1);
    if (n_w1 < 2 || (n_w1 & 1)) return 0;          // libzstd's HUF_readStats sanity rule
    sl.huf_bits = max_bits; sl.nw = nw;
    return used;
}

// Decode `cnt` Huffman symbols of one stream into out (A.4).  Returns false on corruption.
__device__ __forceinline__ uint32_t zk_huf_lookup(const ZkHufSlot& sl, uint32_t idx) {
    return idx < sl.n_low ? sl.low[idx & 511u] : sl.l1[idx >> 2];
}
__device__ bool zk_huf_decode_stream(const ZkHufSlot& sl, int max_bits, const uint8_t* p, uint32_t n, uint8_t* out, uint32_t cnt) {
    ZkBackBits br;
    if (!br.init(p, n)) return false;
    uint32_t i = 0;
    while (i < cnt && ((uintptr_t)(out + i) & 3)) {
        br.refill();
        uint32_t e = zk_huf_lookup(sl, br.peek(max_bits)); br.skip((int)(e >> 8)); out[i++] = (uint8_t)e;
    }
    for (; i + 4 <= cnt; i += 4) {
        br.refill();                                   // >= 33 bits: three codes of <= 11 bits
        uint32_t e0 = zk_huf_lookup(sl, br.peek(max_bits)); br.skip((int)(e0 >> 8));
        uint32_t e1 = zk_huf_lookup(sl, br.peek(max_bits)); br.skip((int)(e1 >> 8));
        uint32_t e2 = zk_huf_lookup(sl, br.peek(max_bits)); br.skip((int)(e2 >> 8));
        br.refill();
        uint32_t e3 = zk_huf_lookup(sl, br.peek(max_bits)); br.skip((int)(e3 >> 8));
        *(uint32_t*)(out + i) = (e0 & 0xFF) | ((e1 & 0xFF) << 8) | ((e2 & 0xFF) << 16) | ((e3 & 0xFF) << 24);
    }
    for (; i < cnt; i++) {
        br.refill();
        uint32_t e = zk_huf_lookup(sl, br.peek(max_bits)); br.skip((int)(e >> 8)); out[i] = (uint8_t)e;
    }
    return br.bp == 0;
}

__global__ void __launch_bounds__(32) zk_huf_kernel(ZkDecodeArgs a) {
    ZK_DYN_SMEM(smem);
    ZkHufSlot* slots = (ZkHufSlot*)smem;
    const int lane = threadIdx.x, si = lane >> 2, stream = lane & 3;
    if (a.counters->overflow) return;
    const uint32_t n = a.counters->n_huf_blocks;
    for (;;) {
        uint32_t g = 0;
        if (lane == 0) g = atomicAdd(&a.work_counter[1], 1u);
        g = __shfl_sync(0xFFFFFFFFu, g, 0);
        uint32_t first = g * ZK_HUF_SLOTS;
        if (first >= n) break;
        const uint32_t my = first + si;
        const bool active = my < n;
        ZkHufSlot& sl = slots[si];
        uint32_t bidx = 0; ZkBlock blk; ZkLitHdr lh; const uint8_t* ebase = nullptr;
        bool live = false;
        if (active) {
            bidx = a.huf_list[my];
            if (bidx < a.cap_blocks) {                              // always: every reserved slot is written by the scan kernel
                blk = a.blocks[bidx];
                live = blk.entry < a.n_entries && a.entries[blk.entry].status == 0;
            }
            if (live) {
                ebase = a.comp + a.c_off[blk.entry];
                zk_parse_lit_hdr(ebase + blk.src, blk.size, lh);  // validated by the scan kernel
            }
        }
        // 1. tree description (own block, or the block a Treeless block refers to) -- one lane per block
        if (live && stream == 0) {
            int st = 0; uint32_t tb = 0;
            if (lh.type == 2) { tb = zk_read_huf_weights(sl, ebase + blk.src + lh.hdr, lh.comp); if (!tb) st = ZKZ_CORRUPTION; }
            else {
                const ZkBlock& rb = a.blocks[blk.huf_ref];
                ZkLitHdr rh; zk_parse_lit_hdr(ebase + rb.src, rb.size, rh);
                if (!zk_read_huf_weights(sl, ebase + rb.src + rh.hdr, rh.comp)) st = ZKZ_CORRUPTION;
            }
            if (!st) {   // start cell of every symbol: weight ascending, symbols in natural order
                uint32_t rank_start[13], cntw[13];
                for (int w = 0; w < 13; w++) cntw[w] = 0;
                for (int s = 0; s < sl.nw; s++) cntw[sl.weights[s]]++;
                uint32_t acc = 0;
                for (int w = 1; w <= sl.huf_bits; w++) { rank_start[w] = acc; acc += cntw[w] << (w - 1); }
                for (int s = 0; s < sl.nw; s++) { int w = sl.weights[s]; if (w) { sl.hpos[s] = (uint16_t)rank_start[w]; rank_start[w] += 1u << (w - 1); } }
                if (acc != (1u << sl.huf_bits)) st = ZKZ_CORRUPTION;
                sl.n_low = cntw[1] + 2u * cntw[2];                 // cells of the two longest code lengths (<= 512)
                if (sl.n_low > 512u) st = ZKZ_CORRUPTION;
            }
            sl.st = st; sl.tree_bytes = tb;
        }
        __syncwarp();
        // 2. fill the decoding table -- the block's four lanes share the symbols
        const bool good = live && sl.st == 0;
        if (good) {
            const int max_bits = sl.huf_bits;
            for (int s = stream; s < sl.nw; s += 4) {
                int w = sl.weights[s];
                if (!w) continue;
                uint32_t len = 1u << (w - 1), pos = sl.hpos[s];
                uint16_t e = (uint16_t)(((max_bits + 1 - w) << 8) | s);
                if (w <= 2) for (uint32_t i = 0; i < len; i++) sl.low[pos + i] = e;
                else for (uint32_t i = 0; i < (len >> 2); i++) sl.l1[(pos >> 2) + i] = e;
            }
        }
        __syncwarp();
        // 3. decode: one lane per stream
        bool ok = true;
        if (good) {
            const uint8_t* q = ebase + blk.src + lh.hdr + sl.tree_bytes;
            uint32_t qn = lh.comp - sl.tree_bytes;
            uint8_t* out = a.lit + blk.lit_base;
            if (lh.streams == 1) {
                if (stream == 0) ok = zk_huf_decode_stream(sl, sl.huf_bits, q, qn, out, lh.regen);
            } else {
                uint32_t seg = (lh.regen + 3) / 4;
                if (qn < 10 || lh.regen < 6 || seg * 3 > lh.regen) ok = false;   // jump table + 4 non-empty streams; libzstd rejects regen < 6
                else {
                    uint32_t s1 = zk_ld_le16(q), s2 = zk_ld_le16(q + 2), s3 = zk_ld_le16(q + 4);
                    if (6 + s1 + s2 + s3 >= qn) ok = false;
                    else {
                        uint32_t s4 = qn - 6 - s1 - s2 - s3;
                        uint32_t off = stream == 0 ? 0 : (stream == 1 ? s1 : (stream == 2 ? s1 + s2 : s1 + s2 + s3));
                        uint32_t len = stream == 0 ? s1 : (stream == 1 ? s2 : (stream == 2 ? s3 : s4));
                        uint32_t cnt = stream < 3 ? seg : lh.regen - 3 * seg;
                        ok = zk_huf_decode_stream(sl, sl.huf_bits, q + 6 + off, len, out + stream * seg, cnt);
                    }
                }
            }
        }
        uint32_t bad = __ballot_sync(0xFFFFFFFFu, !ok);
        if (live && stream == 0) {
            int st = sl.st;
            if (!st && ((bad >> (si * 4)) & 0xFu)) st = ZKZ_CORRUPTION;
            a.blocks[bidx].lit_status = st ? -st : 0;
        }
        __syncwarp();
    }
}

// =============================================================================================
// K-D2: ordered sequence execution with a shared-memory window.
//
// One CTA per seek-table entry, W warps.  The entry's sequences are cut into chunks of 32 (one per
// lane); chunk c belongs to warp c % W.  The last R bytes of output live in a shared-memory ring:
// every copy writes into the ring, dependent (recent) match sources are read from the ring
// (~30-cycle latency instead of an L2 round trip -- the first version spent 60 % of its samples
// waiting on those), and each finished chunk is flushed to HBM with 16-byte stores.
//   * done_pos / done_chunk : in-order publication of finished chunks (everything below done_pos
//     is final AND flushed to HBM);
//   * a chunk may start once its end lies within R/2 of done_pos, so the in-flight region never
//     laps the ring; a source at distance < R/2 from the chunk start is therefore still resident;
//   * chunks larger than R/2, Raw/RLE blocks and literal-only blocks run alone ("direct" path:
//     HBM to HBM, then the ring is re-synchronised from HBM).
// =============================================================================================
#define ZK_LONG 48u     // literal runs / matches at least this long are copied by the whole warp

#define ZK_D2_META 64u          // chunk descriptors kept in shared memory (chunks between the oldest unflushed and the newest started)

struct ZkD2Smem {
    // in-order prefixes, advanced co-operatively by whoever polls ("helping"); nobody ever waits for a predecessor to publish
    uint32_t done_pos, done_chunk;         // every byte below done_pos is final (readable from the ring); chunks [0, done_chunk) are done
    uint32_t flushed_pos, flushed_chunk;   // ... and below flushed_pos it is in HBM too
    int abort_code;
    // per-chunk descriptors, slot = chunk & (ZK_D2_META-1); a field is valid for chunk k iff its tag == k + 1
    uint32_t started[ZK_D2_META], start[ZK_D2_META], end[ZK_D2_META], done[ZK_D2_META], flushed[ZK_D2_META];
    // per-SEQUENCE completion inside a chunk (the dependency chain of a frame runs sequence to sequence, not chunk to chunk):
    uint32_t oe[ZK_D2_META][32];          // end position of each of the chunk's 32 sequences (non-decreasing; lanes past the last = chunk end)
    uint32_t dmask[ZK_D2_META];           // bit j: sequence j is completely written (literals + match)
    uint32_t litdone[ZK_D2_META];         // tag: every literal run of the chunk is in place
};
#define ZK_VOL(x) (*(volatile uint32_t*)&(x))

__device__ __forceinline__ void zk_d2_abort(ZkD2Smem& sm, int code) { atomicCAS(&sm.abort_code, 0, code); }
// warp-uniform view of the abort flag (every lane must take the same branch around collectives)
__device__ __forceinline__ bool zk_d2_aborted(ZkD2Smem& sm) { return __any_sync(0xFFFFFFFFu, *(volatile int*)&sm.abort_code != 0); }

// advance the in-order prefixes as far as the per-chunk flags allow (any thread may do this at any time)
__device__ __noinline__ void zk_d2_help(ZkD2Smem& sm) {
    uint32_t dc = ZK_VOL(sm.done_chunk), dc0 = dc, dp = 0;
    while (ZK_VOL(sm.done[dc & (ZK_D2_META - 1)]) == dc + 1) { dp = ZK_VOL(sm.end[dc & (ZK_D2_META - 1)]); dc++; }
    if (dc != dc0) { atomicMax(&sm.done_pos, dp); __threadfence_block(); atomicMax(&sm.done_chunk, dc); }
    uint32_t fc = ZK_VOL(sm.flushed_chunk), fc0 = fc, fp = 0;
    while (ZK_VOL(sm.flushed[fc & (ZK_D2_META - 1)]) == fc + 1) { fp = ZK_VOL(sm.end[fc & (ZK_D2_META - 1)]); fc++; }
    if (fc != fc0) { atomicMax(&sm.flushed_pos, fp); __threadfence_block(); atomicMax(&sm.flushed_chunk, fc); }
}

// Are all bytes of [src0, need_end) that lie BEFORE this chunk final?  (lane-level; scans the descriptors of the chunks in flight)
__device__ __forceinline__ bool zk_d2_ext_ready(ZkD2Smem& sm, uint32_t c, uint32_t src0, uint32_t need_end, uint32_t chunk_start) {
    if (src0 >= chunk_start) return true;                               // purely intra-chunk
    const uint32_t ne = need_end < chunk_start ? need_end : chunk_start;
    if (ne <= ZK_VOL(sm.done_pos)) return true;
    const uint32_t dc = ZK_VOL(sm.done_chunk);
    for (uint32_t k = c; k-- > dc;) {
        const uint32_t e = k & (ZK_D2_META - 1);
        if (ZK_VOL(sm.started[e]) != k + 1) return false;               // its range is not known yet
        const uint32_t sk = ZK_VOL(sm.start[e]), ek = ZK_VOL(sm.end[e]);
        if (sk < ne && ek > src0 && ZK_VOL(sm.done[e]) != k + 1) return false;
        if (sk <= src0) return true;                                    // older chunks end at or before src0
    }
    return true;                                                         // reached the done prefix
}

// warp-cooperative copy of n bytes HBM -> HBM, non-overlapping (or src entirely before dst with distance >= n)
__device__ __noinline__ void zk_warp_copy(uint8_t* dst, const uint8_t* src, uint32_t n, int lane) {
    uint32_t head = (uint32_t)((16 - ((uintptr_t)dst & 15)) & 15);
    if (head > n) head = n;
    if (lane < (int)head) dst[lane] = src[lane];
    dst += head; src += head; n -= head;
    uint32_t nvec = n >> 4;
    uint32_t mis = (uint32_t)((uintptr_t)src & 3);
    if (mis == 0) {
        if (((uintptr_t)src & 15) == 0) {
            for (uint32_t i = lane; i < nvec; i += 32) ((uint4*)dst)[i] = ((const uint4*)src)[i];
        } else {
            for (uint32_t i = lane; i < nvec; i += 32) {
                const uint32_t* s = (const uint32_t*)src + 4 * i;
                ((uint4*)dst)[i] = make_uint4(s[0], s[1], s[2], s[3]);
            }
        }
    } else {
        const uint32_t* sa = (const uint32_t*)(src - mis);
        uint32_t sh = mis * 8;
        for (uint32_t i = lane; i < nvec; i += 32) {
            const uint32_t* s = sa + 4 * i;
            uint32_t w0 = s[0], w1 = s[1], w2 = s[2], w3 = s[3], w4 = s[4];
            ((uint4*)dst)[i] = make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh),
                                          __funnelshift_r(w2, w3, sh), __funnelshift_r(w3, w4, sh));
        }
    }
    uint32_t done = nvec << 4;
    for (uint32_t i = done + lane; i < n; i += 32) dst[i] = src[i];
}

__device__ __noinline__ void zk_warp_fill(uint8_t* dst, uint32_t byte, uint32_t n, int lane) {
    uint32_t head = (uint32_t)((16 - ((uintptr_t)dst & 15)) & 15);
    if (head > n) head = n;
    if (lane < (int)head) dst[lane] = (uint8_t)byte;
    dst += head; n -= head;
    uint32_t w = byte * 0x01010101u, nvec = n >> 4;
    for (uint32_t i = lane; i < nvec; i += 32) ((uint4*)dst)[i] = make_uint4(w, w, w, w);
    for (uint32_t i = (nvec << 4) + lane; i < n; i += 32) dst[i] = (uint8_t)byte;
}

// warp-cooperative match copy in HBM: dst[0..n) = dst[-off ..), overlap allowed (period doubling)
__device__ __noinline__ void zk_warp_match(uint8_t* dst, uint32_t off, uint32_t n, int lane) {
    const uint8_t* src = dst - off;
    if (off >= n) { zk_warp_copy(dst, src, n, lane); return; }
    uint32_t have = off, done = 0;            // [src, src+have) is final periodic data
    while (done < n) {
        uint32_t c = n - done < have ? n - done : have;
        zk_warp_copy(dst + done, src, c, lane);
        __syncwarp();
        done += c; have += c;
    }
}

// the low min(k, 8) bytes of (lo, hi) -> p[0..): predicated byte stores at immediate offsets (k >= 1)
__device__ __forceinline__ void zk_st_bytes8(uint8_t* p, uint32_t lo, uint32_t hi, uint32_t k) {
    p[0] = (uint8_t)lo;
    if (k > 1) p[1] = (uint8_t)(lo >> 8);
    if (k > 2) p[2] = (uint8_t)(lo >> 16);
    if (k > 3) p[3] = (uint8_t)(lo >> 24);
    if (k > 4) p[4] = (uint8_t)hi;
    if (k > 5) p[5] = (uint8_t)(hi >> 8);
    if (k > 6) p[6] = (uint8_t)(hi >> 16);
    if (k > 7) p[7] = (uint8_t)(hi >> 24);
}

// per-CTA view of the ring: position p (entry-relative) lives at ring[(p + mis) & mask], mis = (out address & 15)
// so that 16-byte groups of the ring line up with 16-byte groups of HBM.
struct ZkRing {
    uint8_t* ring; uint32_t mask, mis; uint8_t* out;
    __device__ __forceinline__ uint8_t& at(uint32_t p) const { return ring[(p + mis) & mask]; }
    // unaligned 8-byte read of positions [p, p+8) (three aligned word reads, wrap-safe)
    __device__ __forceinline__ unsigned long long ld8(uint32_t p) const {
        const uint32_t idx = (p + mis) & mask, wi = idx & ~3u, sh = (idx & 3u) * 8u;
        const uint32_t w0 = *(const uint32_t*)(ring + wi), w1 = *(const uint32_t*)(ring + ((wi + 4) & mask)), w2 = *(const uint32_t*)(ring + ((wi + 8) & mask));
        return (unsigned long long)__funnelshift_r(w0, w1, sh) | ((unsigned long long)__funnelshift_r(w1, w2, sh) << 32);
    }
    // lane-local match copy inside the ring, 8 bytes per step when the period allows it.  This copy sits on the dependency
    // chain of the frame AND was 40 % of all instructions of the kernel when it stored byte by byte through at() (address
    // arithmetic, 64-bit shifts and loop control per byte: ~12 instructions a byte); without a wrap on either side it is three
    // word loads, two funnel shifts and predicated byte stores at immediate offsets.
    __device__ __forceinline__ void copy_near(uint32_t dst, uint32_t src, uint32_t n) const {
        const uint32_t size = mask + 1, di = (dst + mis) & mask, si = (src + mis) & mask;
        if (dst - src >= 8) {
            if (di + n <= size && si + n + 12 <= size) {
                uint8_t* dp = ring + di; const uint32_t* sp = (const uint32_t*)(ring + (si & ~3u)); const uint32_t sh = (si & 3u) * 8u;
                for (uint32_t i = 0; i < n; i += 8) {
                    const uint32_t w0 = sp[0], w1 = sp[1], w2 = sp[2];
                    zk_st_bytes8(dp, __funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), n - i);
                    dp += 8; sp += 2;
                }
            } else {
                for (uint32_t i = 0; i < n; i += 8) {
                    unsigned long long v = ld8(src + i);
                    const uint32_t k = n - i < 8 ? n - i : 8;
                    for (uint32_t q = 0; q < k; q++) { at(dst + i + q) = (uint8_t)v; v >>= 8; }
                }
            }
        } else for (uint32_t i = 0; i < n; i++) at(dst + i) = at(src + i);
    }
    // store the low min(k, 8) bytes of (lo, hi) at positions [p, p + k) of the entry
    __device__ __forceinline__ void st8(uint32_t p, uint32_t lo, uint32_t hi, uint32_t k) const {
        const uint32_t di = (p + mis) & mask;
        if (di + 8 <= mask + 1) zk_st_bytes8(ring + di, lo, hi, k);
        else { unsigned long long v = (unsigned long long)lo | ((unsigned long long)hi << 32); for (uint32_t q = 0; q < k && q < 8; q++) { at(p + q) = (uint8_t)v; v >>= 8; } }
    }
};

// flush [s, e) ring -> HBM: full 16-byte groups with vector stores, the ragged head and tail (neighbours own the rest of those
// groups) byte-parallel by lanes 0..15 / 16..31
__device__ __forceinline__ void zk_ring_flush(const ZkRing& rg, uint32_t s, uint32_t e, int lane) {
    if (e <= s) return;
    const uint32_t sb = s + rg.mis, eb = e + rg.mis;                       // shifted positions: 16-byte groups line up with HBM
    const uint32_t uf0 = (sb + 15) >> 4, uf1 = eb >> 4;                    // full groups [uf0, uf1)
    for (uint32_t u = uf0 + lane; u < uf1; u += 32) { const uint32_t g = u << 4; *(uint4*)(rg.out + (g - rg.mis)) = *(const uint4*)(rg.ring + (g & rg.mask)); }
    const uint32_t head_end = (uf0 << 4) < eb ? (uf0 << 4) : eb;
    if (lane < 16) { const uint32_t q = sb + (uint32_t)lane; if (q < head_end) rg.out[q - rg.mis] = rg.ring[q & rg.mask]; }
    else if (uf1 >= uf0) { const uint32_t q = (uf1 << 4) + (uint32_t)lane - 16u; if (q < eb) rg.out[q - rg.mis] = rg.ring[q & rg.mask]; }
}

// reload [s, e) HBM -> ring (after a direct HBM-to-HBM block)
__device__ __noinline__ void zk_ring_reload(const ZkRing& rg, uint32_t s, uint32_t e, int tid, int nthr) {
    if (e <= s) return;
    const uint32_t u0 = (s + rg.mis) >> 4, u1 = (e + rg.mis - 1) >> 4;
    for (uint32_t u = u0 + tid; u <= u1; u += nthr) {
        const uint32_t g = u << 4;
        const uint32_t lo = g > s + rg.mis ? g : s + rg.mis, hi = g + 16 < e + rg.mis ? g + 16 : e + rg.mis;
        if (hi - lo == 16) *(uint4*)(rg.ring + (g & rg.mask)) = *(const uint4*)(rg.out + (g - rg.mis));
        else for (uint32_t q = lo; q < hi; q++) rg.ring[q & rg.mask] = rg.out[q - rg.mis];
    }
}

// unaligned 8-byte little-endian load from HBM (three aligned 4-byte loads issued back to back)
__device__ __forceinline__ unsigned long long zk_ld8_unaligned(const uint8_t* p) {
    uintptr_t a = (uintptr_t)p; uint32_t mis = (uint32_t)(a & 3);
    const uint32_t* q = (const uint32_t*)(a - mis);
    uint32_t w0 = q[0], w1 = q[1];
    if (mis == 0) return (unsigned long long)w0 | ((unsigned long long)w1 << 32);
    uint32_t w2 = q[2], sh = mis * 8;
    return (unsigned long long)__funnelshift_r(w0, w1, sh) | ((unsigned long long)__funnelshift_r(w1, w2, sh) << 32);
}

// Place the literal runs of one chunk.  The runs are CONTIGUOUS in the block's literal buffer ([lit_lo, lit_hi)), so the
// warp reads them with coalesced loads, 32 bytes a step, and every byte finds its destination by a 5-step search over the
// lanes' cumulative literal ends (le is non-decreasing across lanes).  A per-lane byte loop paid one HBM round trip per
// byte and was the real bottleneck of the first exec kernels.  TO_RING: destination is the ring, else HBM directly.
template <bool TO_RING>
__device__ __forceinline__ void zk_chunk_literals(const ZkRing& rg, const uint8_t* lit, int lit_kind, uint32_t lit_byte, uint32_t le, uint32_t le_prev,
                                                  uint32_t o_lit, int lane) {
    const uint32_t lit_lo = __shfl_sync(0xFFFFFFFFu, le_prev, 0), lit_hi = __shfl_sync(0xFFFFFFFFu, le, 31);
    for (uint32_t base = lit_lo; base < lit_hi; base += 256) {
        // issue up to eight coalesced 32-byte loads first (one memory latency for 256 literal bytes), then place them
        uint32_t bytes[8];
#pragma unroll
        for (int u = 0; u < 8; u++) {
            const uint32_t t = base + u * 32 + lane;
            bytes[u] = lit_byte;
            if (t < lit_hi && lit_kind != 1) bytes[u] = lit[t];
        }
#pragma unroll
        for (int u = 0; u < 8; u++) {
            const uint32_t t = base + u * 32 + lane;
            if (base + u * 32 >= lit_hi) break;           // warp-uniform
            const bool active = t < lit_hi;
            int lo = 0, hi = 31;                          // owner = first lane whose le > t
#pragma unroll
            for (int step = 0; step < 5; step++) {
                const int mid = (lo + hi) >> 1;
                const uint32_t v = __shfl_sync(0xFFFFFFFFu, le, mid);
                if (v > t) hi = mid; else lo = mid + 1;
            }
            const uint32_t d0 = __shfl_sync(0xFFFFFFFFu, o_lit, lo), l0 = __shfl_sync(0xFFFFFFFFu, le_prev, lo);
            if (active) {
                const uint32_t dest = d0 + (t - l0);
                if (TO_RING) rg.at(dest) = (uint8_t)bytes[u]; else rg.out[dest] = (uint8_t)bytes[u];
            }
        }
    }
}

// chunk c's bytes are final in the ring: dependants may read them
__device__ __forceinline__ void zk_d2_mark_done(ZkD2Smem& sm, uint32_t c, int lane) {
    __threadfence_block();
    __syncwarp();
    if (lane == 0) {
        const uint32_t e = c & (ZK_D2_META - 1);
        ZK_VOL(sm.dmask[e]) = 0xFFFFFFFFu; ZK_VOL(sm.litdone[e]) = c + 1; ZK_VOL(sm.done[e]) = c + 1;
        zk_d2_help(sm);
    }
    __syncwarp();
}
// ... and now they are in HBM as well (far readers and ring reuse depend on this one)
__device__ __forceinline__ void zk_d2_mark_flushed(ZkD2Smem& sm, uint32_t c, int lane) {
    __threadfence_block();
    __syncwarp();
    if (lane == 0) { ZK_VOL(sm.flushed[c & (ZK_D2_META - 1)]) = c + 1; zk_d2_help(sm); }
    __syncwarp();
}

// announce chunk c = [start_pos, end_pos) and the end position of each of its sequences (seq_end per lane)
__device__ __forceinline__ void zk_d2_announce(ZkD2Smem& sm, uint32_t c, uint32_t start_pos, uint32_t end_pos, uint32_t seq_end, uint32_t premask, int lane) {
    const uint32_t e = c & (ZK_D2_META - 1);
    ZK_VOL(sm.oe[e][lane]) = seq_end;
    if (lane == 0) { ZK_VOL(sm.start[e]) = start_pos; ZK_VOL(sm.end[e]) = end_pos; ZK_VOL(sm.dmask[e]) = premask; }
    __threadfence_block();
    __syncwarp();
    if (lane == 0) ZK_VOL(sm.started[e]) = c + 1;
    __syncwarp();
}
// sequences `mask` of chunk c are completely written
__device__ __forceinline__ void zk_d2_progress(ZkD2Smem& sm, uint32_t c, uint32_t mask, int lane) {
    __threadfence_block();
    __syncwarp();
    if (lane == 0 && mask) atomicOr(&sm.dmask[c & (ZK_D2_META - 1)], mask);
}

// warp-uniform wait until chunk c = [start_pos, end_pos) may start.  Returns false if the CTA aborted.
// exclusive == false: its end lies within `window` of flushed_pos (the in-flight region never laps the ring);
// exclusive == true: every earlier chunk is done and flushed (the chunk then runs alone, HBM to HBM).
__device__ __forceinline__ bool zk_d2_wait_start(ZkD2Smem& sm, uint32_t c, uint32_t start_pos, uint32_t end_pos, uint32_t window, bool exclusive, int lane) {
    for (;;) {
        uint32_t ok = 0, ab = 0;
        if (lane == 0) {
            ab = *(volatile int*)&sm.abort_code != 0;
            uint32_t fc = ZK_VOL(sm.flushed_chunk), fp = ZK_VOL(sm.flushed_pos);
            ok = exclusive ? (fc == c) : (fc == c || (end_pos - fp <= window && c - fc < ZK_D2_META - 2));
            if (!ok) {           // only then is it worth walking the flags (the walk was 6 % of the kernel's instructions when done on every entry)
                zk_d2_help(sm);
                fc = ZK_VOL(sm.flushed_chunk); fp = ZK_VOL(sm.flushed_pos);
                ok = exclusive ? (fc == c) : (fc == c || (end_pos - fp <= window && c - fc < ZK_D2_META - 2));
            }
            __threadfence_block();
        }
        ok = __shfl_sync(0xFFFFFFFFu, ok, 0); ab = __shfl_sync(0xFFFFFFFFu, ab, 0);
        __syncwarp();
        if (ab) return false;
        if (ok) return true;
        ZK_SPIN();
    }
}

template <int VARIANT>
__device__ __forceinline__ void zk_exec_body(ZkD2Smem& sm, const ZkDecodeArgs& a, uint32_t ring_bytes) {
    ZK_DYN_SMEM(ring_mem);
    const uint32_t e = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, W = blockDim.x >> 5;
    ZkEntry ent = a.entries[e];
    if (ent.status != 0 || a.counters->overflow) return;
    if (threadIdx.x == 0) { sm.done_pos = 0; sm.done_chunk = 0; sm.flushed_pos = 0; sm.flushed_chunk = 0; sm.abort_code = 0; }
    for (uint32_t i = threadIdx.x; i < ZK_D2_META; i += blockDim.x) { sm.started[i] = 0; sm.done[i] = 0; sm.flushed[i] = 0; sm.litdone[i] = 0; }
    __syncthreads();
    uint8_t* out = a.dst + a.d_off[e];
    const unsigned long long cap64 = a.d_off[e + 1] - a.d_off[e];
    const uint32_t cap = cap64 > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)cap64;
    const uint8_t* ebase = a.comp + a.c_off[e];
    ZkRing rg; rg.ring = ring_mem; rg.mask = ring_bytes - 1; rg.mis = (uint32_t)((uintptr_t)out & 15); rg.out = out;
    const uint32_t half = ring_bytes >> 1;

    uint32_t pos = 0, zstart = 0, chunk_base = 0;
    uint32_t R0 = 1, R1 = 4, R2 = 8;
    uint32_t preannounced = 0xFFFFFFFFu;          // chunk id this warp has already announced ahead of time
    // range reads: stop at the first block boundary at or after the wanted prefix (every warp takes the same decision)
    const uint32_t need = a.d_need ? a.d_need[e] : 0xFFFFFFFFu;
    bool stopped = false;
    for (uint32_t bi = 0; bi < ent.n_blocks; bi++) {
        if (zk_d2_aborted(sm)) break;
        if (pos >= need) { stopped = true; break; }
        const uint32_t bidx = ent.first_block + bi;
        const ZkBlock blk = a.blocks[bidx];
        if (blk.flags & ZKB_FIRST) { R0 = 1; R1 = 4; R2 = 8; zstart = pos; }
        if (blk.status != 0 || blk.lit_status != 0) { zk_d2_abort(sm, blk.status ? -blk.status : -blk.lit_status); break; }
        const bool has_seq = blk.type == 2 && blk.nseq > 0;
        const uint32_t nchunks = has_seq ? (blk.nseq + 31) / 32 + 1 : 1;
        if ((unsigned long long)pos + blk.regen > cap) { zk_d2_abort(sm, ZKZ_DST_TOO_SMALL); break; }
        // first chunk index of this block that belongs to this warp
        uint32_t c = chunk_base + ((uint32_t)warp + W - (chunk_base % W)) % W;
        for (; c < chunk_base + nchunks; c += W) {
            const uint32_t j = c - chunk_base;
            if (!has_seq) {
                // ---------------- Raw block / RLE block / literals-only compressed block: direct path, runs alone
                if (!zk_d2_wait_start(sm, c, pos, pos + blk.regen, 0, true, lane)) break;
                zk_d2_announce(sm, c, pos, pos + blk.regen, pos + blk.regen, 0u, lane);
                if (blk.type == 0) zk_warp_copy(out + pos, ebase + blk.src, blk.size, lane);
                else if (blk.type == 1) zk_warp_fill(out + pos, ebase[blk.src], blk.size, lane);
                else if (blk.lit_kind == 1) zk_warp_fill(out + pos, blk.lit_byte, blk.lit_size, lane);
                else zk_warp_copy(out + pos, blk.lit_kind == 0 ? ebase + blk.lit_src : a.lit + blk.lit_base, blk.lit_size, lane);
                __syncwarp();
                { uint32_t en = pos + blk.regen; zk_ring_reload(rg, en > half ? en - half : 0, en, lane, 32); }
                zk_d2_mark_done(sm, c, lane);
                zk_d2_mark_flushed(sm, c, lane);
                continue;
            }
            const uint32_t* s_lit = a.seq_lit_end + blk.seq_base;
            const uint32_t* s_out = a.seq_out_end + blk.seq_base;
            const uint8_t* lit = blk.lit_kind == 0 ? ebase + blk.lit_src : a.lit + blk.lit_base;
            if (j == nchunks - 1) {
                // ---------------- trailing literals of the block
                const uint32_t le = s_lit[blk.nseq - 1], oe = s_out[blk.nseq - 1];
                const uint32_t n = blk.lit_size - le, st0 = pos + oe, en = pos + blk.regen;
                const bool direct = n > half;
                if (!zk_d2_wait_start(sm, c, st0, en, half, direct, lane)) break;
                zk_d2_announce(sm, c, st0, en, en, 0u, lane);
                if (direct) {
                    if (blk.lit_kind == 1) zk_warp_fill(out + st0, blk.lit_byte, n, lane);
                    else zk_warp_copy(out + st0, lit + le, n, lane);
                    __syncwarp();
                    zk_ring_reload(rg, en - half, en, lane, 32);
                    zk_d2_mark_done(sm, c, lane);
                } else {
                    for (uint32_t i = lane; i < n; i += 32) rg.at(st0 + i) = blk.lit_kind == 1 ? blk.lit_byte : lit[le + i];
                    zk_d2_mark_done(sm, c, lane);
                    zk_ring_flush(rg, st0, en, lane);
                }
                zk_d2_mark_flushed(sm, c, lane);
                continue;
            }
            // ---------------- 32 sequences, one per lane
#if !defined(ZK_EMUL) && defined(ZK_EXEC_TRACE_BUILD)       // per-chunk clock64 stamps of entry 0 (tools/exec_trace.py): a debug build only --
#define ZK_STAMP(k) do { if (a.trace && e == 0 && c < 1024 && lane == 0) a.trace[c * 8 + (k)] = clock64(); } while (0)   // the checks were 3 % of the kernel's instructions
#else
#define ZK_STAMP(k) do { } while (0)
#endif
            ZK_STAMP(0);
            const uint32_t s = j * 32 + lane;
            const bool valid = s < blk.nseq;
            uint32_t le = 0, oe = 0, offv = 0;
            {   // lanes past the last sequence of the block repeat its cumulative ends (zero-length runs; keeps `le` monotone)
                const uint32_t sc = valid ? s : blk.nseq - 1;
                le = s_lit[sc]; oe = s_out[sc];
                if (valid) offv = a.seq_off[blk.seq_base + s];
            }
            uint32_t le_prev = __shfl_up_sync(0xFFFFFFFFu, le, 1), oe_prev = __shfl_up_sync(0xFFFFFFFFu, oe, 1);
            if (lane == 0) { le_prev = s ? s_lit[s - 1] : 0; oe_prev = s ? s_out[s - 1] : 0; }
            const uint32_t ll = le - le_prev, ml = (oe - oe_prev) - ll;
            const uint32_t o_lit = pos + oe_prev, md = o_lit + ll;          // entry-relative positions
            uint32_t off = offv;
            bool bad = false;
            if (valid) {
                if (offv & ZK_SYM) {
                    uint32_t sl = ZK_SYM_SLOT(offv), dl = ZK_SYM_DELTA(offv);
                    uint32_t r = sl == 0 ? R0 : (sl == 1 ? R1 : R2);
                    bad = r <= dl; off = r - dl;
                }
                if (off == 0 || off > md - zstart) bad = true;
            }
            if (__any_sync(0xFFFFFFFFu, bad)) { zk_d2_abort(sm, ZKZ_CORRUPTION); break; }
            const uint32_t chunk_start = pos + __shfl_sync(0xFFFFFFFFu, oe_prev, 0);
            const uint32_t chunk_end = pos + __shfl_sync(0xFFFFFFFFu, oe, min(31u, blk.nseq - 1 - j * 32));
            const bool direct = chunk_end - chunk_start > half;
            ZK_STAMP(1);
            if (!zk_d2_wait_start(sm, c, chunk_start, chunk_end, half, direct, lane)) break;
            if (preannounced != c) zk_d2_announce(sm, c, chunk_start, chunk_end, pos + oe, 0u, lane);
            // Announce this warp's NEXT chunk of the block right away (its sequence ends are one coalesced load away): chunks of
            // other warps that depend on it can then resolve their producers without waiting for this warp to get there.
            {
                const uint32_t jn = j + (uint32_t)W;
                if (jn < nchunks - 1) {
                    uint32_t okp = 0;
                    if (lane == 0) okp = (c + (uint32_t)W) - ZK_VOL(sm.flushed_chunk) < ZK_D2_META - 2;
                    if (__shfl_sync(0xFFFFFFFFu, okp, 0)) {
                        const uint32_t sn = jn * 32 + lane, scn = sn < blk.nseq ? sn : blk.nseq - 1;
                        const uint32_t oen = s_out[scn];
                        uint32_t stn = 0;
                        if (lane == 0) stn = s_out[jn * 32 - 1];
                        stn = __shfl_sync(0xFFFFFFFFu, stn, 0);
                        const uint32_t enn = __shfl_sync(0xFFFFFFFFu, oen, 31);
                        zk_d2_announce(sm, c + (uint32_t)W, pos + stn, pos + enn, pos + oen, 0u, lane);
                        preannounced = c + (uint32_t)W;
                    }
                }
            }
            ZK_STAMP(2);

            if (direct) {
                // ======== huge chunk: HBM -> HBM, alone in flight (it is the oldest chunk)
                {
                    // short runs byte-parallel; long runs with the vectorised warp copy
                    uint32_t longlit = __ballot_sync(0xFFFFFFFFu, valid && ll >= 256);
                    if (!longlit) zk_chunk_literals<false>(rg, lit, blk.lit_kind, blk.lit_byte, le, le_prev, o_lit, lane);
                    else {
                        if (valid && ll < 256) {
                            uint8_t* d = out + o_lit;
                            if (blk.lit_kind == 1) for (uint32_t i = 0; i < ll; i++) d[i] = blk.lit_byte;
                            else { const uint8_t* sp = lit + le_prev; for (uint32_t i = 0; i < ll; i++) d[i] = sp[i]; }
                        }
                        while (longlit) {
                            int l = __ffs((int)longlit) - 1; longlit &= longlit - 1;
                            uint32_t n = __shfl_sync(0xFFFFFFFFu, ll, l), d = __shfl_sync(0xFFFFFFFFu, o_lit, l), sp = __shfl_sync(0xFFFFFFFFu, le_prev, l);
                            if (blk.lit_kind == 1) zk_warp_fill(out + d, blk.lit_byte, n, lane);
                            else zk_warp_copy(out + d, lit + sp, n, lane);
                        }
                    }
                }
                __syncwarp();
                const uint32_t need_end = md - off + (ml < off ? ml : off);
                uint32_t pending = __ballot_sync(0xFFFFFFFFu, valid && ml > 0);
                while (pending) {
                    const int first = __ffs((int)pending) - 1;
                    const uint32_t frontier = __shfl_sync(0xFFFFFFFFu, md, first);
                    const bool mine = (pending >> lane) & 1;
                    const bool ready = mine && (need_end <= frontier || lane == first);
                    const uint32_t rmask = __ballot_sync(0xFFFFFFFFu, ready);
                    if (ready && ml < ZK_LONG) {
                        uint8_t* d = out + md; const uint8_t* sp = d - off;
                        for (uint32_t i = 0; i < ml; i++) d[i] = sp[i];
                    }
                    uint32_t longm = __ballot_sync(0xFFFFFFFFu, ready && ml >= ZK_LONG);
                    while (longm) {
                        int l = __ffs((int)longm) - 1; longm &= longm - 1;
                        uint32_t n = __shfl_sync(0xFFFFFFFFu, ml, l), d = __shfl_sync(0xFFFFFFFFu, md, l), o = __shfl_sync(0xFFFFFFFFu, off, l);
                        zk_warp_match(out + d, o, n, lane);
                    }
                    __syncwarp();
                    pending &= ~rmask;
                }
                zk_ring_reload(rg, chunk_end - half, chunk_end, lane, 32);
                zk_d2_mark_done(sm, c, lane);
                zk_d2_mark_flushed(sm, c, lane);
                continue;
            }

            // ======== normal chunk: build the output in the ring, then flush
            // literal runs: no dependencies (HBM scratch -> ring)
            zk_chunk_literals<true>(rg, lit, blk.lit_kind, blk.lit_byte, le, le_prev, o_lit, lane);
            {   // all literal runs are in place: sequences without a match (and the lanes past the last one) are complete
                const uint32_t withm = __ballot_sync(0xFFFFFFFFu, valid && ml > 0);
                zk_d2_progress(sm, c, ~withm, lane);
                if (lane == 0) ZK_VOL(sm.litdone[c & (ZK_D2_META - 1)]) = c + 1;
            }
            __syncwarp();
            ZK_STAMP(3);

            // matches.  near: the whole source is still resident in the ring (distance < R/2 from the chunk start);
            // far: it is read from HBM and must be published (done_pos).  A lane may go once its source is final.
            const uint32_t src0 = md - off;
            const bool near_src = src0 + half >= chunk_start;          // src0 >= chunk_start - R/2
            const uint32_t need_end = src0 + (ml < off ? ml : off);
            uint32_t pending = __ballot_sync(0xFFFFFFFFu, valid && ml > 0);
            bool aborted = false;
            // dataflow readiness: a match may go as soon as the bytes of its source are final -- the part that lies before this
            // chunk is tracked per chunk (descriptors in shared memory), the part inside this chunk by lane order.  Sources older
            // than R/2 are in HBM by construction of the start rule (flushed_pos >= chunk_end - R/2 > any far source).
            // Step 1 (once): which in-flight chunks [klo, khi] produce my source?  Step 2 (poll): are they done?  The poll loop is
            // the critical link of the frame's dependency chain, so it only reads those few flags.
            uint32_t klo = 1, khi = 0;                                  // empty range: nothing to wait for outside this chunk
            uint32_t mask_lo = 0, mask_hi = 0;                          // which sequences of chunk klo / khi produce my source
            {
                bool resolved = !(valid && ml > 0) || !near_src || src0 >= chunk_start;
                const uint32_t ne = need_end < chunk_start ? need_end : chunk_start;
                for (;;) {
                    if (!resolved) {
                        // chunk ids are consecutive and their start positions increase with the id: two binary searches over
                        // the in-flight chunks [dc, c) find the chunks holding src0 and ne-1 (a linear walk cost one shared-memory
                        // round trip per chunk of distance and dominated the kernel)
                        const uint32_t dp = ZK_VOL(sm.done_pos), dc = ZK_VOL(sm.done_chunk);
                        if (ne <= dp || dc >= c) { resolved = true; klo = 1; khi = 0; }
                        else {
                            bool ok = true;
                            uint32_t lo = dc, hi = c - 1;                       // khi = largest k with start[k] < ne (start[dc] == done_pos < ne)
                            while (lo < hi) {
                                const uint32_t mid = (lo + hi + 1) >> 1, e = mid & (ZK_D2_META - 1);
                                if (ZK_VOL(sm.started[e]) != mid + 1) { ok = false; break; }
                                if (ZK_VOL(sm.start[e]) < ne) lo = mid; else hi = mid - 1;
                            }
                            const uint32_t kh = lo;
                            lo = dc; hi = kh;                                   // klo = largest k <= khi with start[k] <= src0, else dc
                            while (ok && lo < hi) {
                                const uint32_t mid = (lo + hi + 1) >> 1, e = mid & (ZK_D2_META - 1);
                                if (ZK_VOL(sm.started[e]) != mid + 1) { ok = false; break; }
                                if (ZK_VOL(sm.start[e]) <= src0) lo = mid; else hi = mid - 1;
                            }
                            const uint32_t kl = lo;
                            if (ok && (ZK_VOL(sm.started[kl & (ZK_D2_META - 1)]) != kl + 1 || ZK_VOL(sm.started[kh & (ZK_D2_META - 1)]) != kh + 1)) ok = false;
                            if (ok) {
                                resolved = true; klo = kl; khi = kh;
                                // first sequence of klo whose end lies beyond src0; last sequence of khi that starts before ne
                                int a = 0, b = 0;
                                { const uint32_t e = klo & (ZK_D2_META - 1); int lo2 = 0, hi2 = 31;
                                  for (int st = 0; st < 5; st++) { int mid = (lo2 + hi2) >> 1; if (ZK_VOL(sm.oe[e][mid]) > src0) hi2 = mid; else lo2 = mid + 1; } a = lo2; }
                                { const uint32_t e = khi & (ZK_D2_META - 1); int lo2 = 0, hi2 = 31;
                                  for (int st = 0; st < 5; st++) { int mid = (lo2 + hi2) >> 1; if (ZK_VOL(sm.oe[e][mid]) >= ne) hi2 = mid; else lo2 = mid + 1; } b = lo2; }
                                mask_lo = 0xFFFFFFFFu << a;
                                mask_hi = b >= 31 ? 0xFFFFFFFFu : ((2u << b) - 1u);
                                if (klo == khi) { mask_lo &= mask_hi; mask_hi = mask_lo; }
                            }
                        }
                    }
                    if (__all_sync(0xFFFFFFFFu, resolved)) break;
                    if (zk_d2_aborted(sm)) { aborted = true; break; }
                    ZK_SPIN();
                }
            }
            ZK_STAMP(4);
            bool stamped5 = false;
            while (pending && !aborted) {
                const bool mine = (pending >> lane) & 1;
                bool ext_ok = true;
                if (mine && khi >= klo) {
                    const uint32_t dc = ZK_VOL(sm.done_chunk);
                    for (uint32_t k = khi + 1; k-- > klo;) {
                        if (k < dc) break;                                                   // it and everything older is done
                        const uint32_t e = k & (ZK_D2_META - 1);
                        const uint32_t need = k == khi ? mask_hi : (k == klo ? mask_lo : 0xFFFFFFFFu);
                        if (ZK_VOL(sm.started[e]) != k + 1 || ZK_VOL(sm.litdone[e]) != k + 1 || (ZK_VOL(sm.dmask[e]) & need) != need) { ext_ok = false; break; }
                    }
                    if (ext_ok) khi = 0, klo = 1;                       // sticky
                }
                const int first = __ffs((int)pending) - 1;
                const uint32_t md_first = __shfl_sync(0xFFFFFFFFu, md, first);   // inside this chunk everything below it is final
                const bool ready = mine && ext_ok && (need_end <= md_first || lane == first);
                const uint32_t rmask = __ballot_sync(0xFFFFFFFFu, ready);
                if (!rmask) { if (zk_d2_aborted(sm)) { aborted = true; break; } ZK_SPIN(); continue; }
                __threadfence_block();             // acquire: the flags were read before the data is
                if (!stamped5) { ZK_STAMP(5); stamped5 = true; }
                if (ready && ml < ZK_LONG) {
                    if (near_src) rg.copy_near(md, src0, ml);
                    else {   // far source (HBM, never overlapping): 8 bytes per round trip
                        const uint8_t* sp = out + src0;
                        for (uint32_t i = 0; i < ml; i += 8) {
                            unsigned long long v = zk_ld8_unaligned(sp + i);
                            const uint32_t nb = ml - i < 8 ? ml - i : 8;
                            for (uint32_t q = 0; q < nb; q++) { rg.at(md + i + q) = (uint8_t)v; v >>= 8; }
                        }
                    }
                }
                uint32_t longm = __ballot_sync(0xFFFFFFFFu, ready && ml >= ZK_LONG);
                while (longm) {
                    int l = __ffs((int)longm) - 1; longm &= longm - 1;
                    const uint32_t n = __shfl_sync(0xFFFFFFFFu, ml, l), d = __shfl_sync(0xFFFFFFFFu, md, l), o = __shfl_sync(0xFFFFFFFFu, off, l);
                    const bool nr = __shfl_sync(0xFFFFFFFFu, (uint32_t)near_src, l) != 0;
                    if (!nr) { const uint8_t* sp = out + (d - o); for (uint32_t i = lane; i < n; i += 32) rg.at(d + i) = sp[i]; }
                    else if (o >= n) { for (uint32_t i = lane; i < n; i += 32) rg.at(d + i) = rg.at(d - o + i); }
                    else if (o >= 32) {           // overlapping, period >= 32: 32 bytes per step are already final
                        for (uint32_t i0 = 0; i0 < n; i0 += 32) { uint32_t i = i0 + lane; if (i < n) rg.at(d + i) = rg.at(d - o + i); __syncwarp(); }
                    } else {                      // short period: replicate the pattern
                        for (uint32_t i = lane; i < n; i += 32) rg.at(d + i) = rg.at(d - o + (i % o));
                    }
                }
                zk_d2_progress(sm, c, rmask, lane);    // dependants of these sequences may go now (not only when the whole chunk is done)
                __syncwarp();
                pending &= ~rmask;
            }
            if (aborted) break;
            ZK_STAMP(6);
            zk_d2_mark_done(sm, c, lane);                          // dependants can read the ring now ...
            ZK_STAMP(7);
            zk_ring_flush(rg, chunk_start, chunk_end, lane);       // ... while the HBM flush happens off the critical chain
            zk_d2_mark_flushed(sm, c, lane);
        }
        // advance to the next block
        if (has_seq) {
            uint32_t v[3] = { blk.rep_out[0], blk.rep_out[1], blk.rep_out[2] }, n[3];
            for (int q = 0; q < 3; q++) {
                if (v[q] & ZK_SYM) { uint32_t sl = ZK_SYM_SLOT(v[q]); uint32_t r = sl == 0 ? R0 : (sl == 1 ? R1 : R2); n[q] = r - ZK_SYM_DELTA(v[q]); }
                else n[q] = v[q];
            }
            R0 = n[0]; R1 = n[1]; R2 = n[2];
        }
        pos += blk.regen;
        chunk_base += nchunks;
        if (blk.flags & ZKB_LAST) {
            if ((blk.flags & ZKB_HAS_FCS) && blk.fcs != (unsigned long long)(pos - zstart)) { zk_d2_abort(sm, ZKZ_CORRUPTION); break; }
            if (threadIdx.x == 0) { a.blocks[bidx].hash_start = zstart; a.blocks[bidx].hash_len = pos - zstart; }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int code = sm.abort_code;
        if (!code && !stopped && (unsigned long long)pos != cap64) code = pos < cap64 ? ZKZ_SRC_SIZE_WRONG : ZKZ_DST_TOO_SMALL;
        a.entries[e].status = code ? -code : 0;
        a.entries[e].produced = pos;
        if (code) atomicAdd(&a.counters->n_errors, 1u);
    }
}

// =============================================================================================
// K-D2 (second generation): the same job with in-order bookkeeping only.
//
// Profiling the dataflow kernel above (profiles/ncu_summary_bench_r1.txt) showed about 3 500 warp instructions per
// 32-sequence chunk at 15 warps per SM: it was bound by instruction issue, not by the dependency chain of a frame (a
// frame whose every chunk waits for its predecessor would still finish in ~2 ms at ~1 000 cycles per chunk).  This
// version keeps the shared-memory ring, the 32-sequence chunks dealt round-robin to the W warps of the CTA and the ring
// discipline (start rule, near / far sources, direct path for oversized chunks), and replaces the per-sequence dataflow
// (descriptor search, completion masks, pre-announcement) by ONE monotone counter:
//   done_pos     every byte below it is final in the ring (or in HBM, for the direct path);  a match may go as soon as
//                the part of its source that lies before its own chunk is below done_pos and the part inside its chunk
//                is below the chunk's own frontier (the destination of its first pending match);
//   the OLDEST unfinished chunk publishes its frontier after every round, so dependants in the next chunk start while it
//   is still running; finished chunks are published in order by whoever polls (per-chunk flags, "helping").
// About a fifth of the instructions per chunk, <= 64 registers, so 32 warps per SM stay resident.
// =============================================================================================
#define ZK_X2_META 64u
#define ZK_X2_G 1u                       // items per group (one warp runs a group's items back to back: only group boundaries cost a cross-warp hand-off)
struct ZkX2Smem {
    unsigned long long ev_done, ev_flush;  // events (mbarriers): done_pos / done_chunk moved; flushed_pos / flushed_chunk moved
    uint32_t done_pos, done_chunk;         // every byte below done_pos is final and readable; chunks [0, done_chunk) are done
    uint32_t flushed_pos, flushed_chunk;   // ... and below flushed_pos it is in HBM too (ring slots may be reused)
    int abort_code;
    uint32_t end[ZK_X2_META], done[ZK_X2_META], flushed[ZK_X2_META];   // slot = chunk & 63; valid for chunk k iff tag == k + 1 (end: written before done)
};
#define ZK_X2_HINT_NS 20000u               // upper bound of one sleep (a missed wake-up costs at most this)

__device__ __forceinline__ void zk_x2_abort(ZkX2Smem& sm, int code) {
    // exactly ONE thread of the CTA ever signals the abort: an event has an arrival count of one, and a warp-wide arrive
    // (32 arrivals in one instruction) would underflow it
    if (atomicCAS(&sm.abort_code, 0, code) == 0) {
        __threadfence_block();
        zk_event_signal(&sm.ev_done); zk_event_signal(&sm.ev_flush);
    }
}
__device__ __forceinline__ bool zk_x2_aborted(ZkX2Smem& sm) { return __any_sync(0xFFFFFFFFu, *(volatile int*)&sm.abort_code != 0); }

// advance the in-order prefixes as far as the per-chunk flags allow and wake the sleepers (called by whoever just set a flag)
__device__ __noinline__ void zk_x2_advance_done(ZkX2Smem& sm) {
    uint32_t dc = ZK_VOL(sm.done_chunk), dc0 = dc, dp = 0;
    while (ZK_VOL(sm.done[dc & (ZK_X2_META - 1)]) == dc + 1) { dp = ZK_VOL(sm.end[dc & (ZK_X2_META - 1)]); dc++; }
    if (dc != dc0) { atomicMax(&sm.done_pos, dp); __threadfence_block(); atomicMax(&sm.done_chunk, dc); __threadfence_block(); zk_event_signal(&sm.ev_done); }
}
__device__ __noinline__ void zk_x2_advance_flushed(ZkX2Smem& sm) {
    uint32_t fc = ZK_VOL(sm.flushed_chunk), fc0 = fc, fp = 0;
    while (ZK_VOL(sm.flushed[fc & (ZK_X2_META - 1)]) == fc + 1) { fp = ZK_VOL(sm.end[fc & (ZK_X2_META - 1)]); fc++; }
    if (fc != fc0) { atomicMax(&sm.flushed_pos, fp); __threadfence_block(); atomicMax(&sm.flushed_chunk, fc); __threadfence_block(); zk_event_signal(&sm.ev_flush); }
}

// warp-uniform wait until an item of group g (ending at end_pos) may start; false if the CTA aborted.
// exclusive: every earlier group is done and flushed (the item then runs alone, HBM to HBM; earlier items of the same group
// were flushed by this very warp).
__device__ __forceinline__ bool zk_x2_wait_start(ZkX2Smem& sm, uint32_t g, uint32_t end_pos, uint32_t window, bool exclusive, int lane) {
    uint32_t ok = 0;
    if (lane == 0) {
        uint32_t ph = 2;                                                     // parity not known yet
        for (;;) {
            const uint32_t fg = ZK_VOL(sm.flushed_chunk), fp = ZK_VOL(sm.flushed_pos);
            if (exclusive ? (fg == g) : (fg == g || (end_pos - fp <= window && g - fg < ZK_X2_META - 2))) { ok = 1; break; }
            if (*(volatile int*)&sm.abort_code != 0) break;
            if (ph == 2) { ph = zk_event_parity(&sm.ev_flush); continue; }   // learn the phase, then look again before sleeping
            if (zk_event_sleep(&sm.ev_flush, ph, ZK_X2_HINT_NS)) ph ^= 1;
        }
    }
    return __shfl_sync(0xFFFFFFFFu, ok, 0) != 0;
}
// lane 0: sleep until done_pos >= want (returns the value seen) or the CTA aborts (returns 0xFFFFFFFF)
__device__ __forceinline__ uint32_t zk_x2_wait_done_pos(ZkX2Smem& sm, uint32_t want) {
    uint32_t ph = 2;
    for (;;) {
        const uint32_t dp = ZK_VOL(sm.done_pos);
        if (dp >= want) return dp;
        if (*(volatile int*)&sm.abort_code != 0) return 0xFFFFFFFFu;
        if (ph == 2) { ph = zk_event_parity(&sm.ev_done); continue; }
        if (zk_event_sleep(&sm.ev_done, ph, ZK_X2_HINT_NS)) ph ^= 1;
    }
}
// an item of group g, ending at end_pos, is final in the ring (or in HBM).  The last item of a group publishes the group;
// before that, the OLDEST group publishes its progress item by item (dependants need not wait for the whole group).
__device__ __forceinline__ void zk_x2_item_done(ZkX2Smem& sm, uint32_t g, uint32_t end_pos, bool last, int lane) {
    __threadfence_block();
    __syncwarp();
    if (lane == 0) {
        if (last) { ZK_VOL(sm.end[g & (ZK_X2_META - 1)]) = end_pos; __threadfence_block(); ZK_VOL(sm.done[g & (ZK_X2_META - 1)]) = g + 1; __threadfence_block(); zk_x2_advance_done(sm); }
        else if (ZK_VOL(sm.done_chunk) == g && end_pos > ZK_VOL(sm.done_pos)) { atomicMax(&sm.done_pos, end_pos); __threadfence_block(); zk_event_signal(&sm.ev_done); }
    }
}
__device__ __forceinline__ void zk_x2_item_flushed(ZkX2Smem& sm, uint32_t g, uint32_t end_pos, bool last, int lane) {
    __threadfence_block();
    __syncwarp();
    if (lane == 0) {
        if (last) { ZK_VOL(sm.flushed[g & (ZK_X2_META - 1)]) = g + 1; __threadfence_block(); zk_x2_advance_flushed(sm); }
        else if (ZK_VOL(sm.flushed_chunk) == g && end_pos > ZK_VOL(sm.flushed_pos)) { atomicMax(&sm.flushed_pos, end_pos); __threadfence_block(); zk_event_signal(&sm.ev_flush); }
    }
    __syncwarp();
}

__device__ __forceinline__ void zk_exec2_body(ZkX2Smem& sm, const ZkDecodeArgs& a, uint32_t ring_bytes) {
    ZK_DYN_SMEM(ring_mem);
    const uint32_t e = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, W = blockDim.x >> 5;
    ZkEntry ent = a.entries[e];
    if (ent.status != 0 || a.counters->overflow) return;
    if (threadIdx.x == 0) { sm.done_pos = 0; sm.done_chunk = 0; sm.flushed_pos = 0; sm.flushed_chunk = 0; sm.abort_code = 0; zk_event_init(&sm.ev_done); zk_event_init(&sm.ev_flush); }
    for (uint32_t i = threadIdx.x; i < ZK_X2_META; i += blockDim.x) { sm.done[i] = 0; sm.flushed[i] = 0; sm.end[i] = 0; }
    __syncthreads();
    uint8_t* out = a.dst + a.d_off[e];
    const unsigned long long cap64 = a.d_off[e + 1] - a.d_off[e];
    const uint32_t cap = cap64 > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)cap64;
    const uint8_t* ebase = a.comp + a.c_off[e];
    ZkRing rg; rg.ring = ring_mem; rg.mask = ring_bytes - 1; rg.mis = (uint32_t)((uintptr_t)out & 15); rg.out = out;
    const uint32_t half = ring_bytes >> 1;

    uint32_t pos = 0, zstart = 0, chunk_base = 0, gstart = 0;
    uint32_t R0 = 1, R1 = 4, R2 = 8;
    const uint32_t need = a.d_need ? a.d_need[e] : 0xFFFFFFFFu;      // range reads: stop at the first block boundary at or after the wanted prefix
    bool stopped = false;
    for (uint32_t bi = 0; bi < ent.n_blocks; bi++) {
        if (zk_x2_aborted(sm)) break;
        if (pos >= need) { stopped = true; break; }
        const uint32_t bidx = ent.first_block + bi;
        const ZkBlock blk = a.blocks[bidx];
        if (blk.flags & ZKB_FIRST) { R0 = 1; R1 = 4; R2 = 8; zstart = pos; }
        if (blk.status != 0 || blk.lit_status != 0) { zk_x2_abort(sm, blk.status ? -blk.status : -blk.lit_status); break; }
        const bool has_seq = blk.type == 2 && blk.nseq > 0;
        const uint32_t nchunks = has_seq ? (blk.nseq + 31) / 32 + 1 : 1;
        if ((unsigned long long)pos + blk.regen > cap) { zk_x2_abort(sm, ZKZ_DST_TOO_SMALL); break; }
        // items (32-sequence chunks, trailing literals, whole non-sequence blocks) are numbered through the entry; ZK_X2_G
        // consecutive items form a group, group g belongs to warp g % W, which runs its items one after the other
        const uint32_t g_lo = chunk_base / ZK_X2_G;
        for (uint32_t g = g_lo + ((uint32_t)warp + (uint32_t)W - g_lo % (uint32_t)W) % (uint32_t)W; g * ZK_X2_G < chunk_base + nchunks; g += (uint32_t)W)
        for (uint32_t c = g * ZK_X2_G > chunk_base ? g * ZK_X2_G : chunk_base; c < (g + 1) * ZK_X2_G && c < chunk_base + nchunks; c++) {
            const uint32_t j = c - chunk_base;
            const bool glast = (c + 1) % ZK_X2_G == 0;                       // (the entry's last, incomplete group is closed after the loop)
            if (!has_seq) {
                // ---------------- Raw block / RLE block / literals-only compressed block: direct path, runs alone
                if (c % ZK_X2_G == 0) gstart = pos;
                if (!zk_x2_wait_start(sm, g, pos + blk.regen, 0, true, lane)) break;
                if (blk.type == 0) zk_warp_copy(out + pos, ebase + blk.src, blk.size, lane);
                else if (blk.type == 1) zk_warp_fill(out + pos, ebase[blk.src], blk.size, lane);
                else if (blk.lit_kind == 1) zk_warp_fill(out + pos, blk.lit_byte, blk.lit_size, lane);
                else zk_warp_copy(out + pos, blk.lit_kind == 0 ? ebase + blk.lit_src : a.lit + blk.lit_base, blk.lit_size, lane);
                __syncwarp();
                { uint32_t en = pos + blk.regen; zk_ring_reload(rg, en > half ? en - half : 0, en, lane, 32); }
                zk_x2_item_done(sm, g, pos + blk.regen, glast, lane);
                zk_x2_item_flushed(sm, g, pos + blk.regen, glast, lane);
                continue;
            }
            const uint32_t* s_lit = a.seq_lit_end + blk.seq_base;
            const uint32_t* s_out = a.seq_out_end + blk.seq_base;
            const uint8_t* lit = blk.lit_kind == 0 ? ebase + blk.lit_src : a.lit + blk.lit_base;
            if (j == nchunks - 1) {
                // ---------------- trailing literals of the block
                const uint32_t le = s_lit[blk.nseq - 1], oe = s_out[blk.nseq - 1];
                const uint32_t n = blk.lit_size - le, st0 = pos + oe, en = pos + blk.regen;
                const bool direct = n > half;
                if (c % ZK_X2_G == 0) gstart = st0;
                if (!zk_x2_wait_start(sm, g, en, half, direct, lane)) break;
                if (direct) {
                    if (blk.lit_kind == 1) zk_warp_fill(out + st0, blk.lit_byte, n, lane);
                    else zk_warp_copy(out + st0, lit + le, n, lane);
                    __syncwarp();
                    zk_ring_reload(rg, en - half, en, lane, 32);
                    zk_x2_item_done(sm, g, en, glast, lane);
                } else {
                    for (uint32_t i = lane; i < n; i += 32) rg.at(st0 + i) = blk.lit_kind == 1 ? blk.lit_byte : lit[le + i];
                    zk_x2_item_done(sm, g, en, glast, lane);
                    __syncwarp();
                    zk_ring_flush(rg, st0, en, lane);
                }
                zk_x2_item_flushed(sm, g, en, glast, lane);
                continue;
            }
            // ---------------- 32 sequences, one per lane (all loads issued before the first use)
            const uint32_t s = j * 32 + lane;
            const bool valid = s < blk.nseq;
            const uint32_t sc = valid ? s : blk.nseq - 1;      // lanes past the last sequence repeat its cumulative ends (zero-length runs)
            const uint32_t le = s_lit[sc], oe = s_out[sc];
            const uint32_t offv = valid ? a.seq_off[blk.seq_base + s] : 0u;
            uint32_t le_first = 0, oe_first = 0;
            if (lane == 0 && s) { le_first = s_lit[s - 1]; oe_first = s_out[s - 1]; }
            uint32_t le_prev = __shfl_up_sync(0xFFFFFFFFu, le, 1), oe_prev = __shfl_up_sync(0xFFFFFFFFu, oe, 1);
            if (lane == 0) { le_prev = le_first; oe_prev = oe_first; }
            const uint32_t ll = le - le_prev; uint32_t ml = (oe - oe_prev) - ll;
            const uint32_t o_lit = pos + oe_prev; uint32_t md = o_lit + ll;  // entry-relative positions (md / ml shrink to the in-frame part of a prefix match below)
            uint32_t off = offv;
            bool bad = false;
            if (valid) {
                if (offv & ZK_SYM) {
                    const uint32_t sl = ZK_SYM_SLOT(offv), dl = ZK_SYM_DELTA(offv);
                    const uint32_t r = sl == 0 ? R0 : (sl == 1 ? R1 : R2);
                    bad = r <= dl; off = r - dl;
                }
                if (off == 0 || off > md - zstart + a.prefix_len) bad = true;
            }
            if (__any_sync(0xFFFFFFFFu, bad)) { zk_x2_abort(sm, ZKZ_CORRUPTION); break; }
            const uint32_t chunk_start = pos + __shfl_sync(0xFFFFFFFFu, oe_prev, 0);
            const uint32_t chunk_end = pos + __shfl_sync(0xFFFFFFFFu, oe, 31);
            const bool direct = chunk_end - chunk_start > half;
            if (c % ZK_X2_G == 0) gstart = chunk_start;
            if (!glast && j + 2 < nchunks) {      // the next item is this warp's too: pull its sequences and the start of its literals towards L1
                const uint32_t le_last = __shfl_sync(0xFFFFFFFFu, le, 31);
                if (lane == 0) { zk_prefetch_l1(s_lit + s + 32); zk_prefetch_l1(s_out + s + 32); zk_prefetch_l1(a.seq_off + blk.seq_base + s + 32); }
                if (lane >= 4 && lane < 8 && blk.lit_kind != 1) zk_prefetch_l1(lit + le_last + (uint32_t)(lane - 4) * 64u);
            }
            if (!zk_x2_wait_start(sm, g, chunk_end, half, direct, lane)) break;

            if (direct) {
                // ======== huge chunk: HBM -> HBM, alone in flight (it is the oldest chunk and everything before it is flushed)
                {
                    uint32_t longlit = __ballot_sync(0xFFFFFFFFu, valid && ll >= 256);
                    if (!longlit) zk_chunk_literals<false>(rg, lit, blk.lit_kind, blk.lit_byte, le, le_prev, o_lit, lane);
                    else {
                        if (valid && ll < 256) {
                            uint8_t* d = out + o_lit;
                            if (blk.lit_kind == 1) for (uint32_t i = 0; i < ll; i++) d[i] = blk.lit_byte;
                            else { const uint8_t* sp = lit + le_prev; for (uint32_t i = 0; i < ll; i++) d[i] = sp[i]; }
                        }
                        while (longlit) {
                            const int l = __ffs((int)longlit) - 1; longlit &= longlit - 1;
                            const uint32_t n = __shfl_sync(0xFFFFFFFFu, ll, l), d = __shfl_sync(0xFFFFFFFFu, o_lit, l), sp = __shfl_sync(0xFFFFFFFFu, le_prev, l);
                            if (blk.lit_kind == 1) zk_warp_fill(out + d, blk.lit_byte, n, lane);
                            else zk_warp_copy(out + d, lit + sp, n, lane);
                        }
                    }
                }
                if (valid && ml > 0 && off > md - zstart) {          // the match starts in the prefix
                    const uint32_t back = off - (md - zstart), la = ml < back ? ml : back;
                    const uint8_t* ps = a.prefix + (a.prefix_len - back);
                    for (uint32_t i = 0; i < la; i++) out[md + i] = ps[i];
                    md += la; ml -= la;
                }
                __threadfence_block();
                __syncwarp();
                const uint32_t need_end = md - off + (ml < off ? ml : off);
                uint32_t pending = __ballot_sync(0xFFFFFFFFu, valid && ml > 0);
                while (pending) {
                    const int first = __ffs((int)pending) - 1;
                    const uint32_t frontier = __shfl_sync(0xFFFFFFFFu, md, first);
                    const bool mine = (pending >> lane) & 1;
                    const bool ready = mine && (need_end <= frontier || lane == first);
                    const uint32_t rmask = __ballot_sync(0xFFFFFFFFu, ready);
                    if (ready && ml < ZK_LONG) {
                        uint8_t* d = out + md; const uint8_t* sp = d - off;
                        for (uint32_t i = 0; i < ml; i++) d[i] = sp[i];
                    }
                    uint32_t longm = __ballot_sync(0xFFFFFFFFu, ready && ml >= ZK_LONG);
                    while (longm) {
                        const int l = __ffs((int)longm) - 1; longm &= longm - 1;
                        const uint32_t n = __shfl_sync(0xFFFFFFFFu, ml, l), d = __shfl_sync(0xFFFFFFFFu, md, l), o = __shfl_sync(0xFFFFFFFFu, off, l);
                        zk_warp_match(out + d, o, n, lane);
                    }
                    __threadfence_block();
                    __syncwarp();
                    pending &= ~rmask;
                }
                zk_ring_reload(rg, chunk_end - half, chunk_end, lane, 32);
                zk_x2_item_done(sm, g, chunk_end, glast, lane);
                zk_x2_item_flushed(sm, g, chunk_end, glast, lane);
                continue;
            }

            // ======== normal chunk: build the output in the ring, then flush
            zk_chunk_literals<true>(rg, lit, blk.lit_kind, blk.lit_byte, le, le_prev, o_lit, lane);      // no dependencies
            if (a.prefix_len && valid && ml > 0 && off > md - zstart) {
                // the match starts in the raw-content prefix that precedes every zstd frame: that part is constant data, copied now;
                // what is left of the match (if anything) starts at the frame's first byte and is an ordinary match
                const uint32_t back = off - (md - zstart), la = ml < back ? ml : back;
                const uint8_t* ps = a.prefix + (a.prefix_len - back);
                for (uint32_t i = 0; i < la; i++) rg.at(md + i) = ps[i];
                md += la; ml -= la;
            }
            // matches.  near: the source is still resident in the ring (distance < R/2 from the chunk start); far: it is in HBM
            // (flushed, by the start rule) and has no dependency on anything in flight.
            const uint32_t src0 = md - off;
            const bool has_m = valid && ml > 0;
            const bool near_src = src0 + half >= chunk_start;
            const uint32_t need_end = src0 + (ml < off ? ml : off);
            const bool ext_dep = near_src && src0 < gstart;                            // part of the source was produced by OTHER warps' groups
            const uint32_t ext_need = need_end < gstart ? need_end : gstart;           // (earlier items of this group are final: program order)
            bool aborted = false;
            // ---- far matches first: nothing to wait for.  Short ones lane by lane with all the loads of up to 16 bytes in flight at
            // once (one round trip for most matches), long ones by the whole warp.
            {
                const bool far_m = has_m && !near_src;
                if (far_m && ml < ZK_LONG) {
                    const uint8_t* sp = out + src0;
                    for (uint32_t i = 0; i < ml; i += 16) {
                        const unsigned long long v0 = zk_ld8_unaligned(sp + i), v1 = ml - i > 8 ? zk_ld8_unaligned(sp + i + 8) : 0ull;
                        rg.st8(md + i, (uint32_t)v0, (uint32_t)(v0 >> 32), ml - i);
                        if (ml - i > 8) rg.st8(md + i + 8, (uint32_t)v1, (uint32_t)(v1 >> 32), ml - i - 8);
                    }
                }
                uint32_t longf = __ballot_sync(0xFFFFFFFFu, far_m && ml >= ZK_LONG);
                while (longf) {
                    const int l = __ffs((int)longf) - 1; longf &= longf - 1;
                    const uint32_t n = __shfl_sync(0xFFFFFFFFu, ml, l), d = __shfl_sync(0xFFFFFFFFu, md, l), o = __shfl_sync(0xFFFFFFFFu, off, l);
                    const uint8_t* sp = out + (d - o);
                    for (uint32_t i = lane; i < n; i += 32) rg.at(d + i) = sp[i];
                }
            }
            uint32_t pending = __ballot_sync(0xFFFFFFFFu, has_m && near_src);
            __threadfence_block();
            __syncwarp();                                                              // literals and far matches are visible to every lane
            uint32_t dp = __shfl_sync(0xFFFFFFFFu, ZK_VOL(sm.done_pos), 0);          // one reading for the whole warp (the branches below must be uniform)
            while (pending) {
                const int first = __ffs((int)pending) - 1;
                const uint32_t frontier = __shfl_sync(0xFFFFFFFFu, md, first);       // inside this chunk everything below it is final
                const bool mine = (pending >> lane) & 1;
                const bool int_ok = mine && need_end <= frontier;                      // (always true for the first pending lane)
                // the smallest done_pos that lets some lane go; sleep until it is reached (one lane sleeps, the warp issues nothing)
                const uint32_t want = __reduce_min_sync(0xFFFFFFFFu, int_ok ? (ext_dep ? ext_need : 0u) : 0xFFFFFFFFu);
                if (want > dp) {
                    uint32_t v = 0;
                    if (lane == 0) v = zk_x2_wait_done_pos(sm, want);
                    dp = __shfl_sync(0xFFFFFFFFu, v, 0);
                    if (dp == 0xFFFFFFFFu) { aborted = true; break; }
                    __threadfence_block();         // acquire: done_pos was read before the data is
                }
                const bool ready = int_ok && (!ext_dep || ext_need <= dp);
                const uint32_t rmask = __ballot_sync(0xFFFFFFFFu, ready);
                if (ready && ml < ZK_LONG) rg.copy_near(md, src0, ml);
                uint32_t longm = __ballot_sync(0xFFFFFFFFu, ready && ml >= ZK_LONG);
                while (longm) {
                    const int l = __ffs((int)longm) - 1; longm &= longm - 1;
                    const uint32_t n = __shfl_sync(0xFFFFFFFFu, ml, l), d = __shfl_sync(0xFFFFFFFFu, md, l), o = __shfl_sync(0xFFFFFFFFu, off, l);
                    if (o >= n) { for (uint32_t i = lane; i < n; i += 32) rg.at(d + i) = rg.at(d - o + i); }
                    else if (o >= 32) {           // overlapping, period >= 32: 32 bytes per step are already final
                        for (uint32_t i0 = 0; i0 < n; i0 += 32) { const uint32_t i = i0 + lane; if (i < n) rg.at(d + i) = rg.at(d - o + i); __syncwarp(); }
                    } else {                      // short period: replicate the pattern
                        for (uint32_t i = lane; i < n; i += 32) rg.at(d + i) = rg.at(d - o + (i % o));
                    }
                }
                pending &= ~rmask;
                __threadfence_block();
                __syncwarp();
                // the oldest unfinished chunk publishes its frontier: dependants in later chunks need not wait for the whole chunk
                if (pending) {
                    const uint32_t nf = __shfl_sync(0xFFFFFFFFu, md, __ffs((int)pending) - 1);
                    if (lane == 0 && ZK_VOL(sm.done_chunk) == g && nf > ZK_VOL(sm.done_pos)) {
                        atomicMax(&sm.done_pos, nf); __threadfence_block(); zk_event_signal(&sm.ev_done);
                    }
                }
            }
            if (aborted) break;
            zk_x2_item_done(sm, g, chunk_end, glast, lane);        // dependants can read the ring now ...
            __syncwarp();
            zk_ring_flush(rg, chunk_start, chunk_end, lane);       // ... while the HBM flush happens off the critical chain
            zk_x2_item_flushed(sm, g, chunk_end, glast, lane);
        }
        // advance to the next block
        if (has_seq) {
            uint32_t v[3] = { blk.rep_out[0], blk.rep_out[1], blk.rep_out[2] }, n[3];
            for (int q = 0; q < 3; q++) {
                if (v[q] & ZK_SYM) { const uint32_t sl = ZK_SYM_SLOT(v[q]); const uint32_t r = sl == 0 ? R0 : (sl == 1 ? R1 : R2); n[q] = r - ZK_SYM_DELTA(v[q]); }
                else n[q] = v[q];
            }
            R0 = n[0]; R1 = n[1]; R2 = n[2];
        }
        pos += blk.regen;
        chunk_base += nchunks;
        if (blk.flags & ZKB_LAST) {
            if ((blk.flags & ZKB_HAS_FCS) && blk.fcs != (unsigned long long)(pos - zstart)) { zk_x2_abort(sm, ZKZ_CORRUPTION); break; }
            if (threadIdx.x == 0) { a.blocks[bidx].hash_start = zstart; a.blocks[bidx].hash_len = pos - zstart; }
        }
    }
    if (chunk_base % ZK_X2_G && (chunk_base / ZK_X2_G) % (uint32_t)W == (uint32_t)warp && !zk_x2_aborted(sm)) {
        // the entry's last group has fewer than ZK_X2_G items: its owner closes it (nobody waits on it any more, but the
        // in-order prefixes stay exact)
        zk_x2_item_done(sm, chunk_base / ZK_X2_G, pos, true, lane);
        zk_x2_item_flushed(sm, chunk_base / ZK_X2_G, pos, true, lane);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int code = sm.abort_code;
        if (!code && !stopped && (unsigned long long)pos != cap64) code = pos < cap64 ? ZKZ_SRC_SIZE_WRONG : ZKZ_DST_TOO_SMALL;
        a.entries[e].status = code ? -code : 0;
        a.entries[e].produced = pos;
        if (code) atomicAdd(&a.counters->n_errors, 1u);
    }
}

__global__ void __launch_bounds__(1024, 1) zk_exec2_kernel(ZkDecodeArgs a, uint32_t ring_bytes) {
    __shared__ ZkX2Smem sm;
    zk_exec2_body(sm, a, ring_bytes);
}

// Two register budgets for the same body: up to 16 warps per entry (<= 128 registers, few entries per SM), and a
// 5-warp variant compiled for 4 CTAs per SM (<= 102 registers) for large batches, where every entry of the batch should
// stay resident and the warps per SM are what hides the latency.
__global__ void __launch_bounds__(512, 1) zk_exec_kernel(ZkDecodeArgs a, uint32_t ring_bytes) {
    __shared__ ZkD2Smem sm;
    zk_exec_body<0>(sm, a, ring_bytes);
}
__global__ void __launch_bounds__(160, 4) zk_exec_kernel_w5(ZkDecodeArgs a, uint32_t ring_bytes) {
    __shared__ ZkD2Smem sm;
    zk_exec_body<1>(sm, a, ring_bytes);
}

// =============================================================================================
// K-D3: XXH64 content checksum (A.8), one warp per entry, lanes 0..3 carry the four accumulators
// =============================================================================================
__global__ void __launch_bounds__(128) zk_xxh64_kernel(ZkDecodeArgs a) {
    const int lane = threadIdx.x & 31;
    const uint32_t e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (e >= a.n_entries) return;
    ZkEntry ent = a.entries[e];
    if (ent.status != 0 || a.counters->overflow) return;
    if (a.d_need && (unsigned long long)a.d_need[e] < a.d_off[e + 1] - a.d_off[e]) return;   // a prefix only: no checksum, as the reference (decode.rs:425-427)
    const uint8_t* out = a.dst + a.d_off[e];
    const uint8_t* ebase = a.comp + a.c_off[e];
    for (uint32_t bi = 0; bi < ent.n_blocks; bi++) {
        const ZkBlock* blk = &a.blocks[ent.first_block + bi];
        uint32_t flags = blk->flags;
        if ((flags & (ZKB_LAST | ZKB_HAS_CSUM)) != (ZKB_LAST | ZKB_HAS_CSUM)) continue;
        uint32_t content = blk->type == 1 ? 1u : blk->size;
        uint32_t want = zk_ld_le32(ebase + blk->src + content);
        unsigned long long h = zk_warp_xxh64(out + blk->hash_start, blk->hash_len, lane);
        if ((uint32_t)h != want) {
            if (lane == 0) { a.entries[e].status = -ZKZ_CHECKSUM_WRONG; atomicAdd(&a.counters->n_errors, 1u); }
            return;
        }
    }
}

// =============================================================================================
// host-side launcher
// =============================================================================================
#ifndef ZK_EMUL
#define ZK_CUDA_OK(x) do { cudaError_t err__ = (x); if (err__ != cudaSuccess) { zk_note_cuda_error(#x, (int)err__); return ZK_INT_CUDA; } } while (0)
#else
#define ZK_CUDA_OK(x) do { (void)(x); } while (0)
#endif

static int zk_grow(void** p, size_t* cap, size_t need, size_t elem) {
    if (*cap >= need && *p) return 0;
    if (*p) cudaFree(*p);
    *p = nullptr; *cap = 0;
    size_t want = need + need / 8 + 64;
    cudaError_t ce = cudaMalloc(p, want * elem);
    if (ce != cudaSuccess) { fprintf(stderr, "zeekstd_b200: cudaMalloc(%zu bytes) failed in the decode workspace: %s\n", want * elem, cudaGetErrorString(ce)); (void)cudaGetLastError(); *p = nullptr; return -(int)ZKZ_MEMORY_ALLOCATION; }
    *cap = want;
    return 0;
}

void zk_decode_ws_free(ZkDecodeWs* ws) {
    void* ptrs[] = { ws->blocks, ws->entries, ws->counters, ws->lit, ws->seq_lit_end, ws->seq_out_end, ws->seq_off, ws->c_off, ws->d_off,
                     ws->huf_list, ws->seq_list, ws->d_need };
    for (void* p : ptrs) if (p) cudaFree(p);
    if (ws->h_need) cudaFreeHost(ws->h_need);
    if (ws->h_entries) cudaFreeHost(ws->h_entries);
    if (ws->h_counters) cudaFreeHost(ws->h_counters);
    if (ws->h_off) cudaFreeHost(ws->h_off);
    if (ws->side) cudaStreamDestroy(ws->side);
    if (ws->ev_scan) cudaEventDestroy(ws->ev_scan);
    if (ws->ev_huf) cudaEventDestroy(ws->ev_huf);
    if (ws->ev_up) cudaEventDestroy(ws->ev_up);
    if (ws->ev_done) cudaEventDestroy(ws->ev_done);
    if (ws->ev_down) cudaEventDestroy(ws->ev_down);
    ws->prof.destroy();
    *ws = ZkDecodeWs();
}

static int zk_decode_ensure(ZkDecodeWs* ws, uint32_t n, size_t need_blocks, size_t need_lit, size_t need_seq) {
    int rc;
    size_t cap;
    if (ws->cap_blocks < need_blocks || !ws->blocks) {
        size_t c1 = ws->cap_blocks, c2 = ws->cap_blocks, c3 = ws->cap_blocks;
        if ((rc = zk_grow((void**)&ws->blocks, &c1, need_blocks, sizeof(ZkBlock)))) return rc;
        if ((rc = zk_grow((void**)&ws->huf_list, &c2, need_blocks, 4))) return rc;
        if ((rc = zk_grow((void**)&ws->seq_list, &c3, need_blocks, 4))) return rc;
        ws->cap_blocks = c1 < c2 ? (c1 < c3 ? c1 : c3) : (c2 < c3 ? c2 : c3);
    }
    cap = ws->cap_lit; if ((rc = zk_grow((void**)&ws->lit, &cap, need_lit + 64, 1))) return rc; ws->cap_lit = cap;
    if (ws->cap_seq < need_seq || !ws->seq_off) {
        size_t c1 = ws->cap_seq, c2 = ws->cap_seq, c3 = ws->cap_seq;
        if ((rc = zk_grow((void**)&ws->seq_lit_end, &c1, need_seq, 4))) return rc;
        if ((rc = zk_grow((void**)&ws->seq_out_end, &c2, need_seq, 4))) return rc;
        if ((rc = zk_grow((void**)&ws->seq_off, &c3, need_seq, 4))) return rc;
        ws->cap_seq = c1 < c2 ? (c1 < c3 ? c1 : c3) : (c2 < c3 ? c2 : c3);
    }
    if (ws->cap_entries < n || !ws->entries) {
        size_t c = ws->cap_entries;
        if ((rc = zk_grow((void**)&ws->entries, &c, n, sizeof(ZkEntry)))) return rc;
        size_t c2 = 0, c3 = 0;
        if (ws->c_off) { cudaFree(ws->c_off); ws->c_off = nullptr; }
        if (ws->d_off) { cudaFree(ws->d_off); ws->d_off = nullptr; }
        if ((rc = zk_grow((void**)&ws->c_off, &c2, c + 1, 8))) return rc;
        if ((rc = zk_grow((void**)&ws->d_off, &c3, c + 1, 8))) return rc;
        if (ws->h_entries) cudaFreeHost(ws->h_entries);
        if (ws->h_off) cudaFreeHost(ws->h_off);
        if (cudaMallocHost((void**)&ws->h_entries, c * sizeof(ZkEntry)) != cudaSuccess) return -(int)ZKZ_MEMORY_ALLOCATION;
        if (cudaMallocHost((void**)&ws->h_off, 2 * (c + 1) * 8) != cudaSuccess) return -(int)ZKZ_MEMORY_ALLOCATION;
        if (ws->d_need) { cudaFree(ws->d_need); ws->d_need = nullptr; }
        if (ws->h_need) { cudaFreeHost(ws->h_need); ws->h_need = nullptr; }
        if (cudaMalloc((void**)&ws->d_need, (c + 1) * 4) != cudaSuccess) return -(int)ZKZ_MEMORY_ALLOCATION;
        if (cudaMallocHost((void**)&ws->h_need, (c + 1) * 4) != cudaSuccess) return -(int)ZKZ_MEMORY_ALLOCATION;
        ws->cap_entries = c;
    }
    if (!ws->counters) {
        if (cudaMalloc((void**)&ws->counters, sizeof(ZkCounters) + 16) != cudaSuccess) return -(int)ZKZ_MEMORY_ALLOCATION;
        if (cudaMallocHost((void**)&ws->h_counters, sizeof(ZkCounters) + 16) != cudaSuccess) return -(int)ZKZ_MEMORY_ALLOCATION;
    }
    return 0;
}

// Enqueue one batch on `stream` (scan, entropy, exec[, checksum], status read-back).  No host sync.
int zk_decode_enqueue(ZkDecodeWs* ws, cudaStream_t stream, const uint8_t* d_comp, const uint64_t* c_off, const uint64_t* d_off,
                      uint32_t n, uint8_t* d_dst, int verify_checksum, int exec_warps) {
    ws->pending_n = 0;
    if (n == 0) return 0;
    unsigned long long total_d = d_off[n] - d_off[0];
    // optimistic scratch sizing; the scan kernel reports exact needs and zk_decode_collect retries if exceeded
    size_t need_blocks = (size_t)(total_d / 32768u) + 4 * (size_t)n + 64;      // this codec's own encoder cuts 32 KiB blocks (libzstd: 128 KiB)
    size_t need_lit = (size_t)total_d + 16 * need_blocks;
    size_t need_seq = (size_t)(total_d / 4) + 1024;
    if (need_blocks < ws->want_blocks) need_blocks = ws->want_blocks;
    if (need_lit < ws->want_lit) need_lit = ws->want_lit;
    if (need_seq < ws->want_seq) need_seq = ws->want_seq;
    int sms = ws->sm_count > 0 ? ws->sm_count : 148;
    int rc = zk_decode_ensure(ws, n, need_blocks, need_lit, need_seq);
    if (rc) return rc;
    memcpy(ws->h_off, c_off, (size_t)(n + 1) * 8);
    memcpy(ws->h_off + (n + 1), d_off, (size_t)(n + 1) * 8);
    // Host pipelines hand in dedicated copy streams (ws->up / ws->down): copies of different compute streams otherwise share
    // copy-engine channels, where the upload of one sub-batch queues behind the status read-back of another that is still
    // waiting for its kernels (measured: sub-batch k + 4 started its upload when sub-batch k had finished its download).
    cudaStream_t us = ws->up ? ws->up : stream, ds = ws->down ? ws->down : stream;
    if (us != stream && !ws->ev_up) {
        ZK_CUDA_OK(cudaEventCreateWithFlags(&ws->ev_up, cudaEventDisableTiming)); ZK_CUDA_OK(cudaEventCreateWithFlags(&ws->ev_done, cudaEventDisableTiming));
        ZK_CUDA_OK(cudaEventCreateWithFlags(&ws->ev_down, cudaEventDisableTiming));
    }
    ZK_CUDA_OK(cudaMemcpyAsync(ws->c_off, ws->h_off, (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, us));
    ZK_CUDA_OK(cudaMemcpyAsync(ws->d_off, ws->h_off + (n + 1), (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, us));
    ZK_CUDA_OK(cudaMemsetAsync(ws->counters, 0, sizeof(ZkCounters) + 16, stream));
    ZkDecodeArgs a;
    a.comp = d_comp; a.c_off = (const unsigned long long*)ws->c_off; a.d_off = (const unsigned long long*)ws->d_off; a.dst = d_dst; a.n_entries = n;
    a.blocks = ws->blocks; a.entries = ws->entries; a.counters = ws->counters;
    a.work_counter = (uint32_t*)((uint8_t*)ws->counters + sizeof(ZkCounters));   // two counters (seq, huf), zeroed with the struct
    a.lit = ws->lit; a.seq_lit_end = ws->seq_lit_end; a.seq_out_end = ws->seq_out_end; a.seq_off = ws->seq_off;
    a.huf_list = ws->huf_list; a.seq_list = ws->seq_list;
    a.cap_blocks = ws->cap_blocks; a.cap_lit = ws->cap_lit - 64; a.cap_seq = ws->cap_seq;
    a.trace = nullptr;
    a.d_need = nullptr;
    a.win_max = ws->win_max;
    a.prefix = ws->prefix; a.prefix_len = ws->prefix ? ws->prefix_len : 0; ws->prefix = nullptr; ws->prefix_len = 0;
    if (ws->need) {
        memcpy(ws->h_need, ws->need, (size_t)n * 4);
        ZK_CUDA_OK(cudaMemcpyAsync(ws->d_need, ws->h_need, (size_t)n * 4, cudaMemcpyHostToDevice, us));
        a.d_need = ws->d_need; ws->need = nullptr;
    }
#ifndef ZK_EMUL
    if (getenv("ZK_EXEC_TRACE")) {
        if (!ws->trace) cudaMalloc((void**)&ws->trace, 1024 * 8 * 8);
        cudaMemsetAsync(ws->trace, 0, 1024 * 8 * 8, stream);
        a.trace = ws->trace;
    }
#endif
    if (us != stream) { ZK_CUDA_OK(cudaEventRecord(ws->ev_up, us)); ZK_CUDA_OK(cudaStreamWaitEvent(stream, ws->ev_up, 0)); }   // also orders the caller's upload of the compressed bytes
    ws->prof.begin(0, stream);
    ZK_LAUNCH(zk_scan_kernel, (n + 127) / 128, 128, 0, stream, a);
    ws->prof.end(0, stream);
    // entropy stage: persistent warp-CTAs pulling groups of blocks from a work counter
    size_t est_blocks = (size_t)(total_d / ZK_BLOCK_MAX) + n;
    const size_t seq_smem = ((sizeof(ZkSeqTabs) + 15) & ~(size_t)15) + sizeof(ZkSeqSlot) * ZK_SEQ_LANES, huf_smem = sizeof(ZkHufSlot) * ZK_HUF_SLOTS;
    if (!ws->attr_set) {
        ZK_CUDA_OK(cudaFuncSetAttribute(zk_seq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)seq_smem));
        ZK_CUDA_OK(cudaFuncSetAttribute(zk_huf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)huf_smem + 65536));
        ZK_CUDA_OK(cudaFuncSetAttribute(zk_exec_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024));
        ZK_CUDA_OK(cudaFuncSetAttribute(zk_exec_kernel_w5, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024));
        ZK_CUDA_OK(cudaFuncSetAttribute(zk_exec2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024));
        ws->attr_set = true;
    }
    uint32_t gs = (uint32_t)sms * ws->seq_ctas, gh = (uint32_t)sms * ws->huf_ctas;          // persistent CTAs: as many as fit (shared memory: 4 x 51 KiB, 5 x 41 KiB)
    size_t need_s = est_blocks / ZK_SEQ_LANES + 1, need_h = est_blocks / ZK_HUF_SLOTS + 1;
    if (need_s < gs) gs = (uint32_t)need_s;
    if (need_h < gh) gh = (uint32_t)need_h;
    // the two entropy kernels are independent: run the Huffman one on a side stream
    cudaStream_t hs = stream;
    if (!ws->no_side) {
        if (!ws->side) {
            ZK_CUDA_OK(cudaStreamCreateWithPriority(&ws->side, cudaStreamNonBlocking, ws->prio));
            ZK_CUDA_OK(cudaEventCreateWithFlags(&ws->ev_scan, cudaEventDisableTiming));
            ZK_CUDA_OK(cudaEventCreateWithFlags(&ws->ev_huf, cudaEventDisableTiming));
        }
        hs = ws->side;
        ZK_CUDA_OK(cudaEventRecord(ws->ev_scan, stream));
        ZK_CUDA_OK(cudaStreamWaitEvent(hs, ws->ev_scan, 0));
    }
    ws->prof.begin(2, hs);
    ZK_LAUNCH(zk_huf_kernel, gh, 32, huf_smem + ws->huf_pad, hs, a);
    ws->prof.end(2, hs);
    if (hs != stream) ZK_CUDA_OK(cudaEventRecord(ws->ev_huf, hs));
    ws->prof.begin(1, stream);
    if (ws->seq_v1) ZK_LAUNCH(zk_seq_kernel, gs, 32 * ZK_SEQ_WARPS, seq_smem, stream, a);
    else {
        const size_t seq2_smem = ((sizeof(ZkSeqTabs) + 127) & ~(size_t)127) + sizeof(ZkSeq2Chain) * ZK_S2_NCH;
        if (!ws->attr_set2) { ZK_CUDA_OK(cudaFuncSetAttribute(zk_seq2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)seq2_smem)); ws->attr_set2 = true; }
        uint32_t g2 = (uint32_t)sms * ws->seq2_ctas;
        const size_t need2 = est_blocks / ZK_S2_NCH + 1;
        if (need2 < g2) g2 = (uint32_t)need2;
        ZK_LAUNCH(zk_seq2_kernel, g2, 32, seq2_smem, stream, a);
    }
    ws->prof.end(1, stream);
    if (hs != stream) ZK_CUDA_OK(cudaStreamWaitEvent(stream, ws->ev_huf, 0));
    // exec stage: ring size / warps per entry chosen from how many entries share the machine
    // Each entry is one serial dependency chain, so throughput comes from entries in flight: pick warps per
    // CTA and ring size such that (if possible) every entry of the batch is resident at once.
    // (`share` > 1: that many sub-batches of a host pipeline run concurrently on different streams)
    int per_sm = (int)(((unsigned long long)n * (unsigned)(ws->share > 0 ? ws->share : 1) + (uint32_t)sms - 1) / (uint32_t)sms);
    if (per_sm < 1) per_sm = 1;
    int W = exec_warps;
    ws->prof.begin(3, stream);
    if (ws->exec_v2 || a.prefix_len) {           // (prefix mode exists in the in-order kernel only)
        // second-generation kernel: <= 64 registers, so 32 warps per SM whatever the split; ring = what is left of the
        // SM's shared memory per resident entry
        if (per_sm > 8) per_sm = 8;
        if (W <= 0) W = 16 / per_sm;        // measured (profiles/README.md): more warps per frame than this make the in-order chain SLOWER
        if (W > 32) W = 32;
        if (W < 2) W = 2;
        uint32_t ring = 128 * 1024;
        while (ring > 8 * 1024 && ((size_t)ring + 2048) * (size_t)per_sm > 220 * 1024) ring >>= 1;
        if (ws->ring_override) ring = ws->ring_override;
        ZK_LAUNCH(zk_exec2_kernel, n, W * 32, ring, stream, a, ring);
    } else {
        // 126 registers/thread -> 16 warps per SM; from four entries per SM on, the 96-register build of the same body
        // (20 warps per SM, <= 5 per entry) keeps every entry of the batch resident with one more warp each
        bool small_regs = false;
        if (W <= 0) {
            if (per_sm >= 4) { W = 20 / per_sm; if (W < 2) W = 2; small_regs = true; }
            else W = 16 / per_sm;
        } else small_regs = W <= 5 && per_sm >= 4;
        if (W > 16) W = 16;
        uint32_t ring = 128 * 1024;
        while (ring > 8 * 1024 && (size_t)ring * (size_t)per_sm > 200 * 1024) ring >>= 1;
        if (ws->ring_override) ring = ws->ring_override;
        if (small_regs) ZK_LAUNCH(zk_exec_kernel_w5, n, W * 32, ring, stream, a, ring);
        else ZK_LAUNCH(zk_exec_kernel, n, W * 32, ring, stream, a, ring);
    }
    ws->prof.end(3, stream);
    if (verify_checksum) { ws->prof.begin(4, stream); ZK_LAUNCH(zk_xxh64_kernel, (n + 3) / 4, 128, 0, stream, a); ws->prof.end(4, stream); }
    if (ds != stream) { ZK_CUDA_OK(cudaEventRecord(ws->ev_done, stream)); ZK_CUDA_OK(cudaStreamWaitEvent(ds, ws->ev_done, 0)); }
    ZK_CUDA_OK(cudaMemcpyAsync(ws->h_entries, ws->entries, (size_t)n * sizeof(ZkEntry), cudaMemcpyDeviceToHost, ds));
    ZK_CUDA_OK(cudaMemcpyAsync(ws->h_counters, ws->counters, sizeof(ZkCounters), cudaMemcpyDeviceToHost, ds));
    ws->launches += 4 + (verify_checksum ? 1 : 0);
    ws->pending_n = n;
    return 0;
}

// Wait for the batch enqueued last on `stream`; returns 0, the first failing entry status, or ZK_ST_RETRY when the
// scratch was too small (ws->want_* then hold the exact needs: the caller re-enqueues the same batch).
int zk_decode_collect(ZkDecodeWs* ws, cudaStream_t stream, int32_t* status_out) {
    uint32_t n = ws->pending_n;
    if (n == 0) return 0;
    if (ws->down && ws->ev_down) ZK_CUDA_OK(cudaEventSynchronize(ws->ev_down));     // recorded by the caller after the output copy on the download stream
    else ZK_CUDA_OK(cudaStreamSynchronize(stream));
#ifndef ZK_EMUL
    { cudaError_t le__ = cudaGetLastError(); if (le__ != cudaSuccess) { zk_note_cuda_error("kernel launch / execution", (int)le__); return ZK_INT_CUDA; } }
#endif
    ws->pending_n = 0;
#ifndef ZK_EMUL
    if (ws->trace && getenv("ZK_EXEC_TRACE")) {
        static unsigned long long host[1024 * 8];
        cudaMemcpy(host, ws->trace, sizeof host, cudaMemcpyDeviceToHost);
        FILE* f = fopen(getenv("ZK_EXEC_TRACE"), "wb"); if (f) { fwrite(host, 1, sizeof host, f); fclose(f); }
    }
#endif
    ws->prof.harvest();
    if (ws->h_counters->overflow) {
        ws->want_blocks = (size_t)ws->h_counters->n_blocks; ws->want_lit = (size_t)ws->h_counters->n_lit; ws->want_seq = (size_t)ws->h_counters->n_seq;
        return ZK_ST_RETRY;
    }
    int worst = 0;
    for (uint32_t i = 0; i < n; i++) {
        int32_t st = ws->h_entries[i].status;
        if (st == ZK_ST_RETRY) st = -(int)ZKZ_MEMORY_ALLOCATION;
        if (status_out) status_out[i] = st;
        if (st && !worst) worst = st;
    }
    return worst;
}

int zk_decode_batch(ZkDecodeWs* ws, cudaStream_t stream, const uint8_t* d_comp, const uint64_t* c_off, const uint64_t* d_off,
                    uint32_t n, uint8_t* d_dst, int verify_checksum, int32_t* status_out, int exec_warps) {
    for (int attempt = 0; attempt < 2; attempt++) {
        int rc = zk_decode_enqueue(ws, stream, d_comp, c_off, d_off, n, d_dst, verify_checksum, exec_warps);
        if (rc) return rc;
        rc = zk_decode_collect(ws, stream, status_out);
        if (rc != ZK_ST_RETRY) return rc;
    }
    fprintf(stderr, "zeekstd_b200: decode scratch still too small after growing to the exact needs (blocks %zu lit %zu seq %zu; caps %zu %zu %zu)\n",
            ws->want_blocks, ws->want_lit, ws->want_seq, ws->cap_blocks, ws->cap_lit, ws->cap_seq);
    return -(int)ZKZ_MEMORY_ALLOCATION;
}
