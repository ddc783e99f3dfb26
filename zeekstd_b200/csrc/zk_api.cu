// zk_api.cu -- the batch half of the C ABI (include/zeekstd_b200.h): context + zk_{de,}compress_frames[_dev].
// The API-mirror half (SeekTable / RawEncoder / Encoder / Decoder) lives in zk_host.cpp and is built on
// top of these entry points only.
#include "zk_ctx.h"
#include "../../include/zeekstd_b200.h"
#include <stdio.h>
#include <time.h>
#include <stdlib.h>
#include <vector>

static thread_local char zk_tls_cuda_msg[256] = "";
void zk_note_cuda_error(const char* what, int code) {
    snprintf(zk_tls_cuda_msg, sizeof zk_tls_cuda_msg, "%s: %s", what, cudaGetErrorString((cudaError_t)code));
}
extern "C" const char* zk_last_cuda_error(void) { return zk_tls_cuda_msg; }
#ifndef ZK_EMUL
#define ZK_RT_OK(x) do { cudaError_t e__ = (x); if (e__ != cudaSuccess) { zk_note_cuda_error(#x, (int)e__); (void)cudaGetLastError(); return ZK_ERR_CUDA; } } while (0)
#else
#define ZK_RT_OK(x) do { (void)(x); } while (0)
#endif

static int zk_host_slots(bool enc);
static size_t zk_env_size(const char* name, size_t dflt) {
    const char* s = getenv(name);
    if (!s || !*s) return dflt;
    return (size_t)strtoull(s, nullptr, 10);
}

// sub-batches in flight of the host-pointer pipelines (measured on B200, tools/e2e_sweep4.sh): decompress wants many
// (its exec stage is latency-bound per frame), compress few (its kernels fill the machine from one 128 MiB sub-batch)
static int zk_host_slots(bool enc) {
    size_t v = zk_env_size(enc ? "ZK_HOST_SLOTS_ENC" : "ZK_HOST_SLOTS", enc ? 4 : 8);
    return (int)(v < 1 ? 1 : (v > ZK_SLOTS ? ZK_SLOTS : v));
}

extern "C" const char* zk_version(void) {
#ifdef ZK_EMUL
    return "zeekstd_b200 0.1 (ZK_EMUL test build: device code interpreted on the CPU; not a product build)";
#else
    return "zeekstd_b200 0.1 (sm_100a)";
#endif
}

extern "C" const char* zk_error_name(int32_t rc) {
    switch (rc) {
    case 0: return "No error detected";
    case ZK_ERR_NUMBER_CONVERSION: return "number conversion failed";
    case ZK_ERR_OFFSET_OUT_OF_RANGE: return "offset out of range";
    case ZK_ERR_FRAME_INDEX_TOO_LARGE: return "frame index too large";
    case ZK_ERR_IO: return "io error";
    case ZK_ERR_NO_DEVICE: return "no usable CUDA device (zeekstd_b200 has no CPU fallback)";
    case ZK_ERR_INVALID_ARG: return "invalid argument";
    case ZK_ERR_CUDA: return "CUDA runtime or kernel failure (see zk_last_cuda_error)";
    // strings of ZSTD_getErrorName for the codes this codec can raise
    case -1: return "Error (generic)";
    case -10: return "Unknown frame descriptor";
    case -12: return "Version not supported";
    case -14: return "Unsupported frame parameter";
    case -16: return "Frame requires too much memory for decoding";
    case -20: return "Data corruption detected";
    case -22: return "Restored data doesn't match checksum";
    case -30: return "Dictionary is corrupted";
    case -32: return "Dictionary mismatch";
    case -40: return "Unsupported parameter";
    case -42: return "Parameter is out of bound";
    case -64: return "Allocation error : not enough memory";
    case -70: return "Destination buffer is too small";
    case -72: return "Src size is incorrect";
    default: return "Unspecified error code";
    }
}

int zk_slot_ensure(ZkSlot* s, size_t need_in, size_t need_out) {
    if (s->cap_in < need_in) {
        if (s->d_in) cudaFree(s->d_in);
        s->d_in = nullptr; s->cap_in = 0;
        size_t want = need_in + need_in / 8 + 256;
        if (cudaMalloc((void**)&s->d_in, want) != cudaSuccess) return ZK_ERR_ZSTD(ZKZ_MEMORY_ALLOCATION);
        s->cap_in = want;
    }
    if (s->cap_out < need_out) {
        if (s->d_out) cudaFree(s->d_out);
        s->d_out = nullptr; s->cap_out = 0;
        size_t want = need_out + need_out / 8 + 256;
        if (cudaMalloc((void**)&s->d_out, want) != cudaSuccess) return ZK_ERR_ZSTD(ZKZ_MEMORY_ALLOCATION);
        s->cap_out = want;
    }
    return 0;
}

extern "C" int32_t zk_ctx_create(int32_t device_ordinal, uint32_t flags, zk_ctx** out) {
    (void)flags;
    if (!out) return ZK_ERR_INVALID_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { (void)cudaGetLastError(); return ZK_ERR_NO_DEVICE; }
    if (device_ordinal < 0 || device_ordinal >= ndev) return ZK_ERR_INVALID_ARG;
    ZK_RT_OK(cudaSetDevice(device_ordinal));
    cudaDeviceProp prop;
    ZK_RT_OK(cudaGetDeviceProperties(&prop, device_ordinal));
    zk_ctx* c = new zk_ctx();
    c->device = device_ordinal;
    c->sm_count = prop.multiProcessorCount > 0 ? prop.multiProcessorCount : 148;
    // ZK_HOST_PRIO (default 1): slot i runs at stream priority (greatest + i): concurrent sub-batches of the host pipelines then
    // complete staggered (oldest slot first) instead of all at once, which keeps the D2H engine busy from early on
    int least = 0, greatest = 0;
    const bool use_prio = zk_env_size("ZK_HOST_PRIO", 1) != 0;
    if (use_prio) cudaDeviceGetStreamPriorityRange(&least, &greatest);
    for (int i = 0; i < ZK_SLOTS; i++) {
        const int prio = use_prio ? (greatest + i < least ? greatest + i : least) : 0;
        if (cudaStreamCreateWithPriority(&c->slot[i].stream, cudaStreamNonBlocking, prio) != cudaSuccess) { delete c; return ZK_ERR_NO_DEVICE; }
        c->slot[i].dws.prio = c->slot[i].ews.prio = prio;
        c->slot[i].dws.sm_count = c->sm_count;
        c->slot[i].dws.ring_override = (uint32_t)zk_env_size("ZK_RING_BYTES", 0);   // tuning / tests: power of two >= 1024
        c->slot[i].dws.huf_pad = (uint32_t)zk_env_size("ZK_HUF_PAD", 0);
        c->slot[i].dws.exec_v2 = zk_env_size("ZK_EXEC_V2", 0) != 0;
        c->slot[i].dws.seq_v1 = zk_env_size("ZK_SEQ_V1", 0) != 0; c->slot[i].dws.seq2_ctas = (uint32_t)zk_env_size("ZK_SEQ2_CTAS", 6);
        c->slot[i].dws.seq_ctas = (uint32_t)zk_env_size("ZK_SEQ_CTAS", 4); c->slot[i].dws.huf_ctas = (uint32_t)zk_env_size("ZK_HUF_CTAS", 8);
        c->slot[i].ews.sm_count = c->sm_count;
    }
    cudaEventCreate(&c->ev0); cudaEventCreate(&c->ev1);
    if (zk_env_size("ZK_HOST_COPY_STREAMS", 1) != 0) {
        cudaStreamCreateWithFlags(&c->up, cudaStreamNonBlocking); cudaStreamCreateWithFlags(&c->down, cudaStreamNonBlocking);
    }
    *out = c;
    return 0;
}

extern "C" void zk_ctx_destroy(zk_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    for (int i = 0; i < ZK_SLOTS; i++) {
        ZkSlot& s = c->slot[i];
        if (s.stream) cudaStreamSynchronize(s.stream);
        zk_decode_ws_free(&s.dws);
        zk_encode_ws_free(&s.ews);
        if (s.d_in) cudaFree(s.d_in);
        if (s.d_out) cudaFree(s.d_out);
        if (s.stream) cudaStreamDestroy(s.stream);
    }
    if (c->up) cudaStreamDestroy(c->up);
    if (c->down) cudaStreamDestroy(c->down);
    if (c->d_prefix) cudaFree(c->d_prefix);
    if (c->d_ldm) cudaFree(c->d_ldm);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    delete c;
}

// context parameters (include/zeekstd_b200.h): sticky, 0 = default
extern "C" int32_t zk_ctx_set_cparameter(zk_ctx* c, int32_t param, int32_t value) {
    if (!c) return ZK_ERR_INVALID_ARG;
    switch (param) {
    case ZK_C_WINDOW_LOG:
        if (value != 0 && (value < ZK_WINDOWLOG_MIN || value > ZK_WINDOWLOG_MAX)) return ZK_ERR_ZSTD(ZKZ_PARAM_OUT_OF_BOUND);
        c->c_window_log = value; return 0;
    case ZK_C_ENABLE_LONG_DISTANCE_MATCHING:
        if (value != 0 && value != 1) return ZK_ERR_ZSTD(ZKZ_PARAM_OUT_OF_BOUND);
        c->c_ldm = value; return 0;
    default: return ZK_ERR_ZSTD(ZKZ_PARAM_UNSUPPORTED);
    }
}

extern "C" int32_t zk_ctx_set_dparameter(zk_ctx* c, int32_t param, int32_t value) {
    if (!c) return ZK_ERR_INVALID_ARG;
    if (param != ZK_D_WINDOW_LOG_MAX) return ZK_ERR_ZSTD(ZKZ_PARAM_UNSUPPORTED);
    if (value != 0 && (value < ZK_WINDOWLOG_MIN || value > ZK_WINDOWLOG_MAX)) return ZK_ERR_ZSTD(ZKZ_PARAM_OUT_OF_BOUND);
    c->d_window_log_max = value;
    for (int i = 0; i < ZK_SLOTS; i++) c->slot[i].dws.win_max = value ? 1ull << value : (1ull << 27) + 1;
    return 0;
}

extern "C" uint64_t zk_ctx_kernel_launches(const zk_ctx* c) { return c ? c->launches() : 0; }
extern "C" float zk_ctx_last_device_ms(const zk_ctx* c) { return c ? c->last_ms : 0.f; }
extern "C" size_t zk_compress_bound(size_t n, uint32_t frame_size) { return zk_encode_bound(n, frame_size); }

extern "C" void zk_ctx_profile(zk_ctx* c, int32_t enable) {
    if (!c) return;
    for (int i = 0; i < ZK_SLOTS; i++) {
        c->slot[i].dws.prof.enabled = enable != 0; c->slot[i].ews.prof.enabled = enable != 0;
        for (int k = 0; k < ZK_PROF_SLOTS; k++) { c->slot[i].dws.prof.ms[k] = c->slot[i].ews.prof.ms[k] = 0.f; c->slot[i].dws.prof.count[k] = c->slot[i].ews.prof.count[k] = 0; }
    }
}
extern "C" void zk_ctx_profile_read(const zk_ctx* c, float* ms, uint32_t* launches) {
    for (int k = 0; k < ZK_PROF_SLOTS; k++) {
        float t = 0.f; uint32_t n = 0;
        for (int i = 0; c && i < ZK_SLOTS; i++) { t += c->slot[i].dws.prof.ms[k] + c->slot[i].ews.prof.ms[k]; n += c->slot[i].dws.prof.count[k] + c->slot[i].ews.prof.count[k]; }
        if (ms) ms[k] = t;
        if (launches) launches[k] = n;
    }
}

// ---------------------------------------------------------------------------------------------
// decompress
// ---------------------------------------------------------------------------------------------
// split [0,n) into sub-batches bounded by output bytes so scratch stays proportional to the sub-batch
static uint32_t zk_next_sub(const uint64_t* d_off, uint32_t first, uint32_t n, size_t max_bytes, uint32_t max_entries) {
    uint32_t e = first + 1;
    while (e < n && e - first < max_entries && d_off[e + 1] - d_off[first] <= max_bytes) e++;
    return e;
}

extern "C" int32_t zk_decompress_frames_dev(zk_ctx* c, const void* d_comp, const uint64_t* c_off, const uint64_t* d_off,
                                            uint32_t n, void* d_dst, int32_t verify, int32_t* status, void* cuda_stream) {
    if (!c || (n && (!d_comp || !c_off || !d_off || !d_dst))) return ZK_ERR_INVALID_ARG;
    if (n == 0) return 0;
    ZK_RT_OK(cudaSetDevice(c->device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : c->slot[0].stream;
    const size_t sub_bytes = zk_env_size("ZK_DEV_SUB_BYTES", (size_t)1 << 30);
    ZkDecodeWs* ws = &c->slot[0].dws;
    ws->share = 1; ws->no_side = zk_env_size("ZK_DEV_SIDE", 1) == 0;
    ws->up = ws->down = nullptr;                           // device-resident data: nothing to copy but offsets and statuses
    cudaEventRecord(c->ev0, st);
    int32_t worst = 0;
    for (uint32_t first = 0; first < n;) {
        uint32_t end = zk_next_sub(d_off, first, n, sub_bytes, 1u << 20);
        int rc = zk_decode_batch(ws, st, (const uint8_t*)d_comp, c_off + first, d_off + first, end - first, (uint8_t*)d_dst,
                                 verify, status ? status + first : nullptr, (int)zk_env_size("ZK_EXEC_WARPS", 0));
        if (rc && !worst) worst = rc;
        if (rc == ZK_INT_CUDA || rc == -(int)ZKZ_MEMORY_ALLOCATION) return rc;
        first = end;
    }
    cudaEventRecord(c->ev1, st);
    cudaEventSynchronize(c->ev1);
    cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1);
    return worst;
}

// ZK_E2E_TRACE=1: per-sub-batch timeline of the host-pointer paths (CUDA events on the slot streams), printed to stderr.
struct ZkTrace {
    bool on = false; cudaEvent_t t0 = nullptr; std::vector<cudaEvent_t> ev; std::vector<int> tag; std::vector<double> host; double h0 = 0;
    static double now() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; }
    void begin(cudaStream_t st) {
        on = getenv("ZK_E2E_TRACE") != nullptr; if (!on) return;
        cudaEventCreate(&t0); cudaEventRecord(t0, st); h0 = now();
    }
    void mark(cudaStream_t st, int sub, int what) {
        if (!on) return;
        cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, st); ev.push_back(e); tag.push_back(sub * 8 + what); host.push_back(now() - h0);
    }
    void end(const char* name) {
        if (!on) return;
        cudaDeviceSynchronize();
        static const char* W[] = {"h2d0", "h2d1", "kern1", "d2h0", "d2h1"};
        for (size_t i = 0; i < ev.size(); i++) {
            float ms = 0; cudaEventElapsedTime(&ms, t0, ev[i]);
            fprintf(stderr, "%s sub %d %s gpu %.3f host %.3f\n", name, tag[i] >> 3, W[tag[i] & 7], ms, host[i]);
            cudaEventDestroy(ev[i]);
        }
        cudaEventDestroy(t0);
    }
};

struct ZkSubDec { uint32_t first = 0, count = 0; std::vector<uint64_t> c_rel, d_rel; bool busy = false; };

static int zk_dec_sub_enqueue(zk_ctx* c, int si, ZkSubDec& sb, const uint8_t* comp, const uint64_t* c_off, const uint64_t* d_off,
                              uint8_t* dst, int verify, ZkTrace* tr = nullptr, int k = 0, const uint32_t* need = nullptr) {
    ZkSlot& s = c->slot[si];
    uint32_t f = sb.first, cnt = sb.count;
    size_t cbytes = (size_t)(c_off[f + cnt] - c_off[f]), obytes = (size_t)(d_off[f + cnt] - d_off[f]);
    int rc = zk_slot_ensure(&s, cbytes + 32, obytes + 32);
    if (rc) return rc;
    sb.c_rel.resize(cnt + 1); sb.d_rel.resize(cnt + 1);
    for (uint32_t j = 0; j <= cnt; j++) { sb.c_rel[j] = c_off[f + j] - c_off[f]; sb.d_rel[j] = d_off[f + j] - d_off[f]; }
    cudaStream_t us = c->up ? c->up : s.stream, ds = c->down ? c->down : s.stream;
    s.dws.up = c->up; s.dws.down = c->down;
    if (tr) tr->mark(us, k, 0);
    ZK_RT_OK(cudaMemcpyAsync(s.d_in, comp + c_off[f], cbytes, cudaMemcpyHostToDevice, us));
    if (tr) tr->mark(us, k, 1);
    s.dws.no_side = zk_env_size("ZK_HOST_SIDE", 1) == 0;
    s.dws.share = (int)zk_env_size("ZK_HOST_SHARE", 3);
    s.dws.need = need ? need + f : nullptr;
    s.dws.prefix = c->cur_prefix_len ? c->d_prefix : nullptr; s.dws.prefix_len = c->cur_prefix_len;
    rc = zk_decode_enqueue(&s.dws, s.stream, s.d_in, sb.c_rel.data(), sb.d_rel.data(), cnt, s.d_out, verify,
                           (int)zk_env_size("ZK_EXEC_WARPS", 0));
    if (rc) return rc;
    if (tr) tr->mark(s.stream, k, 2);
    if (obytes) ZK_RT_OK(cudaMemcpyAsync(dst + d_off[f], s.d_out, obytes, cudaMemcpyDeviceToHost, ds));
    if (ds != s.stream) ZK_RT_OK(cudaEventRecord(s.dws.ev_down, ds));        // what zk_decode_collect waits for
    if (tr) tr->mark(ds, k, 4);
    sb.busy = true;
    return 0;
}

static int zk_dec_sub_finish(zk_ctx* c, int si, ZkSubDec& sb, const uint8_t* comp, const uint64_t* c_off, const uint64_t* d_off,
                             uint8_t* dst, int verify, int32_t* status, const uint32_t* need = nullptr) {
    ZkSlot& s = c->slot[si];
    if (!sb.busy) return 0;
    int rc = zk_decode_collect(&s.dws, s.stream, status ? status + sb.first : nullptr);
    if (rc == ZK_ST_RETRY) {            // scratch was too small for this sub-batch: exact needs are known now
        rc = zk_dec_sub_enqueue(c, si, sb, comp, c_off, d_off, dst, verify, nullptr, 0, need);
        if (rc) { sb.busy = false; return rc; }
        rc = zk_decode_collect(&s.dws, s.stream, status ? status + sb.first : nullptr);
        if (rc == ZK_ST_RETRY) rc = ZK_ERR_ZSTD(ZKZ_MEMORY_ALLOCATION);
    }
    sb.busy = false;
    return rc;
}

extern "C" int32_t zk_decompress_frames(zk_ctx* c, const uint8_t* comp, const uint64_t* c_off, const uint64_t* d_off,
                                        uint32_t n, uint8_t* dst, int32_t verify, int32_t* status) {
    return zk_decompress_frames_upto(c, comp, c_off, d_off, n, dst, nullptr, verify, status);
}

extern "C" int32_t zk_decompress_frames_upto(zk_ctx* c, const uint8_t* comp, const uint64_t* c_off, const uint64_t* d_off,
                                             uint32_t n, uint8_t* dst, const uint32_t* d_need, int32_t verify, int32_t* status) {
    if (!c || (n && (!comp || !c_off || !d_off || !dst))) return ZK_ERR_INVALID_ARG;
    if (n == 0) return 0;
    ZK_RT_OK(cudaSetDevice(c->device));
    const size_t sub_bytes = zk_env_size("ZK_HOST_SUB_BYTES", (size_t)128 << 20);     // measured best on B200 (tools/e2e_sweep2.sh)
    ZkSubDec sub[ZK_SLOTS];
    const int NS = zk_host_slots(false);
    const uint32_t ramp = (uint32_t)zk_env_size("ZK_HOST_RAMP", 0);            // the first `ramp` sub-batches are 1/2^ramp ... 1/2 of the full size
    int32_t worst = 0;
    uint32_t k = 0;
    ZkTrace tr; tr.begin(c->slot[0].stream);
    for (uint32_t first = 0; first < n; k++) {
        int si = (int)(k % NS);
        int rc = zk_dec_sub_finish(c, si, sub[si], comp, c_off, d_off, dst, verify, status, d_need);
        if (rc && !worst) worst = rc;
        // ZK_HOST_RAMP=r (default 0): the first r sub-batches are 1/2^r ... 1/2 of the full size, so that the output copy could start
        // earlier.  Measured on B200 (profiles/README.md): no gain -- a sub-batch of any size spends about one frame latency in
        // K-D2, so a small first sub-batch is not done much sooner than a full one
        const size_t this_sub = k < ramp ? sub_bytes >> (ramp - k) : sub_bytes;
        uint32_t end = zk_next_sub(d_off, first, n, this_sub, 1u << 20);
        sub[si].first = first; sub[si].count = end - first;
        rc = zk_dec_sub_enqueue(c, si, sub[si], comp, c_off, d_off, dst, verify, &tr, (int)k, d_need);
        if (rc) { if (!worst) worst = rc; break; }
        first = end;
    }
    for (int si = 0; si < ZK_SLOTS; si++) {
        int rc = zk_dec_sub_finish(c, si, sub[si], comp, c_off, d_off, dst, verify, status, d_need);
        if (rc && !worst) worst = rc;
    }
    tr.end("dec");
    return worst;
}

// ---------------------------------------------------------------------------------------------
// compress
// ---------------------------------------------------------------------------------------------
static uint32_t zk_frames_of(size_t n, uint32_t frame_size) {
    if (n == 0) return 1;                                   // Encoder::finish() always closes one frame (encode.rs:755-756)
    return (uint32_t)((n + frame_size - 1) / frame_size);
}

extern "C" int32_t zk_compress_frames_dev(zk_ctx* c, const void* d_src, size_t n, uint32_t frame_size, int32_t level, int32_t checksum,
                                          void* d_dst, size_t dst_cap, uint32_t* c_sizes, uint32_t* d_sizes, uint32_t frames_cap,
                                          uint32_t* n_frames, size_t* dst_len, void* cuda_stream) {
    if (!c || !d_dst || (n && !d_src) || frame_size == 0) return ZK_ERR_INVALID_ARG;
    if (frame_size > ZK_SEEKABLE_MAX_FRAME_SIZE) frame_size = ZK_SEEKABLE_MAX_FRAME_SIZE;       // encode.rs:531-534
    if ((n + frame_size - 1) / frame_size > ZK_SEEKABLE_MAX_FRAMES) return ZK_ERR_FRAME_INDEX_TOO_LARGE;
    const uint32_t nf = zk_frames_of(n, frame_size);
    if (nf > frames_cap) return ZK_ERR_ZSTD(ZKZ_DST_TOO_SMALL);
    ZK_RT_OK(cudaSetDevice(c->device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : c->slot[0].stream;
    // sub-batches bound the scratch (about 4x the sub-batch input)
    const size_t sub_bytes = zk_env_size("ZK_DEV_SUB_BYTES", (size_t)1 << 30);
    uint32_t per = (uint32_t)(sub_bytes / frame_size); if (per == 0) per = 1;
    cudaEventRecord(c->ev0, st);
    size_t out_pos = 0;
    for (uint32_t f0 = 0; f0 < nf; f0 += per) {
        const uint32_t cnt = nf - f0 < per ? nf - f0 : per;
        const size_t in_off = (size_t)f0 * frame_size;
        const size_t in_len = n - in_off < (size_t)cnt * frame_size ? n - in_off : (size_t)cnt * frame_size;
        size_t produced = 0;
        c->slot[0].ews.no_side = false;
        c->slot[0].ews.win_log = (uint32_t)c->c_window_log;
        int rc = zk_encode_batch(&c->slot[0].ews, st, (const uint8_t*)d_src + in_off, in_len, frame_size, level, checksum,
                                 (uint8_t*)d_dst + out_pos, dst_cap - out_pos, c_sizes ? c_sizes + f0 : nullptr, cnt, &produced);
        if (rc) return rc;
        out_pos += produced;
    }
    cudaEventRecord(c->ev1, st);
    cudaEventSynchronize(c->ev1);
    cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1);
    if (d_sizes) for (uint32_t f = 0; f < nf; f++) {
        size_t lo = (size_t)f * frame_size; d_sizes[f] = (uint32_t)(n - lo < frame_size ? n - lo : frame_size);
    }
    if (n_frames) *n_frames = nf;
    if (dst_len) *dst_len = out_pos;
    return 0;
}

struct ZkSubEnc { uint32_t f0 = 0, cnt = 0; size_t in_off = 0, in_len = 0, out_pos = 0; bool busy = false; };

extern "C" int32_t zk_compress_frames(zk_ctx* c, const uint8_t* src, size_t n, uint32_t frame_size, int32_t level, int32_t checksum,
                                      uint8_t* dst, size_t dst_cap, uint32_t* c_sizes, uint32_t* d_sizes, uint32_t frames_cap,
                                      uint32_t* n_frames, size_t* dst_len) {
    if (!c || !dst || (n && !src) || frame_size == 0) return ZK_ERR_INVALID_ARG;
    if (frame_size > ZK_SEEKABLE_MAX_FRAME_SIZE) frame_size = ZK_SEEKABLE_MAX_FRAME_SIZE;
    if ((n + frame_size - 1) / frame_size > ZK_SEEKABLE_MAX_FRAMES) return ZK_ERR_FRAME_INDEX_TOO_LARGE;
    const uint32_t nf = zk_frames_of(n, frame_size);
    if (nf > frames_cap) return ZK_ERR_ZSTD(ZKZ_DST_TOO_SMALL);
    ZK_RT_OK(cudaSetDevice(c->device));
    const size_t sub_bytes = zk_env_size("ZK_HOST_SUB_BYTES_ENC", (size_t)96 << 20);    // measured best on B200 (tools/knobs_round.sh)
    uint32_t per = (uint32_t)(sub_bytes / frame_size); if (per == 0) per = 1;
    // The compressed size of a sub-batch is only known when it completes, so output positions are assigned in
    // order at completion time: H2D and kernels of later sub-batches overlap the D2H of earlier ones.
    ZkSubEnc sub[ZK_SLOTS];
    size_t out_pos = 0; int32_t err = 0;
    std::vector<uint32_t> tmp_sizes(per);
    ZkTrace tr; tr.begin(c->slot[0].stream);
    int sub_k[ZK_SLOTS] = {0};
    auto finish = [&](int si) -> int {
        ZkSubEnc& sb = sub[si]; ZkSlot& s = c->slot[si];
        if (!sb.busy) return 0;
        sb.busy = false;
        size_t produced = 0;
        int rc = zk_encode_collect(&s.ews, s.stream, c_sizes ? c_sizes + sb.f0 : tmp_sizes.data(), &produced);
        if (rc) return rc;
        if (out_pos + produced > dst_cap) return ZK_ERR_ZSTD(ZKZ_DST_TOO_SMALL);
        tr.mark(s.stream, sub_k[si], 3);
        if (cudaMemcpyAsync(dst + out_pos, s.d_out, produced, cudaMemcpyDeviceToHost, s.stream) != cudaSuccess) return ZK_ERR_CUDA;
        tr.mark(s.stream, sub_k[si], 4);
        out_pos += produced;
        return 0;
    };
    uint32_t k = 0;
    const int NS = zk_host_slots(true);
    int order[ZK_SLOTS]; int n_inflight = 0;              // completion must follow submission order
    for (uint32_t f0 = 0; f0 < nf && !err; f0 += per, k++) {
        const int si = (int)(k % NS);
        if (n_inflight == NS) {                             // oldest in flight is exactly slot si
            err = finish(si); n_inflight--;
            if (err) break;
        }
        ZkSlot& s = c->slot[si]; ZkSubEnc& sb = sub[si];
        if (cudaStreamSynchronize(s.stream) != cudaSuccess) { err = ZK_ERR_CUDA; break; }   // its previous D2H must be done before d_out is reused
        sb.f0 = f0; sb.cnt = nf - f0 < per ? nf - f0 : per;
        sb.in_off = (size_t)f0 * frame_size;
        sb.in_len = n - sb.in_off < (size_t)sb.cnt * frame_size ? n - sb.in_off : (size_t)sb.cnt * frame_size;
        const size_t bound = zk_encode_bound(sb.in_len, frame_size);
        int rc = zk_slot_ensure(&s, sb.in_len + 32, bound + 32);
        if (rc) { err = rc; break; }
        sub_k[si] = (int)k; tr.mark(s.stream, (int)k, 0);
        if (sb.in_len && cudaMemcpyAsync(s.d_in, src + sb.in_off, sb.in_len, cudaMemcpyHostToDevice, s.stream) != cudaSuccess) { err = ZK_ERR_CUDA; break; }
        tr.mark(s.stream, (int)k, 1);
        s.ews.no_side = zk_env_size("ZK_HOST_SIDE", 1) == 0;
        s.ews.prefix = c->cur_prefix_len ? c->d_prefix : nullptr; s.ews.prefix_len = c->cur_prefix_len;
        s.ews.ldm_tab = c->cur_prefix_len && c->cur_ldm_log ? c->d_ldm : nullptr; s.ews.ldm_log = c->cur_ldm_log;
        s.ews.win_log = c->cur_ldm_win ? c->cur_ldm_win : (uint32_t)c->c_window_log;
        rc = zk_encode_enqueue(&s.ews, s.stream, s.d_in, sb.in_len, frame_size, level, checksum, s.d_out, bound, sb.cnt);
        if (rc) { err = rc; break; }
        tr.mark(s.stream, (int)k, 2);
        sb.busy = true; order[n_inflight++ % ZK_SLOTS] = si;
    }
    // drain in submission order
    for (uint32_t j = 0; j < (uint32_t)NS && !err; j++) {
        const int si = (int)((k + j) % NS);                // oldest first
        int rc = finish(si);
        if (rc) err = rc;
    }
    for (int si = 0; si < ZK_SLOTS; si++) cudaStreamSynchronize(c->slot[si].stream);
    tr.end("enc");
    (void)order;
    if (err) return err;
    if (d_sizes) for (uint32_t f = 0; f < nf; f++) {
        size_t lo = (size_t)f * frame_size; d_sizes[f] = (uint32_t)(n - lo < frame_size ? n - lo : frame_size);
    }
    if (n_frames) *n_frames = nf;
    if (dst_len) *dst_len = out_pos;
    return 0;
}

// ---------------------------------------------------------------------------------------------
// prefix / patch mode (SURVEY.md 8f.3): every frame is coded against the same raw-content prefix
//   RawEncoder::compress_with_prefix   encode.rs:311-338  (cctx.ref_prefix at the start of every frame)
//   Decoder::decompress_with_prefix    decode.rs:201-214, 246-255  (dctx.ref_prefix before the first frame and after every frame end)
// The prefix is uploaded once per call and stays resident; K-C1 searches its tail from the first block of every frame, K-D2
// resolves offsets that reach before a frame's first byte into it.
// ---------------------------------------------------------------------------------------------
static int32_t zk_ctx_set_prefix(zk_ctx* c, const uint8_t* prefix, size_t len) {
    c->cur_prefix_len = 0;
    if (!prefix || len == 0) return 0;
    if (len > 0x7FFFFFFFull) return ZK_ERR_INVALID_ARG;
    ZK_RT_OK(cudaSetDevice(c->device));
    if (c->cap_prefix < len + 64) {
        if (c->d_prefix) cudaFree(c->d_prefix);
        c->d_prefix = nullptr; c->cap_prefix = 0;
        if (cudaMalloc((void**)&c->d_prefix, len + len / 8 + 256) != cudaSuccess) return ZK_ERR_ZSTD(ZKZ_MEMORY_ALLOCATION);
        c->cap_prefix = len + len / 8 + 256;
    }
    for (int i = 0; i < ZK_SLOTS; i++) if (c->slot[i].stream) cudaStreamSynchronize(c->slot[i].stream);    // nobody reads the old prefix any more
    ZK_RT_OK(cudaMemcpy(c->d_prefix, prefix, len, cudaMemcpyHostToDevice));
    c->cur_prefix_len = (uint32_t)len;
    return 0;
}

extern "C" int32_t zk_compress_frames_prefix(zk_ctx* c, const uint8_t* src, size_t n, uint32_t frame_size, int32_t level, int32_t checksum,
                                             const uint8_t* prefix, size_t prefix_len, uint8_t* dst, size_t dst_cap, uint32_t* c_sizes,
                                             uint32_t* d_sizes, uint32_t frames_cap, uint32_t* n_frames, size_t* dst_len) {
    if (!c) return ZK_ERR_INVALID_ARG;
    int32_t rc = zk_ctx_set_prefix(c, prefix, prefix_len);
    if (rc) return rc;
    if (c->c_ldm && c->cur_prefix_len && n) {
        // long-distance matching: index the part of the prefix the window reaches (window log 27 unless set, as libzstd)
        const uint32_t wl = c->c_window_log ? (uint32_t)c->c_window_log : 27u, tl = zk_encode_level_window_log(level);
        const uint32_t win_log = wl > tl ? wl : tl;
        const size_t span = c->cur_prefix_len < (1ull << win_log) ? c->cur_prefix_len : (size_t)1 << win_log;
        const uint32_t log = zk_ldm_index_log(span);
        if (c->cap_ldm < ((size_t)4 << log)) {
            if (c->d_ldm) cudaFree(c->d_ldm);
            c->d_ldm = nullptr; c->cap_ldm = 0;
            if (cudaMalloc((void**)&c->d_ldm, (size_t)4 << log) != cudaSuccess) { c->cur_prefix_len = 0; return ZK_ERR_ZSTD(ZKZ_MEMORY_ALLOCATION); }
            c->cap_ldm = (size_t)4 << log;
        }
        rc = zk_ldm_index_build(c->slot[0].stream, c->d_prefix, c->cur_prefix_len, 1u << win_log, c->d_ldm, log);
        if (!rc && cudaStreamSynchronize(c->slot[0].stream) != cudaSuccess) rc = ZK_ERR_CUDA;
        if (rc) { c->cur_prefix_len = 0; return rc == ZK_INT_CUDA ? ZK_ERR_CUDA : rc; }
        c->cur_ldm_log = log; c->cur_ldm_win = win_log;
    }
    rc = zk_compress_frames(c, src, n, frame_size, level, checksum, dst, dst_cap, c_sizes, d_sizes, frames_cap, n_frames, dst_len);
    c->cur_prefix_len = 0; c->cur_ldm_log = 0; c->cur_ldm_win = 0;
    return rc;
}

extern "C" int32_t zk_decompress_frames_prefix(zk_ctx* c, const uint8_t* comp, const uint64_t* c_off, const uint64_t* d_off, uint32_t n,
                                               uint8_t* dst, const uint32_t* d_need, int32_t verify, int32_t* status,
                                               const uint8_t* prefix, size_t prefix_len) {
    if (!c) return ZK_ERR_INVALID_ARG;
    int32_t rc = zk_ctx_set_prefix(c, prefix, prefix_len);
    if (rc) return rc;
    rc = zk_decompress_frames_upto(c, comp, c_off, d_off, n, dst, d_need, verify, status);
    c->cur_prefix_len = 0;
    return rc;
}
