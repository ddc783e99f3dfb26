// zk_ctx.h -- the context behind the C ABI's opaque zk_ctx (include/zeekstd_b200.h).
// Owns the CUDA streams, events, pinned/HBM staging and the per-slot codec workspaces.
#pragma once
#include "zk_decode.h"
#include "zk_encode.h"

#define ZK_SLOTS 8                        // pipeline depth of the host<->device paths (H2D | kernels | D2H overlap)

struct ZkSlot {
    cudaStream_t stream = nullptr;
    ZkDecodeWs dws;
    ZkEncodeWs ews;
    uint8_t* d_in = nullptr; size_t cap_in = 0;      // device staging for the host-pointer entry points
    uint8_t* d_out = nullptr; size_t cap_out = 0;
};

struct zk_ctx {
    int device = 0;
    int sm_count = 148;
    ZkSlot slot[ZK_SLOTS];
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaStream_t up = nullptr, down = nullptr;            // dedicated copy streams of the host-pointer decompress pipeline
    float last_ms = 0.f;
    uint8_t* d_prefix = nullptr; size_t cap_prefix = 0;   // device copy of the raw-content prefix of the *_prefix entry points
    uint32_t cur_prefix_len = 0;                          // != 0 while such a call is running: every sub-batch gets the prefix
    // context parameters (zk_ctx_set_cparameter / zk_ctx_set_dparameter); 0 = default
    int32_t c_window_log = 0, c_ldm = 0, d_window_log_max = 0;
    // long-distance-matching index of the prefix (zk_ldm_index_build): 2^ldm_log u32 slots, grown on demand
    uint32_t* d_ldm = nullptr; size_t cap_ldm = 0;
    uint32_t cur_ldm_log = 0, cur_ldm_win = 0;            // != 0 while a prefix call with LDM runs: index log, window log
    unsigned long long launches() const {
        unsigned long long n = 0;
        for (int i = 0; i < ZK_SLOTS; i++) n += slot[i].dws.launches + slot[i].ews.launches;
        return n;
    }
};

int zk_slot_ensure(ZkSlot* s, size_t need_in, size_t need_out);
