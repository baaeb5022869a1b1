// fokl_ctx.cuh -- internal context shared by the translation units of libfokl_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>
#include "../../include/fokl_b200.h"

struct fokl_buf {
    void *ptr = nullptr;
    size_t bytes = 0;
};

struct fokl_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string err;
    int64_t launches = 0;
    // what the last fokl_gram_update(_ex) launched (fokl_gram_last_config); gram_cfg[0] < 0: none yet
    int64_t gram_cfg[9] = {-1, 0, 0, 0, 0, 0, 0, 0, 0};
    int num_sms = 148;
    int sm_budget = 0;        // > 0: SMs a batch of candidate models may plan for (fokl_ctx_set_sm_budget)
    size_t smem_optin = 0;
    int max_cluster = 8;      // largest thread-block cluster the eigensolver may use (portable limit)
    bool cluster_probed = false;

    // basis tables (device)
    double *cubic_tab = nullptr;
    int cubic_orders = 0, cubic_pieces = 0;
    double *bern_tab = nullptr;
    int bern_orders = 0, bern_row = 0;

    // deferred error flag written by kernels (device int), checked in fokl_ctx_synchronize
    int *d_flag = nullptr;

    // auxiliary streams (lazily created, non-blocking): independent kernels of one call -- the eigensolver launches
    // of different cluster sizes, the variate tables -- run side by side and are joined back into `stream` by events
    enum { kAux = 3 };
    cudaStream_t aux[kAux] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr;
    cudaEvent_t ev_join[kAux] = {nullptr, nullptr, nullptr};

    // optional high-priority stream for the latency-bound candidate stage (fokl_ctx_set_high_priority): its kernels are
    // dispatched ahead of the pending CTAs of bandwidth- / tensor-bound kernels that another context runs next to them
    bool hp_on = false;
    cudaStream_t hp_stream = nullptr;
    cudaEvent_t ev_hp_in = nullptr, ev_hp_out = nullptr;

    // recorded by fokl_candidates_eval right after its eigensolver launches (fokl_ctx_wait_eig)
    cudaEvent_t ev_eig = nullptr;
    bool ev_eig_set = false;

    // growable scratch buffers, indexed by purpose
    enum { B_META = 0, B_BASIS, B_GRAM, B_CAND_A, B_CAND_B, B_CAND_C, B_CAND_D, B_MISC, B_COUNT };
    fokl_buf bufs[B_COUNT];
};

#define FOKL_CHECK_CTX(ctx) \
    do { if (!(ctx)) return FOKL_EINVAL; } while (0)

#define FOKL_CUDA(ctx, call)                                                                      \
    do {                                                                                          \
        cudaError_t e__ = (call);                                                                 \
        if (e__ != cudaSuccess) {                                                                 \
            char b__[512];                                                                        \
            snprintf(b__, sizeof b__, "%s:%d: %s -> %s", __FILE__, __LINE__, #call,               \
                     cudaGetErrorString(e__));                                                    \
            (ctx)->err = b__;                                                                     \
            return FOKL_ECUDA;                                                                    \
        }                                                                                         \
    } while (0)

#define FOKL_FAIL(ctx, code, msg) \
    do { (ctx)->err = (msg); return (code); } while (0)

// returns nullptr (and sets ctx->err) on failure
void *fokl_scratch(fokl_ctx *ctx, int which, size_t bytes);

// Fork point: everything enqueued on ctx->stream so far.  fokl_aux_fork(i) then makes aux stream `i` wait for the
// most recent fork point and returns it (nullptr on error).
int fokl_fork_point(fokl_ctx *ctx);
cudaStream_t fokl_aux_fork(fokl_ctx *ctx, int i);
// Join: make ctx->stream wait for everything enqueued on aux stream `i`.
int fokl_aux_join(fokl_ctx *ctx, int i);

// Scope guard: inside it ctx->stream is the context's high-priority stream (if enabled), ordered after everything
// enqueued on the caller's stream so far; on exit the caller's stream is ordered after the scope's work.
struct fokl_hp_scope {
    fokl_ctx *ctx;
    cudaStream_t saved = nullptr;
    bool active = false;
    int rc = FOKL_OK;
    explicit fokl_hp_scope(fokl_ctx *c);
    ~fokl_hp_scope();
    fokl_hp_scope(const fokl_hp_scope &) = delete;
    fokl_hp_scope &operator=(const fokl_hp_scope &) = delete;
};

static inline int fokl_bind_device(fokl_ctx *ctx)
{
    FOKL_CUDA(ctx, cudaSetDevice(ctx->device));
    return FOKL_OK;
}

#define FOKL_LAUNCH_CHECK(ctx)                       \
    do {                                             \
        (ctx)->launches += 1;                        \
        FOKL_CUDA(ctx, cudaGetLastError());          \
    } while (0)
