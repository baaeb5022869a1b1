// ctx.cu -- context management and the small utility kernels of libfokl_b200.so (sm_100a).
#include "fokl_ctx.cuh"
#include "fokl_math.cuh"
#include <string.h>

extern "C" int fokl_abi_version(void) { return FOKL_ABI_VERSION; }

void *fokl_scratch(fokl_ctx *ctx, int which, size_t bytes)
{
    fokl_buf &b = ctx->bufs[which];
    if (bytes == 0) bytes = 16;
    if (b.bytes >= bytes) return b.ptr;
    if (b.ptr) {
        // buffers may still be in use by enqueued work: drain the stream before freeing
        cudaStreamSynchronize(ctx->stream);
        cudaFree(b.ptr);
        b.ptr = nullptr;
        b.bytes = 0;
    }
    size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaMalloc(&b.ptr, want);
    if (e != cudaSuccess) {
        cudaGetLastError();
        e = cudaMalloc(&b.ptr, bytes);
        want = bytes;
    }
    if (e != cudaSuccess) {
        char m[256];
        snprintf(m, sizeof m, "workspace allocation of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
        ctx->err = m;
        b.ptr = nullptr;
        return nullptr;
    }
    b.bytes = want;
    return b.ptr;
}

int fokl_fork_point(fokl_ctx *ctx)
{
    if (!ctx->ev_fork) FOKL_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
    FOKL_CUDA(ctx, cudaEventRecord(ctx->ev_fork, ctx->stream));
    return FOKL_OK;
}

cudaStream_t fokl_aux_fork(fokl_ctx *ctx, int i)
{
    if (i < 0 || i >= fokl_ctx::kAux || !ctx->ev_fork) return nullptr;
    if (!ctx->aux[i]) {
        int least = 0, greatest = 0;
        if (ctx->hp_on) cudaDeviceGetStreamPriorityRange(&least, &greatest);
        if (cudaStreamCreateWithPriority(&ctx->aux[i], cudaStreamNonBlocking, ctx->hp_on ? greatest : 0) != cudaSuccess) return nullptr;
        if (cudaEventCreateWithFlags(&ctx->ev_join[i], cudaEventDisableTiming) != cudaSuccess) return nullptr;
    }
    if (cudaStreamWaitEvent(ctx->aux[i], ctx->ev_fork, 0) != cudaSuccess) return nullptr;
    return ctx->aux[i];
}

int fokl_aux_join(fokl_ctx *ctx, int i)
{
    if (i < 0 || i >= fokl_ctx::kAux || !ctx->aux[i]) FOKL_FAIL(ctx, FOKL_ESTATE, "aux stream join without fork");
    FOKL_CUDA(ctx, cudaEventRecord(ctx->ev_join[i], ctx->aux[i]));
    FOKL_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_join[i], 0));
    return FOKL_OK;
}

fokl_hp_scope::fokl_hp_scope(fokl_ctx *c) : ctx(c)
{
    if (!ctx || !ctx->hp_on) return;
    auto fail = [&](cudaError_t e, const char *what) {
        ctx->err = std::string("high-priority scope: ") + what + " -> " + cudaGetErrorString(e);
        rc = FOKL_ECUDA;
    };
    cudaError_t e;
    if (!ctx->hp_stream) {
        int least = 0, greatest = 0;
        if ((e = cudaDeviceGetStreamPriorityRange(&least, &greatest)) != cudaSuccess) { fail(e, "priority range"); return; }
        if ((e = cudaStreamCreateWithPriority(&ctx->hp_stream, cudaStreamNonBlocking, greatest)) != cudaSuccess)
            { fail(e, "stream create"); return; }
        if ((e = cudaEventCreateWithFlags(&ctx->ev_hp_in, cudaEventDisableTiming)) != cudaSuccess) { fail(e, "event create"); return; }
        if ((e = cudaEventCreateWithFlags(&ctx->ev_hp_out, cudaEventDisableTiming)) != cudaSuccess) { fail(e, "event create"); return; }
    }
    if ((e = cudaEventRecord(ctx->ev_hp_in, ctx->stream)) != cudaSuccess) { fail(e, "event record"); return; }
    if ((e = cudaStreamWaitEvent(ctx->hp_stream, ctx->ev_hp_in, 0)) != cudaSuccess) { fail(e, "stream wait"); return; }
    saved = ctx->stream;
    ctx->stream = ctx->hp_stream;
    active = true;
}

fokl_hp_scope::~fokl_hp_scope()
{
    if (!active) return;
    ctx->stream = saved;
    if (cudaEventRecord(ctx->ev_hp_out, ctx->hp_stream) == cudaSuccess) cudaStreamWaitEvent(saved, ctx->ev_hp_out, 0);
}

extern "C" int fokl_ctx_wait_eig(fokl_ctx *waiter, fokl_ctx *src)
{
    FOKL_CHECK_CTX(waiter);
    FOKL_CHECK_CTX(src);
    if (!src->ev_eig_set) return FOKL_OK;
    FOKL_CUDA(waiter, cudaStreamWaitEvent(waiter->stream, src->ev_eig, 0));
    return FOKL_OK;
}

extern "C" int fokl_ctx_set_high_priority(fokl_ctx *ctx, int on)
{
    FOKL_CHECK_CTX(ctx);
    ctx->hp_on = on != 0;
    return FOKL_OK;
}

extern "C" int fokl_ctx_create(fokl_ctx **out, int device, void *cuda_stream)
{
    if (!out) return FOKL_EINVAL;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) return FOKL_ECUDA;
    fokl_ctx *ctx = new fokl_ctx();
    ctx->device = device;
    if (cudaSetDevice(device) != cudaSuccess) { delete ctx; return FOKL_ECUDA; }
    // NULL is the CUDA legacy default stream -- the stream PyTorch enqueues on unless told otherwise, so
    // device buffers produced by torch and kernels launched here stay ordered without extra events.
    ctx->stream = (cudaStream_t)cuda_stream;
    ctx->own_stream = false;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) {
        ctx->num_sms = prop.multiProcessorCount;
        ctx->smem_optin = prop.sharedMemPerBlockOptin;
    }
    if (cudaMalloc(&ctx->d_flag, sizeof(int)) != cudaSuccess ||
        cudaMemsetAsync(ctx->d_flag, 0, sizeof(int), ctx->stream) != cudaSuccess) {
        delete ctx;
        return FOKL_ECUDA;
    }
    *out = ctx;
    return FOKL_OK;
}

extern "C" int fokl_ctx_destroy(fokl_ctx *ctx)
{
    if (!ctx) return FOKL_EINVAL;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (int i = 0; i < fokl_ctx::B_COUNT; ++i)
        if (ctx->bufs[i].ptr) cudaFree(ctx->bufs[i].ptr);
    if (ctx->cubic_tab) cudaFree(ctx->cubic_tab);
    if (ctx->bern_tab) cudaFree(ctx->bern_tab);
    if (ctx->d_flag) cudaFree(ctx->d_flag);
    for (int i = 0; i < fokl_ctx::kAux; ++i) {
        if (ctx->aux[i]) { cudaStreamSynchronize(ctx->aux[i]); cudaStreamDestroy(ctx->aux[i]); }
        if (ctx->ev_join[i]) cudaEventDestroy(ctx->ev_join[i]);
    }
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->hp_stream) { cudaStreamSynchronize(ctx->hp_stream); cudaStreamDestroy(ctx->hp_stream); }
    if (ctx->ev_eig) cudaEventDestroy(ctx->ev_eig);
    if (ctx->ev_hp_in) cudaEventDestroy(ctx->ev_hp_in);
    if (ctx->ev_hp_out) cudaEventDestroy(ctx->ev_hp_out);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return FOKL_OK;
}

extern "C" const char *fokl_last_error(fokl_ctx *ctx) { return ctx ? ctx->err.c_str() : "null ctx"; }

extern "C" int64_t fokl_launch_count(fokl_ctx *ctx) { return ctx ? ctx->launches : -1; }

extern "C" int fokl_ctx_set_sm_budget(fokl_ctx *ctx, int sms)
{
    FOKL_CHECK_CTX(ctx);
    ctx->sm_budget = sms > 0 ? sms : 0;
    return FOKL_OK;
}

extern "C" int fokl_ctx_synchronize(fokl_ctx *ctx)
{
    FOKL_CHECK_CTX(ctx);
    int rc = fokl_bind_device(ctx);
    if (rc) return rc;
    int flag = 0;
    FOKL_CUDA(ctx, cudaMemcpyAsync(&flag, ctx->d_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    FOKL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (flag) {
        FOKL_CUDA(ctx, cudaMemsetAsync(ctx->d_flag, 0, sizeof(int), ctx->stream));
        FOKL_FAIL(ctx, FOKL_ERANGE,
                  "Inputs are not normalized correctly (outside [0, 1]); try clean=True");
    }
    return FOKL_OK;
}

static int upload_table(fokl_ctx *ctx, double **dst, const double *tab, size_t count)
{
    if (*dst) {
        FOKL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        FOKL_CUDA(ctx, cudaFree(*dst));
        *dst = nullptr;
    }
    FOKL_CUDA(ctx, cudaMalloc(dst, count * sizeof(double)));
    FOKL_CUDA(ctx, cudaMemcpyAsync(*dst, tab, count * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    FOKL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return FOKL_OK;
}

extern "C" int fokl_set_phis_cubic(fokl_ctx *ctx, const double *tab, int n_orders, int n_piece)
{
    FOKL_CHECK_CTX(ctx);
    if (!tab || n_orders < 1 || n_piece < 1 || n_piece > 65535) FOKL_FAIL(ctx, FOKL_EINVAL, "bad cubic table");
    int rc = fokl_bind_device(ctx);
    if (rc) return rc;
    rc = upload_table(ctx, &ctx->cubic_tab, tab, (size_t)n_orders * n_piece * 4);
    if (rc) return rc;
    ctx->cubic_orders = n_orders;
    ctx->cubic_pieces = n_piece;
    return FOKL_OK;
}

extern "C" int fokl_set_phis_bernoulli(fokl_ctx *ctx, const double *tab, int n_orders, int row_len)
{
    FOKL_CHECK_CTX(ctx);
    if (!tab || n_orders < 1 || row_len < 2) FOKL_FAIL(ctx, FOKL_EINVAL, "bad bernoulli table");
    int rc = fokl_bind_device(ctx);
    if (rc) return rc;
    rc = upload_table(ctx, &ctx->bern_tab, tab, (size_t)n_orders * row_len);
    if (rc) return rc;
    ctx->bern_orders = n_orders;
    ctx->bern_row = row_len;
    return FOKL_OK;
}

// ------------------------------------------------------------------------------------------------
// small kernels
// ------------------------------------------------------------------------------------------------

__global__ void fill_ones_kernel(double *col, int64_t n)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) col[i] = 1.0;
}

extern "C" int fokl_fill_ones(fokl_ctx *ctx, double *col, int64_t n)
{
    FOKL_CHECK_CTX(ctx);
    if (!col || n < 0) FOKL_FAIL(ctx, FOKL_EINVAL, "fill_ones: bad argument");
    int rc = fokl_bind_device(ctx);
    if (rc) return rc;
    if (n == 0) return FOKL_OK;
    int blocks = (int)((n + 255) / 256 < (int64_t)ctx->num_sms * 8 ? (n + 255) / 256 : (int64_t)ctx->num_sms * 8);
    fill_ones_kernel<<<blocks, 256, 0, ctx->stream>>>(col, n);
    FOKL_LAUNCH_CHECK(ctx);
    return FOKL_OK;
}

// deterministic two-stage reductions ---------------------------------------------------------------
template <int NV>
__device__ __forceinline__ void block_reduce(double (&v)[NV], double *sm /* NV * 32 */)
{
#pragma unroll
    for (int q = 0; q < NV; ++q)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[q] += __shfl_xor_sync(0xffffffffu, v[q], o);
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    if (lane == 0)
        for (int q = 0; q < NV; ++q) sm[q * 32 + warp] = v[q];
    __syncthreads();
    if (warp == 0) {
        for (int q = 0; q < NV; ++q) {
            double x = lane < nwarp ? sm[q * 32 + lane] : 0.0;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
            v[q] = x;
        }
    }
}

__global__ void y_moments_partial(const double *__restrict__ y, int64_t n, double *__restrict__ part)
{
    __shared__ double sm[2 * 32];
    int64_t per = (n + gridDim.x - 1) / gridDim.x;
    int64_t lo = (int64_t)blockIdx.x * per, hi = lo + per < n ? lo + per : n;
    double v[2] = {0.0, 0.0};
    for (int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) {
        double t = y[i];
        v[0] += t;
        v[1] += t * t;
    }
    block_reduce<2>(v, sm);
    if (threadIdx.x == 0) {
        part[2 * blockIdx.x] = v[0];
        part[2 * blockIdx.x + 1] = v[1];
    }
}

__global__ void final_sum_kernel(const double *__restrict__ part, int nblocks, int nv, double *__restrict__ out,
                                 int out_offset)
{
    int q = threadIdx.x;
    if (q >= nv) return;
    double s = 0.0;
    for (int b = 0; b < nblocks; ++b) s += part[(int64_t)b * nv + q];
    out[out_offset + q] = s;
}

__global__ void set_scalar_kernel(double *out, double v) { out[0] = v; }

extern "C" int fokl_y_moments(fokl_ctx *ctx, const double *y, int64_t n, double *out)
{
    FOKL_CHECK_CTX(ctx);
    if (!y || !out || n < 1) FOKL_FAIL(ctx, FOKL_EINVAL, "y_moments: bad argument");
    int rc = fokl_bind_device(ctx);
    if (rc) return rc;
    int blocks = (int)((n + 4095) / 4096);
    if (blocks > ctx->num_sms * 4) blocks = ctx->num_sms * 4;
    if (blocks < 1) blocks = 1;
    double *part = (double *)fokl_scratch(ctx, fokl_ctx::B_MISC, (size_t)blocks * 2 * sizeof(double));
    if (!part) return FOKL_ENOMEM;
    y_moments_partial<<<blocks, 256, 0, ctx->stream>>>(y, n, part);
    FOKL_LAUNCH_CHECK(ctx);
    set_scalar_kernel<<<1, 1, 0, ctx->stream>>>(out, (double)n);
    FOKL_LAUNCH_CHECK(ctx);
    final_sum_kernel<<<1, 32, 0, ctx->stream>>>(part, blocks, 2, out, 1);
    FOKL_LAUNCH_CHECK(ctx);
    return FOKL_OK;
}

// Gram bookkeeping ---------------------------------------------------------------------------------
__global__ void gram_scatter_kernel(const double *__restrict__ block, int p_old, int c, double *__restrict__ G,
                                    int64_t ldg, double *__restrict__ Xty)
{
    int p = p_old + c;
    int64_t total = (int64_t)(p + 1) * c;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (int64_t)gridDim.x * blockDim.x) {
        int i = (int)(t / c), j = (int)(t % c);
        if (i == p) {
            Xty[p_old + j] = block[t];
            continue;
        }
        double v = block[t];
        if (i >= p_old) {
            // diagonal block: take the entry computed for (min, max) so G is exactly symmetric
            int a = i - p_old;
            if (a > j) v = block[(int64_t)(p_old + j) * c + a];
        }
        G[(int64_t)i * ldg + (p_old + j)] = v;
        G[(int64_t)(p_old + j) * ldg + i] = v;
    }
}

extern "C" int fokl_gram_scatter(fokl_ctx *ctx, const double *block, int p_old, int c, double *G, int64_t ldg,
                                 double *Xty)
{
    FOKL_CHECK_CTX(ctx);
    if (!block || !G || !Xty || p_old < 0 || c < 1 || ldg < p_old + c)
        FOKL_FAIL(ctx, FOKL_EINVAL, "gram_scatter: bad argument");
    int rc = fokl_bind_device(ctx);
    if (rc) return rc;
    int64_t total = (int64_t)(p_old + c + 1) * c;
    int blocks = (int)((total + 255) / 256);
    if (blocks > 1024) blocks = 1024;
    gram_scatter_kernel<<<blocks, 256, 0, ctx->stream>>>(block, p_old, c, G, ldg, Xty);
    FOKL_LAUNCH_CHECK(ctx);
    return FOKL_OK;
}

__global__ void gram_compact_kernel(const double *__restrict__ G, int64_t ldg, const double *__restrict__ Xty,
                                    const int *__restrict__ keep, int p_new, double *__restrict__ Go,
                                    int64_t ldo, double *__restrict__ Xo)
{
    int64_t total = (int64_t)p_new * p_new;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (int64_t)gridDim.x * blockDim.x) {
        int a = (int)(t / p_new), b = (int)(t % p_new);
        Go[(int64_t)a * ldo + b] = G[(int64_t)keep[a] * ldg + keep[b]];
        if (b == 0) Xo[a] = Xty[keep[a]];
    }
}

extern "C" int fokl_gram_compact(fokl_ctx *ctx, const double *G, int64_t ldg, const double *Xty,
                                 const int32_t *keep, int p_new, double *G_out, int64_t ldg_out, double *Xty_out)
{
    FOKL_CHECK_CTX(ctx);
    if (!G || !Xty || !keep || !G_out || !Xty_out || p_new < 1 || ldg_out < p_new)
        FOKL_FAIL(ctx, FOKL_EINVAL, "gram_compact: bad argument");
    if (G == G_out || Xty == Xty_out) FOKL_FAIL(ctx, FOKL_EINVAL, "gram_compact: must not alias");
    int rc = fokl_bind_device(ctx);
    if (rc) return rc;
    int *dkeep = (int *)fokl_scratch(ctx, fokl_ctx::B_META, (size_t)p_new * sizeof(int));
    if (!dkeep) return FOKL_ENOMEM;
    FOKL_CUDA(ctx, cudaMemcpyAsync(dkeep, keep, (size_t)p_new * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    int64_t total = (int64_t)p_new * p_new;
    int blocks = (int)((total + 255) / 256);
    if (blocks > 2048) blocks = 2048;
    gram_compact_kernel<<<blocks, 256, 0, ctx->stream>>>(G, ldg, Xty, dkeep, p_new, G_out, ldg_out, Xty_out);
    FOKL_LAUNCH_CHECK(ctx);
    // dkeep is reused by later calls: make sure the async H2D source (pageable) was consumed
    return FOKL_OK;
}

extern "C" int fokl_columns_compact(fokl_ctx *ctx, double *X, int64_t ld, int64_t n, const int32_t *keep, int p_new)
{
    FOKL_CHECK_CTX(ctx);
    if (!X || !keep || p_new < 0 || n < 0 || ld < n) FOKL_FAIL(ctx, FOKL_EINVAL, "columns_compact: bad argument");
    int rc = fokl_bind_device(ctx);
    if (rc) return rc;
    for (int a = 0; a < p_new; ++a) {
        if (keep[a] < a || (a > 0 && keep[a] <= keep[a - 1]))
            FOKL_FAIL(ctx, FOKL_EINVAL, "columns_compact: keep must be ascending with keep[a] >= a");
        if (keep[a] == a) continue;
        FOKL_CUDA(ctx, cudaMemcpyAsync(X + (int64_t)a * ld, X + (int64_t)keep[a] * ld, (size_t)n * sizeof(double),
                                       cudaMemcpyDeviceToDevice, ctx->stream));
    }
    return FOKL_OK;
}

// residual moments -----------------------------------------------------------------------------------
__global__ void residual_partial(const double *__restrict__ X, int64_t ld, int64_t n, int p,
                                 const int *__restrict__ cols, const double *__restrict__ beta,
                                 const double *__restrict__ y, double *__restrict__ part)
{
    extern __shared__ double sb[];   // p betas + 64 reduce
    double *sm = sb + p;
    for (int j = threadIdx.x; j < p; j += blockDim.x) sb[j] = beta[j];
    __syncthreads();
    int64_t per = (n + gridDim.x - 1) / gridDim.x;
    int64_t lo = (int64_t)blockIdx.x * per, hi = lo + per < n ? lo + per : n;
    double v[2] = {0.0, 0.0};
    for (int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) {
        double f = 0.0;
        for (int j = 0; j < p; ++j) {
            int64_t cj = cols ? cols[j] : j;
            f += X[cj * ld + i] * sb[j];
        }
        double r = y[i] - f;
        v[0] += r;
        v[1] += r * r;
    }
    block_reduce<2>(v, sm);
    if (threadIdx.x == 0) {
        part[2 * blockIdx.x] = v[0];
        part[2 * blockIdx.x + 1] = v[1];
    }
}

extern "C" int fokl_residual_moments(fokl_ctx *ctx, const double *X, int64_t ld, int64_t n, int p,
                                     const int32_t *cols, const double *beta, const double *y, double *out)
{
    FOKL_CHECK_CTX(ctx);
    if (!X || !beta || !y || !out || n < 1 || p < 1) FOKL_FAIL(ctx, FOKL_EINVAL, "residual_moments: bad argument");
    int rc = fokl_bind_device(ctx);
    if (rc) return rc;
    int blocks = (int)((n + 1023) / 1024);
    if (blocks > ctx->num_sms * 4) blocks = ctx->num_sms * 4;
    size_t meta = (size_t)blocks * 2 * sizeof(double) + 64;
    char *base = (char *)fokl_scratch(ctx, fokl_ctx::B_MISC, meta + (size_t)p * sizeof(int));
    if (!base) return FOKL_ENOMEM;
    double *part = (double *)base;
    int *dcols = nullptr;
    if (cols) {
        dcols = (int *)(base + meta);
        FOKL_CUDA(ctx, cudaMemcpyAsync(dcols, cols, (size_t)p * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    }
    size_t smem = ((size_t)p + 64) * sizeof(double);
    if (smem > 48 * 1024) {
        if (smem > ctx->smem_optin) FOKL_FAIL(ctx, FOKL_EINVAL, "residual_moments: p too large");
        FOKL_CUDA(ctx, cudaFuncSetAttribute(residual_partial, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    residual_partial<<<blocks, 256, smem, ctx->stream>>>(X, ld, n, p, dcols, beta, y, part);
    FOKL_LAUNCH_CHECK(ctx);
    final_sum_kernel<<<1, 32, 0, ctx->stream>>>(part, blocks, 2, out, 0);
    FOKL_LAUNCH_CHECK(ctx);
    return FOKL_OK;
}

// evaluate: out[i][d] = sum_j X[i][j] betas[d][j] ------------------------------------------------------
template <int DT>
__global__ void predict_draws_kernel(const double *__restrict__ X, int64_t ld, int64_t n, int p,
                                     const double *__restrict__ betas, int n_draws, double *__restrict__ out)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int d0 = blockIdx.y * DT;
    if (i >= n) return;
    double acc[DT];
#pragma unroll
    for (int q = 0; q < DT; ++q) acc[q] = 0.0;
    for (int j = 0; j < p; ++j) {
        double xv = X[(int64_t)j * ld + i];
#pragma unroll
        for (int q = 0; q < DT; ++q) {
            int d = d0 + q;
            double b = d < n_draws ? __ldg(betas + (int64_t)d * p + j) : 0.0;
            acc[q] += xv * b;
        }
    }
#pragma unroll
    for (int q = 0; q < DT; ++q)
        if (d0 + q < n_draws) out[i * n_draws + d0 + q] = acc[q];
}

extern "C" int fokl_predict_draws(fokl_ctx *ctx, const double *X, int64_t ld, int64_t n, int p, const double *betas,
                                  int n_draws, double *out)
{
    FOKL_CHECK_CTX(ctx);
    if (!X || !betas || !out || n < 1 || p < 1 || n_draws < 1) FOKL_FAIL(ctx, FOKL_EINVAL, "predict_draws: bad argument");
    int rc = fokl_bind_device(ctx);
    if (rc) return rc;
    const int DT = 8;
    dim3 grid((unsigned)((n + 127) / 128), (unsigned)((n_draws + DT - 1) / DT));
    predict_draws_kernel<DT><<<grid, 128, 0, ctx->stream>>>(X, ld, n, p, betas, n_draws, out);
    FOKL_LAUNCH_CHECK(ctx);
    return FOKL_OK;
}

// clean/_normalize ---------------------------------------------------------------------------------------
__global__ void minmax_partial(const double *__restrict__ x, int64_t n, int64_t ldx, double *__restrict__ part)
{
    __shared__ double smin[32], smax[32];
    const double *col = x + (int64_t)blockIdx.y * ldx;
    int64_t per = (n + gridDim.x - 1) / gridDim.x;
    int64_t lo = (int64_t)blockIdx.x * per, hi = lo + per < n ? lo + per : n;
    double mn = INFINITY, mx = -INFINITY;
    for (int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) {
        double t = col[i];
        mn = fmin(mn, t);
        mx = fmax(mx, t);
    }
    for (int o = 16; o > 0; o >>= 1) {
        mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    if (lane == 0) { smin[warp] = mn; smax[warp] = mx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < nwarp; ++w) { mn = fmin(mn, smin[w]); mx = fmax(mx, smax[w]); }
        part[2 * ((int64_t)blockIdx.y * gridDim.x + blockIdx.x)] = mn;
        part[2 * ((int64_t)blockIdx.y * gridDim.x + blockIdx.x) + 1] = mx;
    }
}

__global__ void minmax_final(const double *__restrict__ part, int nblocks, double *__restrict__ out)
{
    int k = blockIdx.x;
    if (threadIdx.x != 0) return;
    double mn = INFINITY, mx = -INFINITY;
    for (int b = 0; b < nblocks; ++b) {
        mn = fmin(mn, part[2 * ((int64_t)k * nblocks + b)]);
        mx = fmax(mx, part[2 * ((int64_t)k * nblocks + b) + 1]);
    }
    out[2 * k] = mn;
    out[2 * k + 1] = mx;
}

extern "C" int fokl_column_minmax(fokl_ctx *ctx, const double *x, int64_t n, int64_t ldx, int m, double *minmax_out)
{
    FOKL_CHECK_CTX(ctx);
    if (!x || !minmax_out || n < 1 || m < 1 || ldx < n) FOKL_FAIL(ctx, FOKL_EINVAL, "column_minmax: bad argument");
    int rc = fokl_bind_device(ctx);
    if (rc) return rc;
    int blocks = (int)((n + 4095) / 4096);
    if (blocks > ctx->num_sms * 2) blocks = ctx->num_sms * 2;
    double *part = (double *)fokl_scratch(ctx, fokl_ctx::B_MISC, (size_t)blocks * m * 2 * sizeof(double));
    if (!part) return FOKL_ENOMEM;
    minmax_partial<<<dim3(blocks, m), 256, 0, ctx->stream>>>(x, n, ldx, part);
    FOKL_LAUNCH_CHECK(ctx);
    minmax_final<<<m, 32, 0, ctx->stream>>>(part, blocks, minmax_out);
    FOKL_LAUNCH_CHECK(ctx);
    return FOKL_OK;
}

struct MinMaxArg { double v[64]; };

__global__ void normalize_kernel(double *__restrict__ x, int64_t n, int64_t ldx, MinMaxArg mm)
{
    double *col = x + (int64_t)blockIdx.y * ldx;
    double lo = mm.v[2 * blockIdx.y], hi = mm.v[2 * blockIdx.y + 1];
    double span = __dsub_rn(hi, lo);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        col[i] = __ddiv_rn(__dsub_rn(col[i], lo), span);   // FR:437
}

extern "C" int fokl_normalize(fokl_ctx *ctx, double *x, int64_t n, int64_t ldx, int m, const double *minmax)
{
    FOKL_CHECK_CTX(ctx);
    if (!x || !minmax || n < 1 || m < 1 || ldx < n) FOKL_FAIL(ctx, FOKL_EINVAL, "normalize: bad argument");
    int rc = fokl_bind_device(ctx);
    if (rc) return rc;
    int blocks = (int)((n + 255) / 256);
    if (blocks > ctx->num_sms * 8) blocks = ctx->num_sms * 8;
    // the bounds travel by value, 32 columns per launch: any number of inputs without a device copy of the bounds
    for (int k0 = 0; k0 < m; k0 += 32) {
        int mk = m - k0 < 32 ? m - k0 : 32;
        MinMaxArg mm;
        memset(&mm, 0, sizeof mm);
        for (int k = 0; k < 2 * mk; ++k) mm.v[k] = minmax[2 * k0 + k];
        normalize_kernel<<<dim3(blocks, mk), 256, 0, ctx->stream>>>(x + (int64_t)k0 * ldx, n, ldx, mm);
        FOKL_LAUNCH_CHECK(ctx);
    }
    return FOKL_OK;
}

// train split (FR:532-542 `inputs[trainlog, :]`): count / scan / scatter over tiles of kCompactTile rows --------------
// The kept count is needed on the host before anything is written (ldx_out is checked against it and n_out returned),
// so the count is its own pass; the scatter then re-reads the tile's mask bytes (N bytes against 8 N (m + 1) of values).
static constexpr int kCompactThreads = 256;
static constexpr int kCompactPer = 16;                                   // rows per thread and tile pass
static constexpr int kCompactTile = kCompactThreads * kCompactPer;       // 4096 rows per block

__global__ void __launch_bounds__(kCompactThreads) rows_compact_count(const uint8_t *__restrict__ keep, int64_t n,
                                                                      int64_t *__restrict__ tile_count)
{
    int64_t base = (int64_t)blockIdx.x * kCompactTile;
    int c = 0;
#pragma unroll
    for (int r = 0; r < kCompactPer; ++r) {
        int64_t i = base + r * kCompactThreads + threadIdx.x;
        c += (i < n && keep[i]) ? 1 : 0;
    }
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    __shared__ int warp_c[kCompactThreads / 32];
    if ((threadIdx.x & 31) == 0) warp_c[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < kCompactThreads / 32; ++w) t += warp_c[w];
        tile_count[blockIdx.x] = t;
    }
}

// exclusive scan of the tile counts in place (one block); total -> *total
__global__ void __launch_bounds__(1024) rows_compact_scan(int64_t *__restrict__ tile_off, int64_t tiles,
                                                          int64_t *__restrict__ total)
{
    __shared__ int64_t warp_s[32];
    __shared__ int64_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t b0 = 0; b0 < tiles; b0 += 1024) {
        int64_t i = b0 + threadIdx.x;
        int64_t v = i < tiles ? tile_off[i] : 0, s = v;
        for (int o = 1; o < 32; o <<= 1) {
            int64_t t = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += t;
        }
        if (lane == 31) warp_s[warp] = s;
        __syncthreads();
        if (warp == 0) {
            int64_t w = warp_s[lane];
            for (int o = 1; o < 32; o <<= 1) {
                int64_t t = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += t;
            }
            warp_s[lane] = w;                                            // inclusive over warps
        }
        __syncthreads();
        int64_t incl = s + (warp > 0 ? warp_s[warp - 1] : 0) + carry;
        if (i < tiles) tile_off[i] = incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry = incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}

// one tile per block: each thread's kCompactPer rows get their output position (or -1) from warp ballots and a scan
// of the warp totals, then every column (x's m, then y) is copied through those positions
__global__ void __launch_bounds__(kCompactThreads) rows_compact_scatter(
    const double *__restrict__ x, const double *__restrict__ y, int64_t n, int64_t ldx, int m,
    const uint8_t *__restrict__ keep, const int64_t *__restrict__ tile_off, double *__restrict__ x_out,
    double *__restrict__ y_out, int64_t ldx_out)
{
    __shared__ int warp_c[kCompactThreads / 32];
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int64_t base = (int64_t)blockIdx.x * kCompactTile;
    int64_t out0 = tile_off[blockIdx.x];
    int off = 0;
    int pos[kCompactPer];                                                // position within the tile's output run
#pragma unroll
    for (int r = 0; r < kCompactPer; ++r) {
        int64_t i = base + r * kCompactThreads + threadIdx.x;
        bool k = i < n && keep[i];
        unsigned bal = __ballot_sync(0xffffffffu, k);
        if (lane == 0) warp_c[warp] = __popc(bal);
        __syncthreads();
        int before = 0, all = 0;
#pragma unroll
        for (int w = 0; w < kCompactThreads / 32; ++w) {
            int c = warp_c[w];
            before += w < warp ? c : 0;
            all += c;
        }
        pos[r] = k ? off + before + __popc(bal & ((1u << lane) - 1u)) : -1;
        off += all;
        __syncthreads();
    }
    for (int c = 0; c <= m; ++c) {
        const double *src = c < m ? x + (int64_t)c * ldx : y;
        double *dst = (c < m ? x_out + (int64_t)c * ldx_out : y_out) + out0;
#pragma unroll
        for (int r = 0; r < kCompactPer; ++r) {
            int64_t i = base + r * kCompactThreads + threadIdx.x;
            if (pos[r] >= 0) dst[pos[r]] = src[i];
        }
    }
}

// rows [n_out, ldx_out) of every output column and of y_out = 0.0 (Engine.upload's padding)
__global__ void rows_compact_pad(double *__restrict__ x_out, double *__restrict__ y_out, int m, int64_t n_out,
                                 int64_t ldx_out)
{
    int c = blockIdx.y;
    double *dst = c < m ? x_out + (int64_t)c * ldx_out : y_out;
    for (int64_t i = n_out + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < ldx_out;
         i += (int64_t)gridDim.x * blockDim.x)
        dst[i] = 0.0;
}

extern "C" int fokl_rows_compact(fokl_ctx *ctx, const double *x, const double *y, int64_t n, int64_t ldx, int m,
                                 const uint8_t *keep, double *x_out, double *y_out, int64_t ldx_out, int64_t *n_out)
{
    FOKL_CHECK_CTX(ctx);
    if (!x || !y || !keep || !x_out || !y_out || !n_out || n < 1 || m < 1 || ldx < n || ldx_out < 0)
        FOKL_FAIL(ctx, FOKL_EINVAL, "rows_compact: bad argument");
    int rc = fokl_bind_device(ctx);
    if (rc) return rc;
    int64_t tiles = (n + kCompactTile - 1) / kCompactTile;
    if (tiles > 0x7fffffffLL) FOKL_FAIL(ctx, FOKL_EINVAL, "rows_compact: n too large");
    int64_t *scr = (int64_t *)fokl_scratch(ctx, fokl_ctx::B_MISC, (size_t)(tiles + 1) * sizeof(int64_t));
    if (!scr) return FOKL_ENOMEM;
    rows_compact_count<<<(unsigned)tiles, kCompactThreads, 0, ctx->stream>>>(keep, n, scr);
    FOKL_LAUNCH_CHECK(ctx);
    rows_compact_scan<<<1, 1024, 0, ctx->stream>>>(scr, tiles, scr + tiles);
    FOKL_LAUNCH_CHECK(ctx);
    int64_t kept = 0;
    FOKL_CUDA(ctx, cudaMemcpyAsync(&kept, scr + tiles, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    FOKL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ldx_out < kept) FOKL_FAIL(ctx, FOKL_EINVAL, "rows_compact: ldx_out below the kept row count");
    rows_compact_scatter<<<(unsigned)tiles, kCompactThreads, 0, ctx->stream>>>(x, y, n, ldx, m, keep, scr, x_out,
                                                                               y_out, ldx_out);
    FOKL_LAUNCH_CHECK(ctx);
    if (ldx_out > kept) {
        int64_t pad = ldx_out - kept;
        int blocks = (int)((pad + 255) / 256);
        if (blocks > ctx->num_sms * 4) blocks = ctx->num_sms * 4;
        rows_compact_pad<<<dim3(blocks, m + 1), 256, 0, ctx->stream>>>(x_out, y_out, m, kept, ldx_out);
        FOKL_LAUNCH_CHECK(ctx);
    }
    *n_out = kept;
    return FOKL_OK;
}
