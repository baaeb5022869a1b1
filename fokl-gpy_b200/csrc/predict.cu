// predict.cu -- fokl_predict_summary: per-row mean and two order statistics of X @ betas' without writing the
// N x n_draws product to HBM (evaluate / coverage3 / bss_derivatives at training-set scale).
//
// Rows are processed in chunks whose rows x n_draws block of values (<= kChunkBytes) stays in L2:
//   1. predict_tile_kernel: register-tiled DFMA product of the chunk, v[i][d] = fma chain over j = 0 .. p-1 from 0.0,
//      the exact operation order of predict_draws_kernel (ctx.cu), so both entry points give the same bits;
//   2. predict_summary_kernel: one warp per row reads the row back (staged in shared memory when it is short), forms
//      numpy's pairwise mean, then selects the two ranks on order keys written over the row (predict_math.cuh).
#include "fokl_ctx.cuh"
#include "predict_math.cuh"

namespace {

constexpr int kTileRows = 128, kTileDraws = 64, kTileK = 16, kTileThreads = 256;
constexpr size_t kChunkBytes = 32u << 20;        // one chunk's values: well inside the 126 MB L2
constexpr int kMaxChunkRows = 1 << 16;
constexpr int kStageMaxDraws = 2048;             // rows up to this many draws are summarised from shared memory
constexpr int kSummaryWarps = 4;

// thread (tx, ty) = (lane, warp) owns rows tx + 32 a (a < 4) and draws 8 ty + b (b < 8) of a 128 x 64 tile
__global__ void __launch_bounds__(kTileThreads)
predict_tile_kernel(const double *__restrict__ X, int64_t ld, int64_t n, int p, const double *__restrict__ betas,
                    int n_draws, double *__restrict__ V)
{
    __shared__ double xs[kTileK][kTileRows];
    __shared__ __align__(16) double bs[kTileK][kTileDraws];
    const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
    const int64_t r0 = (int64_t)blockIdx.x * kTileRows;
    const int d0 = blockIdx.y * kTileDraws;
    double acc[4][8];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 8; ++b) acc[a][b] = 0.0;

    for (int j0 = 0; j0 < p; j0 += kTileK) {
        for (int e = tid; e < kTileK * kTileRows; e += kTileThreads) {
            int kk = e / kTileRows, r = e % kTileRows, j = j0 + kk;
            int64_t i = r0 + r;
            xs[kk][r] = (j < p && i < n) ? X[(int64_t)j * ld + i] : 0.0;
        }
        for (int e = tid; e < kTileK * kTileDraws; e += kTileThreads) {
            int kk = e % kTileK, dd = e / kTileK, j = j0 + kk, d = d0 + dd;
            bs[kk][dd] = (j < p && d < n_draws) ? __ldg(betas + (int64_t)d * p + j) : 0.0;
        }
        __syncthreads();
        const int kn = p - j0 < kTileK ? p - j0 : kTileK;   // no FMA past column p-1: fma(0, 0, -0.0) is +0.0
        for (int kk = 0; kk < kn; ++kk) {
            double xv[4], bv[8];
#pragma unroll
            for (int a = 0; a < 4; ++a) xv[a] = xs[kk][tx + 32 * a];
#pragma unroll
            for (int b = 0; b < 8; b += 2) {
                double2 t = *reinterpret_cast<const double2 *>(&bs[kk][8 * ty + b]);
                bv[b] = t.x;
                bv[b + 1] = t.y;
            }
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 8; ++b) acc[a][b] = __fma_rn(xv[a], bv[b], acc[a][b]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        int64_t i = r0 + tx + 32 * a;
        if (i >= n) continue;
#pragma unroll
        for (int b = 0; b < 8; ++b) {
            int d = d0 + 8 * ty + b;
            if (d < n_draws) V[i * n_draws + d] = acc[a][b];
        }
    }
}

__device__ __forceinline__ uint64_t warp_min_u64(uint64_t v)
{
    for (int o = 16; o > 0; o >>= 1) {
        uint64_t y = __shfl_xor_sync(0xffffffffu, v, o);
        v = y < v ? y : v;
    }
    return v;
}

__device__ __forceinline__ uint64_t warp_max_u64(uint64_t v)
{
    for (int o = 16; o > 0; o >>= 1) {
        uint64_t y = __shfl_xor_sync(0xffffffffu, v, o);
        v = y > v ? y : v;
    }
    return v;
}

// shared memory of one warp, in doubles: 256 uint32 counters, the leaf sums, the staged row (stage only)
__host__ __device__ inline int summary_warp_doubles(int n_draws, int leaves, bool stage)
{
    return 128 + leaves + (stage ? n_draws : 0);
}

__global__ void predict_summary_kernel(double *__restrict__ V, int64_t n, int n_draws, int leaves, int stage,
                                       int rank_lo, int rank_hi, double *__restrict__ mean_out,
                                       double *__restrict__ lo_out, double *__restrict__ hi_out)
{
    extern __shared__ double sm[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    double *mine = sm + (size_t)warp * summary_warp_doubles(n_draws, leaves, stage != 0);
    uint32_t *hist = reinterpret_cast<uint32_t *>(mine);
    double *leaf = mine + 128;
    for (int64_t i = (int64_t)blockIdx.x * wpb + warp; i < n; i += (int64_t)gridDim.x * wpb) {
        double *v = V + i * n_draws;
        if (stage) {
            double *row = leaf + leaves;
            for (int d = lane; d < n_draws; d += 32) row[d] = v[d];
            v = row;
            __syncwarp();
        }
        // pairwise mean: the leaves on the lanes, the tree on lane 0
        int2 *span = reinterpret_cast<int2 *>(leaf);
        fokl::pw_leaves(n_draws, [&](int t, int off, int len) {
            if ((t & 31) == lane) span[t] = make_int2(off, len);
        });
        for (int t = lane; t < leaves; t += 32) {
            int2 s = span[t];
            leaf[t] = fokl::pw_leaf(v + s.x, s.y);
        }
        __syncwarp();
        if (lane == 0) mean_out[i] = fokl::pw_mean(fokl::pw_tree(n_draws, leaf), n_draws);
        if (rank_lo >= 0) {
            uint64_t *keys = reinterpret_cast<uint64_t *>(v);
            uint64_t kmin = ~0ull, kmax = 0ull;
            for (int d = lane; d < n_draws; d += 32) {
                uint64_t k = fokl::order_key(v[d]);
                keys[d] = k;
                kmin = k < kmin ? k : kmin;
                kmax = k > kmax ? k : kmax;
            }
            kmin = warp_min_u64(kmin);
            kmax = warp_max_u64(kmax);
            __syncwarp();
            uint64_t klo = fokl::select_key(keys, n_draws, rank_lo, hist, lane, 32, kmin, kmax);
            uint64_t khi = rank_hi == rank_lo ? klo : fokl::select_key(keys, n_draws, rank_hi, hist, lane, 32, kmin, kmax);
            if (lane == 0) {
                lo_out[i] = fokl::key_value(klo);
                hi_out[i] = fokl::key_value(khi);
            }
        }
        __syncwarp();
    }
}

}  // namespace

extern "C" int fokl_predict_summary(fokl_ctx *ctx, const double *X, int64_t ld, int64_t n, int p, const double *betas,
                                    int n_draws, int rank_lo, int rank_hi, double *mean_out, double *lo_out,
                                    double *hi_out)
{
    FOKL_CHECK_CTX(ctx);
    if (!X || !betas || !mean_out || n < 1 || p < 1 || ld < n || n_draws < 1)
        FOKL_FAIL(ctx, FOKL_EINVAL, "predict_summary: bad argument");
    const bool ranks = rank_lo >= 0 || rank_hi >= 0;
    if (ranks && (!lo_out || !hi_out || rank_lo < 0 || rank_hi < 0 || rank_lo >= n_draws || rank_hi >= n_draws))
        FOKL_FAIL(ctx, FOKL_EINVAL, "predict_summary: ranks must both be -1 or both lie in [0, n_draws)");
    if (!ranks && (rank_lo != -1 || rank_hi != -1))
        FOKL_FAIL(ctx, FOKL_EINVAL, "predict_summary: ranks must both be -1 or both lie in [0, n_draws)");
    int rc = fokl_bind_device(ctx);
    if (rc) return rc;

    int64_t rows = (int64_t)(kChunkBytes / ((size_t)n_draws * sizeof(double))) / kTileRows * kTileRows;
    if (rows < kTileRows) rows = kTileRows;
    if (rows > kMaxChunkRows) rows = kMaxChunkRows;
    const int64_t n_up = (n + kTileRows - 1) / kTileRows * kTileRows;
    if (rows > n_up) rows = n_up;
    double *V = (double *)fokl_scratch(ctx, fokl_ctx::B_PREDICT, (size_t)rows * n_draws * sizeof(double));
    if (!V) return FOKL_ENOMEM;

    const int leaves = fokl::pw_leaf_count(n_draws);
    const bool stage = n_draws <= kStageMaxDraws;
    const size_t smem = (size_t)kSummaryWarps * summary_warp_doubles(n_draws, leaves, stage) * sizeof(double);
    if (smem > ctx->smem_optin) FOKL_FAIL(ctx, FOKL_EINVAL, "predict_summary: n_draws too large");
    if (smem > 48 * 1024)
        FOKL_CUDA(ctx, cudaFuncSetAttribute(predict_summary_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            (int)smem));
    for (int64_t r0 = 0; r0 < n; r0 += rows) {
        const int64_t nr = n - r0 < rows ? n - r0 : rows;
        dim3 grid((unsigned)((nr + kTileRows - 1) / kTileRows), (unsigned)((n_draws + kTileDraws - 1) / kTileDraws));
        predict_tile_kernel<<<grid, kTileThreads, 0, ctx->stream>>>(X + r0, ld, nr, p, betas, n_draws, V);
        FOKL_LAUNCH_CHECK(ctx);
        const unsigned blocks = (unsigned)((nr + kSummaryWarps - 1) / kSummaryWarps);
        predict_summary_kernel<<<blocks, 32 * kSummaryWarps, smem, ctx->stream>>>(
            V, nr, n_draws, leaves, stage ? 1 : 0, rank_lo, rank_hi, mean_out + r0, ranks ? lo_out + r0 : nullptr,
            ranks ? hi_out + r0 : nullptr);
        FOKL_LAUNCH_CHECK(ctx);
    }
    return FOKL_OK;
}
