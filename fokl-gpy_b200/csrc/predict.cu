// predict.cu -- fokl_predict_summary: per-row mean and two order statistics of X @ betas' without writing the
// N x n_draws product to HBM (evaluate / coverage3 / bss_derivatives at training-set scale).
//
// Rows are processed in chunks whose rows x n_draws block of values (<= kChunkBytes) stays in L2:
//   1. predict_tile_kernel: register-tiled DFMA product of the chunk, v[i][d] = fma chain over j = 0 .. p-1 from 0.0,
//      the exact operation order of predict_draws_kernel (ctx.cu), so both entry points give the same bits;
//   2. predict_summary_kernel: one warp per row reads the row back (staged in shared memory when it is short), forms
//      numpy's pairwise mean, then selects the two ranks on order keys written over the row (predict_math.cuh).
//
// fokl_deriv_summary (bss_derivatives at training-set scale) runs the same two kernels on one row chunk of the
// derivative design columns, with a table of jobs (one per requested (input, order) pair) indexed by the grid.
#include "fokl_ctx.cuh"
#include "predict_math.cuh"

namespace {

constexpr int kTileRows = 128, kTileDraws = 64, kTileK = 16, kTileThreads = 256;
constexpr size_t kChunkBytes = 32u << 20;        // one chunk's values: well inside the 126 MB L2
constexpr int kMaxChunkRows = 1 << 16;
constexpr int kStageMaxDraws = 2048;             // rows up to this many draws are summarised from shared memory
constexpr int kSummaryWarps = 4;

// one (input, derivative order) pair of fokl_deriv_summary; offsets in doubles
struct TileJob {
    int64_t x_off;      // its first column in X
    int64_t b_off;      // its n_draws x p betas block
    int64_t v_off;      // its first value in V
    int64_t o_off;      // its mean in mean_out (the summary kernel)
    int p;              // its width
    int pad;
};

// thread (tx, ty) = (lane, warp) owns rows tx + 32 a (a < 4) and draws 8 ty + b (b < 8) of a 128 x 64 tile;
// V[i * ldv + d] = v[i][d].  With a job table, blockIdx.z selects the job, which moves X, betas and V and sets p.
__global__ void __launch_bounds__(kTileThreads)
predict_tile_kernel(const double *__restrict__ X, int64_t ld, int64_t n, int p, const double *__restrict__ betas,
                    int n_draws, double *__restrict__ V, int64_t ldv, const TileJob *__restrict__ jobs)
{
    if (jobs) {
        const TileJob jb = jobs[blockIdx.z];
        X += jb.x_off;
        betas += jb.b_off;
        V += jb.v_off;
        p = jb.p;
    }
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
            if (d < n_draws) V[i * ldv + d] = acc[a][b];
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

// mean_out[i * mean_ld] = np.mean(V[i * n_draws ..]).  With a job table, blockIdx.y selects the job, which moves V
// and mean_out (mean only).
__global__ void predict_summary_kernel(double *__restrict__ V, int64_t n, int n_draws, int leaves, int stage,
                                       int rank_lo, int rank_hi, double *__restrict__ mean_out,
                                       double *__restrict__ lo_out, double *__restrict__ hi_out,
                                       const TileJob *__restrict__ jobs, int64_t mean_ld)
{
    extern __shared__ double sm[];
    if (jobs) {
        const TileJob jb = jobs[blockIdx.y];
        V += jb.v_off;
        mean_out += jb.o_off;
    }
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
        if (lane == 0) mean_out[i * mean_ld] = fokl::pw_mean(fokl::pw_tree(n_draws, leaf), n_draws);
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
        predict_tile_kernel<<<grid, kTileThreads, 0, ctx->stream>>>(X + r0, ld, nr, p, betas, n_draws, V, n_draws,
                                                                    nullptr);
        FOKL_LAUNCH_CHECK(ctx);
        const unsigned blocks = (unsigned)((nr + kSummaryWarps - 1) / kSummaryWarps);
        predict_summary_kernel<<<blocks, 32 * kSummaryWarps, smem, ctx->stream>>>(
            V, nr, n_draws, leaves, stage ? 1 : 0, rank_lo, rank_hi, mean_out + r0, ranks ? lo_out + r0 : nullptr,
            ranks ? hi_out + r0 : nullptr, nullptr, 1);
        FOKL_LAUNCH_CHECK(ctx);
    }
    return FOKL_OK;
}

// Derivative summary of rows [r0, r0 + rows): the chunk's derivative columns (K1's derivative form, the code of
// fokl_basis_build_deriv) go to a (c x rows) workspace; then per pair the tile kernel forms its values and either writes
// them straight into out's [rows][m][2][n_draws] layout, or (mean_only) writes them to the L2-sized value scratch, from
// which the summary kernel writes their pairwise means into out's [rows][m][2] layout.  Slots no pair writes get 0.0.
extern "C" int fokl_deriv_summary(fokl_ctx *ctx, int kernel, const double *x, int64_t ldx, int m, int64_t r0,
                                  int64_t rows, const int16_t *terms, const uint8_t *deriv, const double *divisors,
                                  int c, const int64_t *pairs, int n_pairs, const double *betas, int n_draws,
                                  int mean_only, double *out)
{
    FOKL_CHECK_CTX(ctx);
    if (!x || !terms || !deriv || !divisors || !pairs || !betas || !out || m < 1 || r0 < 0 || rows < 1 ||
        ldx < r0 + rows || c < 0 || n_draws < 1 || (mean_only != 0 && mean_only != 1))
        FOKL_FAIL(ctx, FOKL_EINVAL, "deriv_summary: bad argument");
    if (kernel != FOKL_KERNEL_CUBIC && kernel != FOKL_KERNEL_BERNOULLI)
        FOKL_FAIL(ctx, FOKL_EINVAL, "deriv_summary: unknown kernel");
    if (n_pairs < 1 || n_pairs > 2 * (int64_t)m || n_pairs > 65535)
        FOKL_FAIL(ctx, FOKL_EINVAL, "deriv_summary: n_pairs must lie in [1, 2 m]");
    const int64_t slots = 2 * (int64_t)m, depth = mean_only ? 1 : n_draws;
    std::vector<char> taken((size_t)slots, 0);
    std::vector<TileJob> jobs;
    for (int k = 0; k < n_pairs; ++k) {
        const int64_t *pr = pairs + (size_t)k * 5;      // column offset, width, betas offset, input, order - 1
        const int64_t off = pr[0], w = pr[1], boff = pr[2], pm = pr[3], di = pr[4];
        if (off < 0 || w < 0 || off + w > c || boff < 0 || pm < 0 || pm >= m || di < 0 || di > 1 ||
            taken[(size_t)(2 * pm + di)]++)
            FOKL_FAIL(ctx, FOKL_EINVAL, "deriv_summary: bad pair (column range, betas offset or a repeated (m, di))");
        if (w == 0) continue;                            // an empty FMA chain: 0.0, as the zero fill gives
        TileJob jb;
        jb.x_off = off * rows;
        jb.b_off = boff;
        jb.v_off = mean_only ? (int64_t)jobs.size() : (2 * pm + di) * n_draws;    // mean_only: times the rows below
        jb.o_off = 2 * pm + di;
        jb.p = (int)w;
        jb.pad = 0;
        jobs.push_back(jb);
    }
    const int leaves = fokl::pw_leaf_count(n_draws);
    const bool stage = n_draws <= kStageMaxDraws;
    const size_t smem = (size_t)kSummaryWarps * summary_warp_doubles(n_draws, leaves, stage) * sizeof(double);
    if (mean_only && smem > ctx->smem_optin) FOKL_FAIL(ctx, FOKL_EINVAL, "deriv_summary: n_draws too large");
    int rc = fokl_bind_device(ctx);
    if (rc) return rc;

    const int nj = (int)jobs.size();
    // mean_only: rows per pass so that the passes' values of every job stay in L2 together
    int64_t sub = rows;
    if (mean_only && nj) {
        sub = (int64_t)(kChunkBytes / ((size_t)nj * n_draws * sizeof(double))) / kTileRows * kTileRows;
        if (sub < kTileRows) sub = kTileRows;
        const int64_t rows_up = (rows + kTileRows - 1) / kTileRows * kTileRows;
        if (sub > rows_up) sub = rows_up;
        for (TileJob &jb : jobs) jb.v_off *= sub * n_draws;
    }
    const size_t jobs_bytes = ((size_t)nj * sizeof(TileJob) + 255) & ~(size_t)255;
    char *ws = (char *)fokl_scratch(ctx, fokl_ctx::B_DERIV, jobs_bytes + (size_t)c * rows * sizeof(double));
    if (!ws) return FOKL_ENOMEM;
    TileJob *djobs = reinterpret_cast<TileJob *>(ws);
    double *W = reinterpret_cast<double *>(ws + jobs_bytes);
    double *V = nullptr;
    if (mean_only && nj) {
        V = (double *)fokl_scratch(ctx, fokl_ctx::B_PREDICT, (size_t)nj * sub * n_draws * sizeof(double));
        if (!V) return FOKL_ENOMEM;
    }
    // the K1 launches validate the term list before they enqueue anything, so a rejected one leaves `out` untouched
    rc = fokl_basis_build_deriv(ctx, kernel, x + r0, rows, ldx, m, terms, deriv, divisors, c, W, rows);
    if (rc) return rc;
    if (nj) FOKL_CUDA(ctx, cudaMemcpyAsync(djobs, jobs.data(), (size_t)nj * sizeof(TileJob), cudaMemcpyHostToDevice,
                                           ctx->stream));
    if (nj < slots)
        FOKL_CUDA(ctx, cudaMemsetAsync(out, 0, (size_t)rows * slots * depth * sizeof(double), ctx->stream));
    if (!nj) return FOKL_OK;
    const unsigned gy = (unsigned)((n_draws + kTileDraws - 1) / kTileDraws);
    if (!mean_only) {
        dim3 grid((unsigned)((rows + kTileRows - 1) / kTileRows), gy, (unsigned)nj);
        predict_tile_kernel<<<grid, kTileThreads, 0, ctx->stream>>>(W, rows, rows, 0, betas, n_draws, out,
                                                                    slots * n_draws, djobs);
        FOKL_LAUNCH_CHECK(ctx);
        return FOKL_OK;
    }
    if (smem > 48 * 1024)
        FOKL_CUDA(ctx, cudaFuncSetAttribute(predict_summary_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            (int)smem));
    for (int64_t s0 = 0; s0 < rows; s0 += sub) {
        const int64_t nr = rows - s0 < sub ? rows - s0 : sub;
        dim3 grid((unsigned)((nr + kTileRows - 1) / kTileRows), gy, (unsigned)nj);
        predict_tile_kernel<<<grid, kTileThreads, 0, ctx->stream>>>(W + s0, rows, nr, 0, betas, n_draws, V, n_draws,
                                                                    djobs);
        FOKL_LAUNCH_CHECK(ctx);
        dim3 sgrid((unsigned)((nr + kSummaryWarps - 1) / kSummaryWarps), (unsigned)nj);
        predict_summary_kernel<<<sgrid, 32 * kSummaryWarps, smem, ctx->stream>>>(
            V, nr, n_draws, leaves, stage ? 1 : 0, -1, -1, out + s0 * slots, nullptr, nullptr, djobs, slots);
        FOKL_LAUNCH_CHECK(ctx);
    }
    return FOKL_OK;
}
