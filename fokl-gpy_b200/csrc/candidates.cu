// candidates.cu -- K3/K4: per-candidate spectral factorisation, betahat, BIC, eigenbasis Gibbs chain,
// betas = Gamma Q' and the column statistics the forward-selection loop reads (sm_100a).
//
// One CTA per candidate model.  Replaces, per `gibbs` invocation of the reference
// (src/FoKL/FoKLRoutines.py): eigh FR:1499, betahat FR:1502-1504, draw loop FR:1519-1548,
// BIC FR:1551-1554, and the reductions over the draws at FR:1656-1658, 1671.
// The numerical core lives in cand_math.cuh (shared with the host emulation used by the CPU tests).
#include "fokl_ctx.cuh"
#include <stdlib.h>
#include "cand_math.cuh"
#include "eigbig.cuh"
#include "killbig.cuh"
#include <cooperative_groups.h>
#include <algorithm>
#include <queue>
#include <math.h>
#include <string.h>
#include <vector>

namespace {

using fokl::CandConst;
using fokl::Team;

constexpr int kEigThreads = 256;
constexpr int kChainThreads = 256;      // upper bound; launched with ~p/2 threads (two elements per thread in registers)
constexpr int kSmemHeaderDoubles = 64;   // reduction scratch (2*3*8) + flag

struct CandMeta {
    int32_t p;
    int32_t set_off;     // into col_sets
    int32_t chain_idx;   // -1: no chain
    int32_t pad;
    int64_t vec_off;     // sum of p of previous candidates
    int64_t mat_off;     // sum of p^2 of previous candidates
    int64_t wv_off;      // offset (doubles) of this candidate's W|V pair in the global workspace
    int64_t gam_off;     // sum of p of previous *chain* candidates
    uint64_t stream_id;
};

struct EigParams {
    const double *G;
    int64_t ldg;
    const double *Xty;
    const int32_t *col_sets;
    const CandMeta *meta;
    CandConst k;
    double *wv;          // global W|V workspace
    double *lam_raw, *scratch, *ct;   // packed by vec_off
    int32_t *perm;
    double *lamb, *Q, *betahat, *ev;
    int32_t *info;
    int smem_doubles;    // dynamic shared memory available for W|V (after the header)
    int only_flagged;
};

__device__ __forceinline__ Team make_team()
{
    Team t;
    t.tid = threadIdx.x; t.nthr = blockDim.x;
    t.lane = threadIdx.x & 31; t.nlane = 32;
    t.warp = threadIdx.x >> 5; t.nwarp = blockDim.x >> 5;
    return t;
}

__global__ void __launch_bounds__(kEigThreads) cand_eig_kernel(const EigParams P)
{
    extern __shared__ __align__(16) double sh[];
    const Team t = make_team();
    const CandMeta m = P.meta[blockIdx.x];
    // fallback path: only candidates whose Gram failed the Cholesky of cand_chol_kernel (info bit 1) or that are too
    // large for the cluster kernel (info bit 2)
    if (P.only_flagged && !(P.info[blockIdx.x] & 6)) return;
    const int p = m.p;
    const int32_t *idx = P.col_sets + m.set_off;
    double *red = sh;
    volatile int *flag = reinterpret_cast<volatile int *>(sh + 56);
    const bool in_smem = (2 * p * p <= P.smem_doubles);
    double *W = in_smem ? (sh + kSmemHeaderDoubles) : (P.wv + m.wv_off);
    double *V = W + (size_t)p * p;

    for (int e = t.tid; e < p * p; e += t.nthr) {
        int col = e / p, row = e - col * p;
        W[e] = P.G[(int64_t)idx[row] * P.ldg + idx[col]];
    }
    t.sync();
    const double tol = 2.220446049250313e-16 * (2.0 * sqrt((double)p) + 6.0);
    int sweeps = fokl::jacobi_eigh(t, W, V, p, p, 40, tol, flag);
    double *lamb = P.lamb + m.vec_off;
    double *Q = P.Q + m.mat_off;
    fokl::eig_finish(t, W, V, p, p, P.lam_raw + m.vec_off, P.perm + m.vec_off, lamb, Q);
    double ev = fokl::ols_and_bic(t, P.G, P.ldg, P.Xty, idx, p, lamb, Q, P.k, P.ct + m.vec_off,
                                  P.betahat + m.vec_off, P.scratch + m.vec_off, red);
    if (t.tid == 0) {
        P.ev[blockIdx.x] = ev;
        P.info[blockIdx.x] = (P.info[blockIdx.x] & 6) | (sweeps << 8);
    }
}

// ---- Cholesky factor of every candidate's Gram (pre-pass of the cluster eigensolver) --------------------------------
// L is written to the candidate's Q slot (p x p, column-major, zeros above the diagonal); the cluster kernel reads
// it and later overwrites the slot with the eigenvectors.  info bit 1 (value 2): Gram not positive definite.
constexpr int kCholThreads = 1024;

struct CholParams {
    const double *G;
    int64_t ldg;
    const int32_t *col_sets;
    const CandMeta *meta;
    double *Q;
    int32_t *info;
    int smem_doubles;
};

__global__ void __launch_bounds__(kCholThreads) cand_chol_kernel(const CholParams P)
{
    extern __shared__ __align__(16) double sh[];
    const Team t = make_team();
    const CandMeta m = P.meta[blockIdx.x];
    if (m.pad) {                       // too large for the cluster eigensolver: blocked solver (2) or fallback kernel (1)
        if (t.tid == 0) P.info[blockIdx.x] = (m.pad == 2) ? 8 : 4;
        return;
    }
    const int p = m.p;
    const int32_t *idx = P.col_sets + m.set_off;
    double *Lg = P.Q + m.mat_off;
    const bool in_smem = ((int64_t)p * (p + 1) / 2 <= P.smem_doubles);
    bool ok;
    if (in_smem) {
        // packed lower triangle in shared memory; written out in the square form the eigensolver reads
        double *L = sh;
        for (int col = t.warp; col < p; col += t.nwarp) {
            double *Lc = L + fokl::chol_col(col, p) - col;
            const int64_t gcol = (int64_t)idx[col] * P.ldg;
            for (int row = col + t.lane; row < p; row += t.nlane) Lc[row] = P.G[gcol + idx[row]];    // G is symmetric
        }
        t.sync();
        ok = fokl::cholesky_lower_packed(t, L, p);
        for (int col = t.warp; col < p; col += t.nwarp) {
            const double *Lc = L + fokl::chol_col(col, p) - col;
            for (int row = t.lane; row < p; row += t.nlane) Lg[(int64_t)col * p + row] = row >= col ? Lc[row] : 0.0;
        }
    } else {
        for (int e = t.tid; e < p * p; e += t.nthr) {
            int col = e / p, row = e - col * p;
            Lg[e] = (row >= col) ? P.G[(int64_t)idx[row] * P.ldg + idx[col]] : 0.0;
        }
        t.sync();
        ok = fokl::cholesky_lower(t, Lg, p);
    }
    if (t.tid == 0) P.info[blockIdx.x] = ok ? 0 : 2;
}

// ---- cluster eigensolver: one-sided Jacobi on the Cholesky factor, columns distributed over a CTA cluster -------------
// A cluster of cs CTAs holds the n = 2 cs m columns of W (n >= p, zero columns pad) in shared memory, m "top" and m
// "bottom" columns per CTA; the pair (top[k], bottom[k]) is rotated by one warp.  After every round the columns move
// one position along the chess-tournament ring (top row to the right, bottom row to the left, top[0] of CTA 0
// fixed): inside a CTA that is an index rotation, and only the two columns that cross a CTA boundary travel, pushed
// into the neighbour's staging buffer through distributed shared memory, one cluster barrier per round.  n - 1 rounds
// visit every pair once (a sweep); sweeps repeat until no pair needed a rotation.
constexpr int kEigJThreads = 512;       // <= 16 column pairs per CTA in flight, 128 registers per thread
constexpr int kEigJMaxNV = 11;          // double2 per lane per column: p <= 64 * 11 = 704
constexpr int kEigJMaxCluster = 16;
constexpr int kEigJHeaderDoubles = 256;   // team_sum3 scratch: 2 * 3 * 32 warps

struct EigJParams {
    const double *G;
    int64_t ldg;
    const double *Xty;
    const int32_t *col_sets;
    const CandMeta *meta;
    const int32_t *list;     // candidates of this launch (one cluster each)
    CandConst k;
    double *lam_raw;         // per candidate p + 64 doubles at vec_off + 64 * cand
    double *scratch, *ct;    // packed by vec_off
    double *lamb, *Q, *betahat, *ev;
    int32_t *info;
};

__host__ __device__ inline int eigj_padded_n(int p, int cs)
{
    if (cs == 1) return (p + 1) & ~1;
    const int unit = 2 * cs;
    int n = ((p + unit - 1) / unit) * unit;
    if (n < 4 * cs) n = 4 * cs;        // at least two pair slots per CTA (the ring needs a rotating top slot in CTA 0)
    return n;
}
__host__ __device__ inline int eigj_ld(int p) { return (p + 1) & ~1; }   // even: columns are moved as double2
__host__ __device__ inline int eigj_slots(int p, int cs)                // column buffers per CTA
{
    const int n = eigj_padded_n(p, cs);
    return cs == 1 ? n : 2 * (n / (2 * cs) + 1);                         // cs > 1: m + 1 top and m + 1 bottom (one spare each)
}
__host__ __device__ inline size_t eigj_smem_bytes(int p, int cs)
{
    return (size_t)eigj_slots(p, cs) * (eigj_ld(p) + 1) * sizeof(double) + (size_t)(2 * kEigJMaxCluster + 8) * sizeof(int) +
           kEigJHeaderDoubles * sizeof(double);
}
__host__ __device__ inline int eigj_threads(int p, int cs)
{
    const int pairs = eigj_padded_n(p, cs) / (2 * cs);
    int w = pairs < 1 ? 1 : (pairs > kEigJThreads / 32 ? kEigJThreads / 32 : pairs);
    if (w < 4) w = 4;                                                      // ols_and_bic / ranking like a few warps
    return 32 * w;
}

// Physical slot of a logical position (cluster layout, cs > 1) from the running round counters rt = round mod (m+1),
// r0 = round mod m.  Every row keeps one spare slot: the column that leaves a CTA is written by the rotating warp
// straight into the *spare* slot of its destination row (possibly in the neighbouring CTA, through distributed shared
// memory), and the slot it vacates is the next spare.
struct RingLayout {
    int m, cr, rt, r0;
    __device__ __forceinline__ static int wrap_neg(int x, int mod) { return x < 0 ? x + mod : x; }
    __device__ __forceinline__ static int wrap_pos(int x, int mod) { return x >= mod ? x - mod : x; }
    __device__ __forceinline__ int top(int k) const
    {
        if (cr == 0) return k == 0 ? m : wrap_neg(k - 1 - r0, m);         // CTA 0: logical 0 is the fixed player (slot m)
        return wrap_neg(k - rt, m + 1);
    }
    __device__ __forceinline__ int top_spare(int c) const { return c == 0 ? wrap_neg(m - 1 - r0, m) : wrap_neg(m - rt, m + 1); }
    __device__ __forceinline__ int bot(int k) const { return (m + 1) + wrap_pos(k + rt, m + 1); }
    __device__ __forceinline__ int bot_spare() const { return (m + 1) + wrap_pos(m + rt, m + 1); }
    __device__ __forceinline__ void advance()
    {
        rt = (rt + 1 == m + 1) ? 0 : rt + 1;
        r0 = (r0 + 1 == m) ? 0 : r0 + 1;
    }
};

// One warp orthogonalises a pair of columns.  Both columns are loaded once into registers (NV double2 per lane), the
// three inner products, the rotation and the stores work from there; a column whose destination differs from its
// source (it leaves this CTA's row) is written there whether or not a rotation was needed.
// Returns 0 = no rotation needed, 1 = rotated a pair that was already orthogonal to tol_small (relative cosine), 2 = rotated.
template <int NV>
__device__ __forceinline__ int pair_rotate_reg(const double *a, const double *b, double *a_out, double *b_out, int nv2,
                                               double tol, double tol_small, int lane)
{
    const double2 *a2 = reinterpret_cast<const double2 *>(a), *b2 = reinterpret_cast<const double2 *>(b);
    double2 av[NV], bv[NV];
#pragma unroll
    for (int q = 0; q < NV; ++q) {
        const int i = lane + 32 * q;
        if (i < nv2) { av[q] = a2[i]; bv[q] = b2[i]; }
        else { av[q] = make_double2(0.0, 0.0); bv[q] = make_double2(0.0, 0.0); }
    }
    double al = 0.0, be = 0.0, ga = 0.0;
#pragma unroll
    for (int q = 0; q < NV; ++q) {
        al = fma(av[q].x, av[q].x, al); al = fma(av[q].y, av[q].y, al);
        be = fma(bv[q].x, bv[q].x, be); be = fma(bv[q].y, bv[q].y, be);
        ga = fma(av[q].x, bv[q].x, ga); ga = fma(av[q].y, bv[q].y, ga);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        al += __shfl_xor_sync(0xffffffffu, al, o);
        be += __shfl_xor_sync(0xffffffffu, be, o);
        ga += __shfl_xor_sync(0xffffffffu, ga, o);
    }
    const bool rot = ga * ga > (tol * tol) * (al * be);          // |ga| > tol sqrt(al be) without the square root
    double2 *ao = reinterpret_cast<double2 *>(a_out), *bo = reinterpret_cast<double2 *>(b_out);
    if (rot) {
        // Rotation that annihilates ga, from the double angle: with d = |b|^2 - |a|^2 and r = sqrt(d^2 + 4 ga^2),
        // cos 2t = |d| / r, sin 2t = 2 ga sign(d) / r; c = sqrt((1 + cos 2t) / 2), s = sin 2t / (2 c).  Two dependent
        // rsqrt and a few multiplies (no division, no sqrt); c^2 + s^2 = 1 to rounding.
        const double d = be - al;
        const double rinv = fokl::rsqrt_pos(fma(d, d, 4.0 * ga * ga));      // branch-free MUFU seed + two Newton steps
        const double u = fma(0.5 * fabs(d), rinv, 0.5);             // (1 + cos 2t) / 2  in [1/2, 1]
        const double ic = fokl::rsqrt_pos(u);
        const double c = u * ic;
        const double s = copysign(ga * rinv, ga * d) * ic;          // d == 0 -> sign(ga): the 45 degree rotation
#pragma unroll
        for (int q = 0; q < NV; ++q) {
            const int i = lane + 32 * q;
            if (i < nv2) {
                ao[i] = make_double2(c * av[q].x - s * bv[q].x, c * av[q].y - s * bv[q].y);
                bo[i] = make_double2(s * av[q].x + c * bv[q].x, s * av[q].y + c * bv[q].y);
            }
        }
    } else {
        if (a_out != a) {
#pragma unroll
            for (int q = 0; q < NV; ++q) {
                const int i = lane + 32 * q;
                if (i < nv2) ao[i] = av[q];
            }
        }
        if (b_out != b) {
#pragma unroll
            for (int q = 0; q < NV; ++q) {
                const int i = lane + 32 * q;
                if (i < nv2) bo[i] = bv[q];
            }
        }
    }
    return rot ? (ga * ga > (tol_small * tol_small) * (al * be) ? 2 : 1) : 0;
}

struct EigJShared {
    double *cols, *tags;      // column buffers (ld doubles each) and the original column index of each (-1 = padding)
    int *flags, *any_flag;
};

// All sweeps of one candidate.  Returns the number of sweeps; `ring` is left at the final round.
template <int NV>
__device__ int eigj_sweeps(cooperative_groups::cluster_group &cluster, const Team &t, const EigJShared &S, RingLayout &ring,
                           int cs, int cr, int n, int m, int ld, double tol)
{
    const double tol_small = sqrt(tol / (4.0 * (double)(n > 1 ? n : 1)));
    const int nv2 = ld / 2, h = n / 2;
    int sweeps = 0;
    for (; sweeps < 40; ++sweeps) {
        if (cs == 1) {
            // classic round-robin on static columns: pair k of round r is ((r + k) mod (n-1), (r - k) mod (n-1)), n-1 fixed
            const int nm1 = n - 1;
            for (int r = 0; r < nm1; ++r) {
                for (int k = t.warp; k < h; k += t.nwarp) {
                    int i, j;
                    if (k == 0) { i = nm1; j = r; }
                    else { i = RingLayout::wrap_pos(r + k, nm1); j = RingLayout::wrap_pos(r - k + nm1, nm1); }
                    double *a = S.cols + (size_t)i * ld, *b = S.cols + (size_t)j * ld;
                    const int lvl = pair_rotate_reg<NV>(a, b, a, b, nv2, tol, tol_small, t.lane);
                    if (lvl && t.lane == 0) atomicMax(S.any_flag, lvl);
                }
                __syncthreads();
            }
        } else {
            for (int r = 0; r < n - 1; ++r) {
                for (int k = t.warp; k < m; k += t.nwarp) {
                    const int sa = ring.top(k), sb = ring.bot(k);
                    double *a = S.cols + (size_t)sa * ld, *b = S.cols + (size_t)sb * ld;
                    double *a_out = a, *b_out = b;
                    if (k == m - 1) {            // top column leaves to the right (last CTA: into its own bottom row)
                        const int dst = (cr < cs - 1) ? ring.top_spare(cr + 1) : ring.bot_spare();
                        double *dcol = S.cols + (size_t)dst * ld, *dtag = S.tags + dst;
                        if (cr < cs - 1) { dcol = cluster.map_shared_rank(dcol, cr + 1); dtag = cluster.map_shared_rank(dtag, cr + 1); }
                        a_out = dcol;
                        if (t.lane == 0) *dtag = S.tags[sa];
                    }
                    if (k == 0) {                // bottom column leaves to the left (CTA 0: into its own top row)
                        const int dst = (cr > 0) ? ring.bot_spare() : ring.top_spare(0);
                        double *dcol = S.cols + (size_t)dst * ld, *dtag = S.tags + dst;
                        if (cr > 0) { dcol = cluster.map_shared_rank(dcol, cr - 1); dtag = cluster.map_shared_rank(dtag, cr - 1); }
                        b_out = dcol;
                        if (t.lane == 0) *dtag = S.tags[sb];
                    }
                    const int lvl = pair_rotate_reg<NV>(a, b, a_out, b_out, nv2, tol, tol_small, t.lane);
                    if (lvl && t.lane == 0) atomicMax(S.any_flag, lvl);
                }
                if (r == n - 2) {
                    // end of the sweep: tell every CTA of the cluster whether this one rotated anything
                    __syncthreads();
                    if (t.tid < cs) {
                        int *remote = cluster.map_shared_rank(S.flags, t.tid);
                        remote[(sweeps & 1) * kEigJMaxCluster + cr] = S.any_flag[0];
                    }
                }
                cluster.sync();
                ring.advance();
            }
        }
        int any;
        if (cs == 1) {
            any = S.any_flag[0];
        } else {
            any = 0;
            for (int c = 0; c < cs; ++c) any = max(any, S.flags[(sweeps & 1) * kEigJMaxCluster + c]);
        }
        __syncthreads();
        if (t.tid == 0) S.any_flag[0] = 0;
        __syncthreads();
        // Quadratic convergence: a sweep whose rotated pairs were all orthogonal to tol_small already leaves cosines of
        // order tol_small^2 per later rotation of the same column, p tol_small^2 <= tol / 4 in all -- the sweep that would
        // only confirm it is not run.
        if (any <= 1) { ++sweeps; break; }
    }
    return sweeps;
}

__global__ void __launch_bounds__(kEigJThreads, 1) cand_eigj_kernel(const EigJParams P)
{
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const int cs = (int)cluster.num_blocks(), cr = (int)cluster.block_rank();
    const int cand = P.list[blockIdx.x / cs];
    const CandMeta cm = P.meta[cand];
    if (P.info[cand] & 6) return;                 // whole cluster takes the same branch: the fallback kernel does it
    extern __shared__ __align__(16) double sh[];
    const Team t = make_team();
    const int p = cm.p;
    const int n = eigj_padded_n(p, cs), ld = eigj_ld(p), slots = eigj_slots(p, cs);
    const int m = n / (2 * cs), h = n / 2;
    double *red = sh;                                         // reductions of ols_and_bic
    EigJShared S;
    S.cols = sh + kEigJHeaderDoubles;
    S.tags = S.cols + (size_t)slots * ld;
    S.flags = reinterpret_cast<int *>(S.tags + slots);        // [2][kEigJMaxCluster]
    S.any_flag = S.flags + 2 * kEigJMaxCluster;               // [0] this CTA rotated something in this sweep
    const double *Lg = P.Q + cm.mat_off;
    const double tol = 2.220446049250313e-16 * (2.0 * sqrt((double)p) + 6.0);
    RingLayout ring;
    ring.m = m; ring.cr = cr; ring.rt = 0; ring.r0 = 0;

    // ---- load the Cholesky factor: columns >= p are zero padding (tag -1) ----------------------------------------------
    // cs == 1: column g in slot g.  cs > 1: top logical k <- column cr*m + k, bottom logical k <- column h + cr*m + k.
    const int n_local = (cs == 1) ? n : 2 * m;
    for (int k = t.warp; k < n_local; k += t.nwarp) {
        int g, slot;
        if (cs == 1) { g = k; slot = k; }
        else if (k < m) { g = cr * m + k; slot = ring.top(k); }
        else { g = h + cr * m + (k - m); slot = ring.bot(k - m); }
        double *dst = S.cols + (size_t)slot * ld;
        for (int e = t.lane; e < ld; e += 32) dst[e] = (e < p && g < p) ? Lg[(size_t)g * p + e] : 0.0;
        if (t.lane == 0) S.tags[slot] = (g < p) ? (double)g : -1.0;
    }
    if (t.tid < 2 * kEigJMaxCluster) S.flags[t.tid] = 0;
    if (t.tid == 0) S.any_flag[0] = 0;
    __syncthreads();
    if (cs > 1) cluster.sync();      // every CTA is resident and initialised before anybody writes into a neighbour

    int sweeps;
    const int nv = (ld / 2 + 31) / 32;
    switch (nv) {
    case 1: sweeps = eigj_sweeps<1>(cluster, t, S, ring, cs, cr, n, m, ld, tol); break;
    case 2: sweeps = eigj_sweeps<2>(cluster, t, S, ring, cs, cr, n, m, ld, tol); break;
    case 3: sweeps = eigj_sweeps<3>(cluster, t, S, ring, cs, cr, n, m, ld, tol); break;
    case 4: sweeps = eigj_sweeps<4>(cluster, t, S, ring, cs, cr, n, m, ld, tol); break;
    case 5: case 6: sweeps = eigj_sweeps<6>(cluster, t, S, ring, cs, cr, n, m, ld, tol); break;
    case 7: case 8: sweeps = eigj_sweeps<8>(cluster, t, S, ring, cs, cr, n, m, ld, tol); break;
    default: sweeps = eigj_sweeps<kEigJMaxNV>(cluster, t, S, ring, cs, cr, n, m, ld, tol); break;
    }

    // ---- eigenvalues = squared column norms; rank them across the cluster; eigenvectors = normalised columns ------------
    double *lam_all = P.lam_raw + cm.vec_off + 64 * (int64_t)cand;     // n entries, indexed cr * n_local + k
    auto live_slot = [&](int k) { return cs == 1 ? k : (k < m ? ring.top(k) : ring.bot(k - m)); };
    for (int k = t.warp; k < n_local; k += t.nwarp) {
        const int slot = live_slot(k);
        const double *w = S.cols + (size_t)slot * ld;
        double s = 0.0;
        for (int e = t.lane; e < p; e += 32) s += w[e] * w[e];
        s = fokl::warp_sum1(t, s);
        if (t.lane == 0) lam_all[cr * n_local + k] = (S.tags[slot] < 0.0) ? -1.0 : s;    // padding columns: marked, not ranked
    }
    __threadfence();
    if (cs > 1) cluster.sync(); else __syncthreads();
    double *lamb = P.lamb + cm.vec_off;
    double *Q = P.Q + cm.mat_off;
    for (int k = t.warp; k < n_local; k += t.nwarp) {
        const int slot = live_slot(k);
        const double *w = S.cols + (size_t)slot * ld;
        if (S.tags[slot] < 0.0) continue;
        const int gme = cr * n_local + k;
        const double lj = lam_all[gme];
        int rank = 0;
        for (int g = t.lane; g < n; g += 32) {
            const double li = lam_all[g];
            if (li >= 0.0 && (li < lj || (li == lj && g < gme))) ++rank;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) rank += __shfl_xor_sync(0xffffffffu, rank, o);
        const double inv = 1.0 / sqrt(lj);
        for (int e = t.lane; e < p; e += 32) Q[(size_t)rank * p + e] = w[e] * inv;
        if (t.lane == 0) lamb[rank] = lj;
    }
    __threadfence();
    if (cs > 1) cluster.sync(); else __syncthreads();
    if (cr != 0) return;
    const int32_t *idx = P.col_sets + cm.set_off;
    double ev = fokl::ols_and_bic(t, P.G, P.ldg, P.Xty, idx, p, lamb, Q, P.k, P.ct + cm.vec_off, P.betahat + cm.vec_off,
                                  P.scratch + cm.vec_off, red);
    if (t.tid == 0) {
        P.ev[cand] = ev;
        P.info[cand] = (P.info[cand] & 6) | (sweeps << 8);
    }
}

// betahat + BIC of the candidates factorised by the blocked eigensolver (eigbig.cuh), one CTA each
struct OlsParams {
    const double *G;
    int64_t ldg;
    const double *Xty;
    const int32_t *col_sets;
    const CandMeta *meta;
    const int32_t *list;
    CandConst k;
    double *scratch, *ct, *lamb, *Q, *betahat, *ev;
    int32_t *info;
    const int32_t *sweeps;
};

__global__ void __launch_bounds__(1024) cand_ols_kernel(const OlsParams P)
{
    __shared__ double red[2 * 3 * 32];
    const Team t = make_team();
    const int cand = P.list[blockIdx.x];
    const int st = P.sweeps[cand];
    if (st < 0) {                      // Gram not positive definite: the two-matrix fallback kernel takes the model
        if (t.tid == 0) P.info[cand] = 2;
        return;
    }
    const CandMeta cm = P.meta[cand];
    const int32_t *idx = P.col_sets + cm.set_off;
    double ev = fokl::ols_and_bic(t, P.G, P.ldg, P.Xty, idx, cm.p, P.lamb + cm.vec_off, P.Q + cm.mat_off, P.k,
                                  P.ct + cm.vec_off, P.betahat + cm.vec_off, P.scratch + cm.vec_off, red);
    if (t.tid == 0) {
        P.ev[cand] = ev;
        P.info[cand] = (st << 8) | (st >= eigb::kMaxSweeps ? 16 : 0);
    }
}

struct ChainParams {
    const CandMeta *meta;
    const int32_t *chain_list;
    CandConst k;
    const double *lamb, *ct;
    int rng_mode;
    uint64_t seed;
    const double *variates;   // injected: caller's table (packed over all candidates); philox: d_var (packed over chains)
    double *var_philox;       // philox: table filled by cand_variates_kernel
    const double *sign_fix;
    double *gam, *sigs, *taus;
    int32_t *info;
};

// offset (doubles) of the D x (p + 2) variate table of chain `slot` = candidate c
__device__ __forceinline__ int64_t variates_offset(const ChainParams &P, const CandMeta &m, int c)
{
    return (P.rng_mode == FOKL_RNG_INJECTED) ? (int64_t)P.k.draws * (m.vec_off + 2 * (int64_t)c)
                                             : (int64_t)P.k.draws * (m.gam_off + 2 * (int64_t)m.chain_idx);
}

// Philox table of every chain: one thread per variate (grid.y = chain), so the RNG (log / cos / rejection loops)
// is off the sequential critical path of the draw loop.
__global__ void __launch_bounds__(256) cand_variates_kernel(const ChainParams P)
{
    const int c = P.chain_list[blockIdx.y];
    const CandMeta m = P.meta[c];
    const int p = m.p, w = p + 2;
    const int64_t total = (int64_t)P.k.draws * w;
    fokl::Philox g;
    g.k0 = (uint32_t)P.seed;
    g.k1 = (uint32_t)(P.seed >> 32);
    const uint32_t slo = (uint32_t)m.stream_id, shi = (uint32_t)(m.stream_id >> 32) & 0x7fffffffu;
    const double astar = fokl::chain_astar(P.k, p), atau_star = fokl::chain_atau_star(P.k, p);
    double *out = P.var_philox + variates_offset(P, m, c);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int d = (int)(i / w), e = (int)(i - (int64_t)d * w);
        out[i] = fokl::philox_variate(g, slo, shi, d, e, p, astar, atau_star);
    }
}

__global__ void __launch_bounds__(kChainThreads) cand_chain_kernel(const ChainParams P)
{
    __shared__ double red[2 * 3 * (kChainThreads / 32)];
    const Team t = make_team();
    const int c = P.chain_list[blockIdx.x];
    const CandMeta m = P.meta[c];
    const int p = m.p;
    const int D = P.k.draws;
    const double *var = (P.rng_mode == FOKL_RNG_INJECTED ? P.variates : P.var_philox) + variates_offset(P, m, c);
    const double *sf = P.sign_fix ? P.sign_fix + m.vec_off : nullptr;
    int bad = fokl::gibbs_chain(t, p, P.lamb + m.vec_off, P.ct + m.vec_off, P.k, var, sf, P.gam + (int64_t)D * m.gam_off,
                                P.sigs + (int64_t)D * c, P.taus + (int64_t)D * c, red, P.rng_mode == FOKL_RNG_PHILOX);
    if (t.tid == 0 && bad) atomicOr(P.info + c, 1);
}

// One warp per chain, E elements per lane in registers (models of up to 32 E columns).
template <int E>
__global__ void __launch_bounds__(32) cand_chain_warp_kernel(const ChainParams P)
{
    const int c = P.chain_list[blockIdx.x];
    const CandMeta m = P.meta[c];
    const int D = P.k.draws;
    const double *var = (P.rng_mode == FOKL_RNG_INJECTED ? P.variates : P.var_philox) + variates_offset(P, m, c);
    const double *sf = P.sign_fix ? P.sign_fix + m.vec_off : nullptr;
    int bad = fokl::gibbs_chain_warp<E>(threadIdx.x, m.p, P.lamb + m.vec_off, P.ct + m.vec_off, P.k, var, sf,
                                        P.gam + (int64_t)D * m.gam_off, P.sigs + (int64_t)D * c, P.taus + (int64_t)D * c,
                                        P.rng_mode == FOKL_RNG_PHILOX);
    if (threadIdx.x == 0 && bad) atomicOr(P.info + c, 1);
}

// betas[k][i] = sum_r Gamma[k][r] * Q[r*p + i]   (FR:1528 in the eigenbasis: beta = Q gamma)
struct BetasParams {
    const CandMeta *meta;
    const int32_t *chain_list;
    const double *gam, *Q;
    double *betas;          // packed at D * vec_off
    int D, tiles_i;
};

__global__ void __launch_bounds__(256) cand_betas_kernel(const BetasParams P)
{
    __shared__ double As[16][64 + 1];
    __shared__ double Bs[16][64];
    const int c = P.chain_list[blockIdx.y];
    const CandMeta m = P.meta[c];
    const int p = m.p;
    const int ti = blockIdx.x % P.tiles_i, tk = blockIdx.x / P.tiles_i;
    const int i0 = ti * 64, k0 = tk * 64;
    if (i0 >= p) return;
    const double *A = P.gam + (int64_t)P.D * m.gam_off;
    const double *B = P.Q + m.mat_off;
    double *C = P.betas + (int64_t)P.D * m.vec_off;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    double acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
    for (int r0 = 0; r0 < p; r0 += 16) {
        {
            int row = tid >> 2, rr = (tid & 3) * 4;
            int k = k0 + row;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                int r = r0 + rr + q;
                As[rr + q][row] = (k < P.D && r < p) ? A[(int64_t)k * p + r] : 0.0;
            }
            int br = tid >> 4, ii = (tid & 15) * 4;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                int r = r0 + br, i = i0 + ii + q;
                Bs[br][ii + q] = (r < p && i < p) ? B[(int64_t)r * p + i] : 0.0;
            }
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < 16; ++r) {
            double a[4], b[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) { a[q] = As[r][ty * 4 + q]; b[q] = Bs[r][tx * 4 + q]; }
#pragma unroll
            for (int x = 0; x < 4; ++x)
#pragma unroll
                for (int z = 0; z < 4; ++z) acc[x][z] += a[x] * b[z];
        }
        __syncthreads();
    }
#pragma unroll
    for (int x = 0; x < 4; ++x) {
        int k = k0 + ty * 4 + x;
        if (k >= P.D) continue;
#pragma unroll
        for (int z = 0; z < 4; ++z) {
            int i = i0 + tx * 4 + z;
            if (i < p) C[(int64_t)k * p + i] = acc[x][z];
        }
    }
}

struct StatsParams {
    const CandMeta *meta;
    const int32_t *chain_list;
    const double *betas;
    double *stats;
    int D, from0, from1;
};

// Column statistics of the draws (FR:1656-1658, 1671): per column the mean over rows from1.., the standard deviation
// over rows from1.. (two-pass, like numpy) and the mean over rows from0...  A CTA takes 32 columns; its 16 row lanes
// walk interleaved rows (coalesced 256-byte reads, 16 independent partial sums per column instead of one 1000-deep
// dependent chain) and are summed in a fixed order.
constexpr int kStatsRows = 16;

__global__ void __launch_bounds__(32 * kStatsRows) cand_stats_kernel(const StatsParams P)
{
    __shared__ double red[2][kStatsRows][33];
    const int c = P.chain_list[blockIdx.y];
    const CandMeta m = P.meta[c];
    const int p = m.p;
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int i = blockIdx.x * 32 + tx;
    if (blockIdx.x * 32 >= p) return;
    const bool on = i < p;
    const double *B = P.betas + (int64_t)P.D * m.vec_off;
    double s0 = 0.0, s1 = 0.0;
    if (on)
        for (int k = P.from0 + ty; k < P.D; k += kStatsRows) {
            const double v = B[(int64_t)k * p + i];
            s0 += v;
            if (k >= P.from1) s1 += v;
        }
    red[0][ty][tx] = s0;
    red[1][ty][tx] = s1;
    __syncthreads();
    s0 = 0.0; s1 = 0.0;
    for (int r = 0; r < kStatsRows; ++r) { s0 += red[0][r][tx]; s1 += red[1][r][tx]; }
    // a window that starts at or after row D (D <= 3 with the windows of FR:1656-1658) is empty: its mean and standard
    // deviation are NaN, as numpy's of an empty slice
    const double n0 = (double)(P.D - P.from0), n1 = (double)(P.D - P.from1);
    const double m0 = n0 > 0.0 ? s0 / n0 : nan(""), m1 = n1 > 0.0 ? s1 / n1 : nan("");
    double q = 0.0;
    if (on)
        for (int k = P.from1 + ty; k < P.D; k += kStatsRows) {
            const double d = B[(int64_t)k * p + i] - m1;
            q += d * d;
        }
    __syncthreads();
    red[0][ty][tx] = q;
    __syncthreads();
    if (ty == 0 && on) {
        q = 0.0;
        for (int r = 0; r < kStatsRows; ++r) q += red[0][r][tx];
        double *S = P.stats + 3 * m.vec_off;
        S[i] = m1;
        S[p + i] = n1 > 0.0 ? sqrt(q / n1) : nan("");
        S[2 * p + i] = m0;
    }
}

struct KillParams {
    const double *G;
    int64_t ldg;
    const double *Xty;
    const int32_t *cols, *props;
    int p, k;
    CandConst c;
    double *L_global, *z, *beta, *wbuf, *ev;
    int32_t *info;
    int smem_doubles;
};

constexpr int kKillThreads = 1024;

__global__ void __launch_bounds__(kKillThreads) kill_scores_kernel(const KillParams P)
{
    extern __shared__ __align__(16) double sh[];
    const Team t = make_team();
    double *red = sh;
    volatile int *flag = reinterpret_cast<volatile int *>(sh + 2 * 3 * (kKillThreads / 32));
    double *L = ((int64_t)P.p * P.p <= P.smem_doubles) ? (sh + 2 * 3 * (kKillThreads / 32) + 2) : P.L_global;
    int bad = fokl::kill_scores(t, P.G, P.ldg, P.Xty, P.cols, P.p, P.props, P.k, P.c, L, P.z, P.beta, P.wbuf, P.ev,
                                flag, red);
    if (t.tid == 0) P.info[0] = bad;
}

struct KillLoopParams {
    const double *G;
    int64_t ldg;
    const double *Xty;
    const int32_t *cols, *cand_pos;
    const double *bv0, *bv1;
    int p, vm;
    CandConst c;
    fokl::KillLoopIn in;
    double *T_global;
    int32_t *out_i;
    double *out_ev;
    int smem_doubles;
    const double *T0;        // tableau after the forward sweeps (kill_tableau_kernel) or null
    int ldt0;
};

__global__ void __launch_bounds__(kKillThreads) kill_loop_kernel(const KillLoopParams P)
{
    extern __shared__ __align__(16) double sh[];
    const Team t = make_team();
    int *shi = reinterpret_cast<int *>(sh);                       // 4 ints
    double *rowbuf = sh + 2;                                      // p + 1 doubles (+ 1 pad): copy of the pivot row
    // packed symmetric tableau in shared memory when it fits, else the full form in global memory (L2)
    const bool packed = P.smem_doubles > 0;
    double *T = packed ? (sh + 2 + ((P.p + 2) & ~1)) : P.T_global;
    fokl::kill_loop(t, P.G, P.ldg, P.Xty, P.cols, P.p, P.cand_pos, P.bv0, P.bv1, P.vm, P.c, P.in, T, P.out_i, P.out_ev,
                    shi, rowbuf, packed, P.T0, P.ldt0);
}

// ---- the kill loop's tableau AFTER its p forward sweeps, from the model's eigendecomposition -------------------------------
// Sweeping all p pivots of [A b; b' c] gives [-A^-1  A^-1 b; b' A^-1  c - b' A^-1 b].  When the model is the substage's
// full model its eigendecomposition A = Q Lam Q' has just been computed (FR:1499), so the block is a plain
// symmetric product, A^-1 = (Q Lam^-1/2)(Q Lam^-1/2)', that every SM can work on -- instead of p strictly sequential
// rank-one updates by one CTA (or p grid barriers for a wide model).  b, c: centred like fokl::kill_loop_t.
// Usable flag (T0[(p + 1) ldt]): 1.0 iff lam_min > 1e-10 max_k A_kk -- then every pivot of the sequential form would
// have passed its own test (pivot >= lam_min), so both forms take the same path; otherwise the kill kernels run the
// sequential sweeps with their own positive-definiteness test as before.
struct KillTabParams {
    const double *G;
    int64_t ldg;
    const double *Xty;
    const int32_t *cols;
    int p, ldt;
    const double *lamb, *Qt;     // eigenvalues ascending; Qt[k * p + i] = component i of eigenvector k
    double ybar, cc;             // mean of y; yty - n ybar^2
    double *w;                   // p doubles: (Q' b)_k / lam_k
    double *T0;                  // (p + 1) x ldt, + the flag
};

__global__ void __launch_bounds__(256) kill_w_kernel(const KillTabParams P)
{
    const int lane = threadIdx.x & 31, k = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (k >= P.p) return;
    const int64_t row0 = (int64_t)P.cols[0] * P.ldg;
    const double *q = P.Qt + (int64_t)k * P.p;
    double s = 0.0;
    for (int i = lane; i < P.p; i += 32) s = fma(q[i], P.Xty[P.cols[i]] - P.ybar * P.G[row0 + P.cols[i]], s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) P.w[k] = s / P.lamb[k];
}

constexpr int kTabTile = 32;
__global__ void __launch_bounds__(256) kill_tableau_kernel(const KillTabParams P)
{
    __shared__ double As[kTabTile][kTabTile + 1], Bs[kTabTile][kTabTile + 1];
    __shared__ double red[8];
    const int p = P.p, ldt = P.ldt, tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
    const int nt = (p + kTabTile - 1) / kTabTile;
    const int n_tiles = nt * (nt + 1) / 2;
    if ((int)blockIdx.x == n_tiles) {
        // last row / column: betahat = Q w; corner: c - sum w_k^2 lam_k; the usable flag
        for (int j = tid; j < p; j += 256) {
            double b = 0.0;
            for (int k = 0; k < p; ++k) b = fma(P.Qt[(int64_t)k * p + j], P.w[k], b);
            P.T0[(int64_t)p * ldt + j] = b;
            P.T0[(int64_t)j * ldt + p] = b;
        }
        double s = 0.0, dmax = 0.0;
        for (int k = tid; k < p; k += 256) {
            s = fma(P.w[k] * P.w[k], P.lamb[k], s);
            dmax = fmax(dmax, P.G[(int64_t)P.cols[k] * P.ldg + P.cols[k]]);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s += __shfl_xor_sync(0xffffffffu, s, o);
            dmax = fmax(dmax, __shfl_xor_sync(0xffffffffu, dmax, o));
        }
        __shared__ double red2[8];
        if (tx == 0) { red[ty] = s; red2[ty] = dmax; }
        __syncthreads();
        if (tid == 0) {
            double st = 0.0, dm = 0.0;
            for (int q = 0; q < 8; ++q) { st += red[q]; dm = fmax(dm, red2[q]); }
            const double sse = P.cc - st;
            P.T0[(int64_t)p * ldt + p] = sse;
            const double l0 = P.lamb[0];
            const bool ok = l0 > 1e-10 * dm && sse == sse && fabs(sse) < 1.79e308;
            P.T0[(int64_t)(p + 1) * ldt] = ok ? 1.0 : 0.0;
        }
        return;
    }
    // tile (bi >= bj) of -A^-1 from the linear tile index
    int bi = (int)((sqrt(8.0 * (double)blockIdx.x + 1.0) - 1.0) * 0.5);
    while (bi * (bi + 1) / 2 > (int)blockIdx.x) --bi;
    while ((bi + 1) * (bi + 2) / 2 <= (int)blockIdx.x) ++bi;
    const int bj = (int)blockIdx.x - bi * (bi + 1) / 2;
    const int i0 = bi * kTabTile, j0 = bj * kTabTile;
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    for (int k0 = 0; k0 < p; k0 += kTabTile) {
#pragma unroll
        for (int m = 0; m < 4; ++m) {
            const int kk = ty + 8 * m, k = k0 + kk;
            const bool kin = k < p;
            const double il = kin ? 1.0 / P.lamb[k] : 0.0;
            As[kk][tx] = (kin && i0 + tx < p) ? P.Qt[(int64_t)k * p + i0 + tx] * il : 0.0;
            Bs[kk][tx] = (kin && j0 + tx < p) ? P.Qt[(int64_t)k * p + j0 + tx] : 0.0;
        }
        __syncthreads();
#pragma unroll 8
        for (int kk = 0; kk < kTabTile; ++kk) {
            const double b = Bs[kk][tx];
#pragma unroll
            for (int m = 0; m < 4; ++m) acc[m] = fma(As[kk][ty + 8 * m], b, acc[m]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int m = 0; m < 4; ++m) {
        const int i = i0 + ty + 8 * m, j = j0 + tx;
        if (i < p && j < p && i >= j) {                 // (diagonal tiles: one writer per symmetric pair)
            P.T0[(int64_t)i * ldt + j] = -acc[m];
            P.T0[(int64_t)j * ldt + i] = -acc[m];
        }
    }
}

template <typename T>
T *carve(char *&cur, size_t count)
{
    uintptr_t a = ((uintptr_t)cur + 15) & ~(uintptr_t)15;
    T *r = reinterpret_cast<T *>(a);
    cur = reinterpret_cast<char *>(a + count * sizeof(T));
    return r;
}

}  // namespace

extern "C" int fokl_candidates_eval(fokl_ctx *ctx, const double *G, int64_t ldg, const double *Xty,
                                    const int32_t *col_sets, const int32_t *set_offsets, int n_cand,
                                    const fokl_hypers *hyp, const uint8_t *run_chain, int rng_mode, uint64_t seed,
                                    const uint64_t *stream_ids, const double *variates, const double *sign_fix,
                                    double *ev, double *betahat, double *lamb, double *Q, double *betas,
                                    double *sigs, double *taus, double *stats, int32_t *info)
{
    FOKL_CHECK_CTX(ctx);
    if (!G || !Xty || !col_sets || !set_offsets || !hyp || !ev || !info || n_cand < 1)
        FOKL_FAIL(ctx, FOKL_EINVAL, "candidates_eval: bad argument");
    if (rng_mode != FOKL_RNG_NONE && rng_mode != FOKL_RNG_INJECTED && rng_mode != FOKL_RNG_PHILOX)
        FOKL_FAIL(ctx, FOKL_EINVAL, "candidates_eval: unknown rng_mode");
    if (rng_mode == FOKL_RNG_INJECTED && !variates) FOKL_FAIL(ctx, FOKL_EINVAL, "candidates_eval: variates required");
    if (rng_mode != FOKL_RNG_NONE && hyp->draws < 1) FOKL_FAIL(ctx, FOKL_EINVAL, "candidates_eval: draws < 1");
    int rc = fokl_bind_device(ctx);
    if (rc) return rc;
    fokl_hp_scope hp(ctx);
    if (hp.rc) return hp.rc;

    const int D = hyp->draws;
    const size_t smem_cap = ctx->smem_optin ? ctx->smem_optin : 48 * 1024;
    const int smem_wv_cap = (int)((smem_cap - kSmemHeaderDoubles * sizeof(double)) / sizeof(double));

    if (!ctx->cluster_probed) {
        // clusters of 16 CTAs are "non-portable": use them only if this device can co-schedule one at full shared memory
        ctx->cluster_probed = true;
        if (cudaFuncSetAttribute(cand_eigj_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess &&
            cudaFuncSetAttribute(cand_eigj_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cap) == cudaSuccess) {
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(kEigJMaxCluster);
            cfg.blockDim = dim3(kEigJThreads);
            cfg.dynamicSmemBytes = smem_cap;
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeClusterDimension;
            attr[0].val.clusterDim.x = kEigJMaxCluster;
            attr[0].val.clusterDim.y = 1;
            attr[0].val.clusterDim.z = 1;
            cfg.attrs = attr;
            cfg.numAttrs = 1;
            int nc = 0;
            if (cudaOccupancyMaxActiveClusters(&nc, cand_eigj_kernel, &cfg) == cudaSuccess && nc >= 1) ctx->max_cluster = kEigJMaxCluster;
        }
        cudaGetLastError();
    }
    int force_cs = 0;                    // tuning knob for tools/eig_batch_diag.py: force the eigensolver's cluster size
    if (const char *e = getenv("FOKL_EIGJ_CS")) force_cs = atoi(e);
    // models at least this wide go to the blocked DMMA eigensolver (eigbig.cuh) instead of the cluster solver
    int eigb_min_p = 64 * kEigJMaxNV + 1;
    if (const char *e = getenv("FOKL_EIGB_MIN_P")) eigb_min_p = std::max(2, atoi(e));
    eigb_min_p = std::min(eigb_min_p, 64 * kEigJMaxNV + 1);
    std::vector<int32_t> big_list;
    if (force_cs != 1 && force_cs != 2 && force_cs != 4 && force_cs != 8 && force_cs != 16) force_cs = 0;
    std::vector<CandMeta> meta(n_cand);
    std::vector<int32_t> chain_list;
    std::vector<int> eig_class(n_cand, 0);
    int64_t vec = 0, mat = 0, wv = 0, gam = 0;
    int pmax = 0, pmax_chain = 0;
    for (int c = 0; c < n_cand; ++c) {
        int p = set_offsets[c + 1] - set_offsets[c];
        if (p < 1 || ldg < p) FOKL_FAIL(ctx, FOKL_EINVAL, "candidates_eval: empty or oversized column set");
        if (col_sets[set_offsets[c]] < 0) FOKL_FAIL(ctx, FOKL_EINVAL, "candidates_eval: negative column index");
        CandMeta &m = meta[c];
        m.p = p; m.set_off = set_offsets[c]; m.pad = 0;
        m.vec_off = vec; m.mat_off = mat;
        // cluster size of the Jacobi eigensolver: the smallest whose column buffers fit in shared memory; raised below
        if (p >= eigb_min_p) {
            m.pad = 2;                                                     // blocked one-sided Jacobi on the tensor pipe
            big_list.push_back(c);
        } else {
            int cs = force_cs > 0 ? force_cs : 1;
            while (cs <= kEigJMaxCluster && eigj_smem_bytes(p, cs) > smem_cap) cs *= 2;
            if (cs > ctx->max_cluster) { m.pad = 2; big_list.push_back(c); }   // no cluster of that size on this device
            else eig_class[c] = cs;
        }
        // W | V workspace of the two-matrix fallback (Gram not positive definite): only models of the cluster class
        const bool in_smem = (2 * (int64_t)p * p <= smem_wv_cap);
        m.wv_off = wv;
        if (!in_smem && m.pad != 2) wv += 2 * (int64_t)p * p;
        const bool chain = rng_mode != FOKL_RNG_NONE && (!run_chain || run_chain[c]);
        m.chain_idx = chain ? (int32_t)chain_list.size() : -1;
        m.gam_off = gam;
        m.stream_id = stream_ids ? stream_ids[c] : (uint64_t)c;
        if (chain) { chain_list.push_back(c); gam += p; pmax_chain = std::max(pmax_chain, p); }
        vec += p; mat += (int64_t)p * p;
        pmax = std::max(pmax, p);
    }
    const int n_chain = (int)chain_list.size();
    const int total_p = set_offsets[n_cand];

    // ---- cluster sizes of the batch ---------------------------------------------------------------------------------
    // A candidate's eigensolve is a fixed number of rounds whose length shrinks with the cluster size until every column
    // pair has a warp of its own, and a cluster pays one cluster barrier + DSMEM exchange per round: per round about
    // a(p) * ceil(pairs per CTA / 16) + [cs > 1] * b(p) microseconds with a = 0.25 + 0.0035 p, b = 0.005 p
    // (fit to profiles/r01_eig_batch_diag.txt).  A batch ends with its slowest candidate, so while the batch still fits the
    // device in one wave (sum of cluster sizes <= SMs) the cluster of the currently slowest candidate is raised.
    if (force_cs == 0) {
        auto est = [&](int p, int cs) {
            const int n = eigj_padded_n(p, cs);
            const int pairs = (n / 2 + cs - 1) / cs;
            const double a = 0.25 + 0.0035 * p, b = cs > 1 ? 0.005 * p : 0.0;
            return (double)(n - 1) * (a * ((pairs + kEigJThreads / 32 - 1) / (kEigJThreads / 32)) + b);
        };
        int64_t ctas = 0;
        const int sm_budget = (ctx->sm_budget > 0 && ctx->sm_budget < ctx->num_sms) ? ctx->sm_budget : ctx->num_sms;
        std::priority_queue<std::pair<double, int>> heap;
        for (int c = 0; c < n_cand; ++c) {
            ctas += std::max(eig_class[c], 1);
            if (eig_class[c] > 0) heap.push({est(meta[c].p, eig_class[c]), c});
        }
        while (!heap.empty()) {
            const double t = heap.top().first;
            const int c = heap.top().second;
            heap.pop();
            const int cs = eig_class[c], p = meta[c].p;
            int best = cs;
            double tb = t;
            for (int c2 = cs * 2; c2 <= ctx->max_cluster && ctas - cs + c2 <= sm_budget; c2 *= 2) {
                const double t2 = est(p, c2);
                if (t2 < 0.97 * t) { best = c2; tb = t2; break; }
            }
            if (best == cs) break;              // the slowest candidate cannot be made faster: the batch time is set
            ctas += best - cs;
            eig_class[c] = best;
            heap.push({tb, c});
        }
    }

    // ---- plan of the blocked eigensolver (models too wide for a cluster) -------------------------------------
    const int n_big = (int)big_list.size();
    const int sm_budget_b = (ctx->sm_budget > 0 && ctx->sm_budget < ctx->num_sms) ? ctx->sm_budget : ctx->num_sms;
    std::vector<eigb::Job> jobs;
    int64_t wbig = 0;
    int eigb_team = 1, eigb_teams = 0, eigb_nb_max = 2;
    if (n_big > 0) {
        std::sort(big_list.begin(), big_list.end(), [&](int x, int y) { return meta[x].p > meta[y].p || (meta[x].p == meta[y].p && x < y); });
        for (int c : big_list) {
            eigb::Job J;
            J.cand = c; J.p = meta[c].p; J.ld = (meta[c].p + 15) & ~15;
            J.nb = (meta[c].p + eigb::kB - 1) / eigb::kB; J.nb += J.nb & 1;
            J.set_off = meta[c].set_off; J.pad = 0;
            J.w_off = wv + wbig; J.vec_off = meta[c].vec_off; J.mat_off = meta[c].mat_off;
            meta[c].wv_off = J.w_off;                  // the not-positive-definite fallback reuses the area as W | V
            wbig += 2 * (int64_t)J.ld * J.nb * eigb::kB + (((int64_t)J.p / 2 + 16) & ~(int64_t)15);   // W (+ the fallback's V) + the column order (int32)
            eigb_nb_max = std::max(eigb_nb_max, (int)J.nb);
            jobs.push_back(J);
        }
        int occ = 0;
        FOKL_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, eigb::eigb_kernel, eigb::kThreads, eigb::kSmemBytes));
        if (occ < 1) FOKL_FAIL(ctx, FOKL_ECUDA, "candidates_eval: blocked eigensolver does not fit an SM");
        const int resident = occ * sm_budget_b;
        // teams: as many models in flight as keep their W matrices L2-resident (~96 MB), one CTA per block pair at most
        const int pairs_max = jobs[0].nb / 2;
        const int64_t w_bytes = (int64_t)jobs[0].ld * jobs[0].nb * eigb::kB * (int64_t)sizeof(double);
        int in_flight = (int)std::max<int64_t>(1, std::min<int64_t>(n_big, (96ll << 20) / std::max<int64_t>(w_bytes, 1)));
        if (const char *e = getenv("FOKL_EIGB_TEAM")) eigb_team = std::max(1, atoi(e));
        else eigb_team = std::max(1, std::min(pairs_max, resident / in_flight));
        eigb_team = std::min(eigb_team, resident);
        eigb_teams = std::max(1, std::min(n_big, resident / eigb_team));
    }
    // ---- metadata upload ---------------------------------------------------------------------------------
    std::vector<int32_t> eig_list;                 // candidates grouped by cluster size
    int class_begin[6] = {0, 0, 0, 0, 0, 0};       // cs = 1, 2, 4, 8, 16
    bool any_fallback = false;
    for (int q = 0, cs = 1; q < 5; ++q, cs *= 2) {
        class_begin[q] = (int)eig_list.size();
        for (int c = 0; c < n_cand; ++c)
            if (eig_class[c] == cs) eig_list.push_back(c);
    }
    class_begin[5] = (int)eig_list.size();
    for (int c = 0; c < n_cand; ++c) any_fallback = any_fallback || meta[c].pad;
    size_t meta_bytes = 64 + (size_t)total_p * sizeof(int32_t) + (size_t)n_cand * sizeof(CandMeta) +
                        (size_t)(n_chain + 1) * sizeof(int32_t) + (size_t)(n_cand + 1) * sizeof(int32_t) + 96 +
                        (size_t)(big_list.size() + 1) * (sizeof(eigb::Job) + sizeof(int32_t)) + 64;
    char *dmeta = (char *)fokl_scratch(ctx, fokl_ctx::B_META, meta_bytes);
    if (!dmeta) return FOKL_ENOMEM;
    std::vector<char> hmeta(meta_bytes, 0);
    char *dcur = dmeta;
    int32_t *d_sets = carve<int32_t>(dcur, total_p);
    CandMeta *d_meta = carve<CandMeta>(dcur, n_cand);
    int32_t *d_chain = carve<int32_t>(dcur, n_chain + 1);
    int32_t *d_eig_list = carve<int32_t>(dcur, n_cand + 1);
    int32_t *d_big_list = carve<int32_t>(dcur, n_big + 1);
    eigb::Job *d_jobs = carve<eigb::Job>(dcur, n_big + 1);
    if (n_big) {
        memcpy(hmeta.data() + ((char *)d_big_list - dmeta), big_list.data(), (size_t)n_big * sizeof(int32_t));
        memcpy(hmeta.data() + ((char *)d_jobs - dmeta), jobs.data(), (size_t)n_big * sizeof(eigb::Job));
    }
    if (!eig_list.empty())
        memcpy(hmeta.data() + ((char *)d_eig_list - dmeta), eig_list.data(), eig_list.size() * sizeof(int32_t));
    memcpy(hmeta.data() + ((char *)d_sets - dmeta), col_sets, (size_t)total_p * sizeof(int32_t));
    memcpy(hmeta.data() + ((char *)d_meta - dmeta), meta.data(), (size_t)n_cand * sizeof(CandMeta));
    if (n_chain) memcpy(hmeta.data() + ((char *)d_chain - dmeta), chain_list.data(), (size_t)n_chain * sizeof(int32_t));
    FOKL_CUDA(ctx, cudaMemcpyAsync(dmeta, hmeta.data(), (size_t)(dcur - dmeta), cudaMemcpyHostToDevice, ctx->stream));

    // ---- workspaces --------------------------------------------------------------------------------------
    double *d_wv = nullptr;
    if (wv + wbig > 0) {
        d_wv = (double *)fokl_scratch(ctx, fokl_ctx::B_CAND_A, (size_t)(wv + wbig) * sizeof(double));
        if (!d_wv) return FOKL_ENOMEM;
    }
    size_t b_bytes = 512 + (size_t)vec * (6 * sizeof(double) + sizeof(int32_t)) + (size_t)n_cand * 64 * sizeof(double) +
                     (Q ? 0 : (size_t)mat * sizeof(double));
    char *bcur = (char *)fokl_scratch(ctx, fokl_ctx::B_CAND_B, b_bytes);
    if (!bcur) return FOKL_ENOMEM;
    double *d_lam_raw = carve<double>(bcur, vec);
    double *d_lam_all = carve<double>(bcur, vec + (size_t)n_cand * 64);
    double *d_scratch = carve<double>(bcur, vec);
    double *d_ct = carve<double>(bcur, vec);
    double *d_lamb = lamb ? lamb : carve<double>(bcur, vec);
    double *d_betahat = betahat ? betahat : carve<double>(bcur, vec);
    int32_t *d_perm = carve<int32_t>(bcur, vec);
    double *d_Q = Q ? Q : carve<double>(bcur, mat);

    CandConst k;
    k.a = hyp->a; k.b = hyp->b; k.atau = hyp->atau; k.btau = hyp->btau;
    k.sigsqd0 = hyp->sigsqd0; k.tausqd0 = hyp->tausqd0; k.yty = hyp->yty; k.sum_y = hyp->sum_y;
    k.n = (double)hyp->n; k.draws = D; k.from0 = hyp->stat_from0; k.from1 = hyp->stat_from1;

    // ---- chain workspaces (allocated up front: the Philox variate tables are filled while the eigensolver runs) --------
    const bool philox = rng_mode == FOKL_RNG_PHILOX;
    double *d_gam = nullptr, *d_var = nullptr, *d_betas = nullptr, *d_sigs = nullptr, *d_taus = nullptr;
    if (n_chain > 0) {
        // a window may start at or after row D (an empty window: NaN statistics), never before row 0
        if (hyp->stat_from0 < 0 || hyp->stat_from1 < 0)
            FOKL_FAIL(ctx, FOKL_EINVAL, "candidates_eval: negative statistic window start");
        size_t c_bytes = 256 + ((size_t)D * gam + (philox ? (size_t)D * (gam + 2 * (size_t)n_chain) : 0)) * sizeof(double);
        char *ccur = (char *)fokl_scratch(ctx, fokl_ctx::B_CAND_C, c_bytes);
        if (!ccur) return FOKL_ENOMEM;
        d_gam = carve<double>(ccur, (size_t)D * gam);
        d_var = philox ? carve<double>(ccur, (size_t)D * (gam + 2 * (size_t)n_chain)) : nullptr;
        size_t d_bytes = 256 + (betas ? 0 : (size_t)D * vec * sizeof(double)) + (sigs ? 0 : (size_t)D * n_cand * sizeof(double)) +
                         (taus ? 0 : (size_t)D * n_cand * sizeof(double));
        char *ecur = (char *)fokl_scratch(ctx, fokl_ctx::B_CAND_D, d_bytes);
        if (!ecur) return FOKL_ENOMEM;
        d_betas = betas ? betas : carve<double>(ecur, (size_t)D * vec);
        d_sigs = sigs ? sigs : carve<double>(ecur, (size_t)D * n_cand);
        d_taus = taus ? taus : carve<double>(ecur, (size_t)D * n_cand);
    }
    ChainParams CP;
    CP.meta = d_meta; CP.chain_list = d_chain; CP.k = k; CP.lamb = d_lamb; CP.ct = d_ct;
    CP.rng_mode = rng_mode; CP.seed = seed; CP.variates = variates; CP.var_philox = d_var; CP.sign_fix = sign_fix;
    CP.gam = d_gam; CP.sigs = d_sigs; CP.taus = d_taus; CP.info = info;
    bool variates_forked = false;

    // ---- eig + betahat + BIC -------------------------------------------------------------------------------
    // (1) Cholesky factor of every candidate (into its Q slot); (2) per cluster-size class, the cluster Jacobi on the
    // factor + betahat + BIC; (3) the two-matrix Jacobi for candidates whose Gram is not positive definite or that do
    // not fit a cluster (exits immediately for everyone else).
    {
        CholParams C;
        C.G = G; C.ldg = ldg; C.col_sets = d_sets; C.meta = d_meta; C.Q = d_Q; C.info = info;
        int64_t need = 0;
        for (int c = 0; c < n_cand; ++c) {
            const int64_t tri = (int64_t)meta[c].p * (meta[c].p + 1) / 2;
            if (!meta[c].pad && tri * (int64_t)sizeof(double) <= (int64_t)smem_cap) need = std::max<int64_t>(need, tri);
        }
        C.smem_doubles = (int)need;
        FOKL_CUDA(ctx, cudaFuncSetAttribute(cand_chol_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cap));
        cand_chol_kernel<<<n_cand, kCholThreads, (size_t)need * sizeof(double), ctx->stream>>>(C);
        FOKL_LAUNCH_CHECK(ctx);
    }
    {
        EigJParams J;
        J.G = G; J.ldg = ldg; J.Xty = Xty; J.col_sets = d_sets; J.meta = d_meta; J.k = k;
        J.lam_raw = d_lam_all; J.scratch = d_scratch; J.ct = d_ct; J.lamb = d_lamb; J.Q = d_Q; J.betahat = d_betahat;
        J.ev = ev; J.info = info;
        FOKL_CUDA(ctx, cudaFuncSetAttribute(cand_eigj_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cap));
        // one launch per cluster size; the launches are independent of one another, so the second and later ones go to
        // auxiliary streams and fill the SMs the first leaves idle (largest clusters = longest candidates first)
        int used_aux = 0;
        bool first = true;
        rc = fokl_fork_point(ctx);           // after the Cholesky pre-pass, before any eigensolver launch
        if (rc) return rc;
        if (n_chain > 0 && philox) {
            // Philox table of every chain (independent of the eigensolver): last auxiliary stream
            cudaStream_t sv = fokl_aux_fork(ctx, fokl_ctx::kAux - 1);
            if (!sv) FOKL_FAIL(ctx, FOKL_ECUDA, "candidates_eval: auxiliary stream");
            const int64_t per_chain = (int64_t)D * (pmax_chain + 2);
            dim3 grid((unsigned)std::min<int64_t>((per_chain + 255) / 256, 2048), (unsigned)n_chain);
            cand_variates_kernel<<<grid, 256, 0, sv>>>(CP);
            FOKL_LAUNCH_CHECK(ctx);
            variates_forked = true;
        }
        for (int q = 4, cs = 16; q >= 0; --q, cs /= 2) {
            const int cnt = class_begin[q + 1] - class_begin[q];
            if (cnt == 0) continue;
            size_t smem = 0;
            int threads = 32;
            for (int e = class_begin[q]; e < class_begin[q + 1]; ++e) {
                smem = std::max(smem, eigj_smem_bytes(meta[eig_list[e]].p, cs));
                threads = std::max(threads, eigj_threads(meta[eig_list[e]].p, cs));
            }
            J.list = d_eig_list + class_begin[q];
            cudaStream_t st = ctx->stream;
            if (!first && used_aux < fokl_ctx::kAux - 1) {
                st = fokl_aux_fork(ctx, used_aux);
                if (!st) FOKL_FAIL(ctx, FOKL_ECUDA, "candidates_eval: auxiliary stream");
                ++used_aux;
            }
            first = false;
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3((unsigned)(cnt * cs));
            cfg.blockDim = dim3((unsigned)threads);
            cfg.dynamicSmemBytes = smem;
            cfg.stream = st;
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeClusterDimension;
            attr[0].val.clusterDim.x = (unsigned)cs;
            attr[0].val.clusterDim.y = 1;
            attr[0].val.clusterDim.z = 1;
            cfg.attrs = attr;
            cfg.numAttrs = 1;
            FOKL_CUDA(ctx, cudaLaunchKernelEx(&cfg, cand_eigj_kernel, J));
            FOKL_LAUNCH_CHECK(ctx);
        }
        for (int i = 0; i < used_aux; ++i) {
            rc = fokl_aux_join(ctx, i);
            if (rc) return rc;
        }
    }
    if (n_big > 0) {
        // Cholesky + blocked one-sided Jacobi (eigbig.cuh): one cooperative launch, teams of CTAs fetch models from a
        // dispenser
        const int vstride = (eigb_nb_max + 31) & ~31;
        const size_t sync_ints = (size_t)eigb_teams * (2 + eigb::kFlagStride + vstride) + 32 + (size_t)n_cand;
        int *d_sync = (int *)fokl_scratch(ctx, fokl_ctx::B_MISC, sync_ints * sizeof(int));
        if (!d_sync) return FOKL_ENOMEM;
        FOKL_CUDA(ctx, cudaMemsetAsync(d_sync, 0, sync_ints * sizeof(int), ctx->stream));
        eigb::Params E;
        E.G = G; E.ldg = ldg; E.col_sets = d_sets; E.jobs = d_jobs; E.n_jobs = n_big; E.team = eigb_team;
        E.W = d_wv; E.lam_raw = d_lam_all; E.lamb = d_lamb; E.Q = d_Q;
        E.bar = reinterpret_cast<unsigned *>(d_sync);
        E.slot = d_sync + eigb_teams;
        E.next = d_sync + 2 * eigb_teams;
        E.flags = d_sync + 2 * eigb_teams + 32;
        E.ver = E.flags + (size_t)eigb_teams * eigb::kFlagStride;
        E.ver_stride = vstride;
        E.status = E.ver + (size_t)eigb_teams * vstride;
        E.max_inner = 1;
        if (const char *e = getenv("FOKL_EIGB_INNER")) E.max_inner = std::max(1, atoi(e));
        E.sort_diag = 1;
        if (const char *e = getenv("FOKL_EIGB_SORT")) E.sort_diag = atoi(e) != 0;
        void *args[] = {(void *)&E};
        FOKL_CUDA(ctx, cudaLaunchCooperativeKernel((const void *)eigb::eigb_kernel, dim3((unsigned)(eigb_teams * eigb_team)),
                                                   dim3(eigb::kThreads), args, eigb::kSmemBytes, ctx->stream));
        FOKL_LAUNCH_CHECK(ctx);
        OlsParams O;
        O.G = G; O.ldg = ldg; O.Xty = Xty; O.col_sets = d_sets; O.meta = d_meta; O.list = d_big_list; O.k = k;
        O.scratch = d_scratch; O.ct = d_ct; O.lamb = d_lamb; O.Q = d_Q; O.betahat = d_betahat; O.ev = ev; O.info = info;
        O.sweeps = E.status;
        cand_ols_kernel<<<n_big, 1024, 0, ctx->stream>>>(O);
        FOKL_LAUNCH_CHECK(ctx);
    }
    {
        EigParams P;
        P.G = G; P.ldg = ldg; P.Xty = Xty; P.col_sets = d_sets; P.meta = d_meta; P.k = k;
        P.wv = d_wv; P.lam_raw = d_lam_raw; P.scratch = d_scratch; P.ct = d_ct; P.perm = d_perm;
        P.lamb = d_lamb; P.Q = d_Q; P.betahat = d_betahat; P.ev = ev; P.info = info;
        P.only_flagged = 1;
        int64_t need = 2 * (int64_t)pmax * pmax;
        int wv_doubles = (int)std::min<int64_t>(need, smem_wv_cap);
        if (need > smem_wv_cap) {
            // the largest candidate spills to global memory; still give smaller ones what they need
            int best = 0;
            for (int c = 0; c < n_cand; ++c) {
                int64_t q = 2 * (int64_t)meta[c].p * meta[c].p;
                if (q <= smem_wv_cap) best = std::max<int>(best, (int)q);
            }
            wv_doubles = best;
        }
        P.smem_doubles = wv_doubles;
        size_t smem = (size_t)(kSmemHeaderDoubles + wv_doubles) * sizeof(double);
        FOKL_CUDA(ctx, cudaFuncSetAttribute(cand_eig_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cap));
        cand_eig_kernel<<<n_cand, kEigThreads, smem, ctx->stream>>>(P);
        FOKL_LAUNCH_CHECK(ctx);
    }
    (void)any_fallback;
    // every eigensolver launch of this call is enqueued: a Gram build on another context that must not take the SMs
    // away from the cluster launches waits for this point (fokl_ctx_wait_eig)
    if (!ctx->ev_eig) FOKL_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_eig, cudaEventDisableTiming));
    FOKL_CUDA(ctx, cudaEventRecord(ctx->ev_eig, ctx->stream));
    ctx->ev_eig_set = true;
    if (n_chain == 0) return FOKL_OK;

    // ---- chain -------------------------------------------------------------------------------------------------
    {
        if (variates_forked) {
            rc = fokl_aux_join(ctx, fokl_ctx::kAux - 1);
            if (rc) return rc;
        }
        if (pmax_chain <= 64) {
            cand_chain_warp_kernel<2><<<n_chain, 32, 0, ctx->stream>>>(CP);
        } else if (pmax_chain <= 128) {
            cand_chain_warp_kernel<4><<<n_chain, 32, 0, ctx->stream>>>(CP);
        } else if (pmax_chain <= 256) {
            cand_chain_warp_kernel<8><<<n_chain, 32, 0, ctx->stream>>>(CP);
        } else {
            const int chain_threads = std::max(32, std::min(kChainThreads, 32 * ((pmax_chain / 2 + 31) / 32)));
            cand_chain_kernel<<<n_chain, chain_threads, 0, ctx->stream>>>(CP);
        }
        FOKL_LAUNCH_CHECK(ctx);
    }
    if (!betas && !stats) return FOKL_OK;
    {
        BetasParams P;
        P.meta = d_meta; P.chain_list = d_chain; P.gam = d_gam; P.Q = d_Q; P.betas = d_betas; P.D = D;
        P.tiles_i = (pmax_chain + 63) / 64;
        dim3 grid((unsigned)(P.tiles_i * ((D + 63) / 64)), (unsigned)n_chain);
        cand_betas_kernel<<<grid, 256, 0, ctx->stream>>>(P);
        FOKL_LAUNCH_CHECK(ctx);
    }
    if (stats) {
        StatsParams P;
        P.meta = d_meta; P.chain_list = d_chain; P.betas = d_betas; P.stats = stats; P.D = D;
        P.from0 = hyp->stat_from0; P.from1 = hyp->stat_from1;
        dim3 grid((unsigned)((pmax_chain + 31) / 32), (unsigned)n_chain);
        cand_stats_kernel<<<grid, dim3(32, kStatsRows), 0, ctx->stream>>>(P);
        FOKL_LAUNCH_CHECK(ctx);
    }
    return FOKL_OK;
}

extern "C" int fokl_kill_scores(fokl_ctx *ctx, const double *G, int64_t ldg, const double *Xty, const int32_t *cols,
                                int p, const int32_t *props, int k, const fokl_hypers *hyp, double *ev, int32_t *info)
{
    FOKL_CHECK_CTX(ctx);
    if (!G || !Xty || !cols || !hyp || !ev || !info || p < 1 || k < 0 || ldg < p || (k > 0 && !props))
        FOKL_FAIL(ctx, FOKL_EINVAL, "kill_scores: bad argument");
    for (int a = 0; a < k; ++a)
        if (props[a] < 1 || props[a] >= p) FOKL_FAIL(ctx, FOKL_EINVAL, "kill_scores: proposal position out of range");
    int rc = fokl_bind_device(ctx);
    if (rc) return rc;
    fokl_hp_scope hp(ctx);
    if (hp.rc) return hp.rc;
    const size_t smem_cap = ctx->smem_optin ? ctx->smem_optin : 48 * 1024;
    const int header = 2 * 3 * (kKillThreads / 32) + 2;
    const int smem_l_cap = (int)(smem_cap / sizeof(double)) - header;
    const bool in_smem = (int64_t)p * p <= smem_l_cap;

    size_t meta_bytes = 64 + (size_t)(p + k + 1) * sizeof(int32_t);
    char *dmeta = (char *)fokl_scratch(ctx, fokl_ctx::B_META, meta_bytes);
    if (!dmeta) return FOKL_ENOMEM;
    std::vector<int32_t> h((size_t)p + k + 1);
    memcpy(h.data(), cols, (size_t)p * sizeof(int32_t));
    if (k) memcpy(h.data() + p, props, (size_t)k * sizeof(int32_t));
    FOKL_CUDA(ctx, cudaMemcpyAsync(dmeta, h.data(), (size_t)(p + k) * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));

    size_t ws = 256 + ((size_t)(in_smem ? 0 : (size_t)p * p) + 2 * (size_t)p + (size_t)(kKillThreads / 32) * p) * sizeof(double);
    char *wcur = (char *)fokl_scratch(ctx, fokl_ctx::B_CAND_A, ws);
    if (!wcur) return FOKL_ENOMEM;
    KillParams P;
    P.G = G; P.ldg = ldg; P.Xty = Xty;
    P.cols = reinterpret_cast<const int32_t *>(dmeta);
    P.props = P.cols + p;
    P.p = p; P.k = k;
    P.c.a = hyp->a; P.c.b = hyp->b; P.c.atau = hyp->atau; P.c.btau = hyp->btau;
    P.c.sigsqd0 = hyp->sigsqd0; P.c.tausqd0 = hyp->tausqd0; P.c.yty = hyp->yty; P.c.sum_y = hyp->sum_y;
    P.c.n = (double)hyp->n; P.c.draws = hyp->draws; P.c.from0 = hyp->stat_from0; P.c.from1 = hyp->stat_from1;
    P.z = carve<double>(wcur, p);
    P.beta = carve<double>(wcur, p);
    P.wbuf = carve<double>(wcur, (size_t)(kKillThreads / 32) * p);
    P.L_global = in_smem ? nullptr : carve<double>(wcur, (size_t)p * p);
    P.ev = ev; P.info = info;
    P.smem_doubles = in_smem ? p * p : 0;
    size_t smem = (size_t)(header + (in_smem ? p * p : 0)) * sizeof(double);
    FOKL_CUDA(ctx, cudaFuncSetAttribute(kill_scores_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cap));
    kill_scores_kernel<<<1, kKillThreads, smem, ctx->stream>>>(P);
    FOKL_LAUNCH_CHECK(ctx);
    return FOKL_OK;
}

extern "C" int fokl_kill_loop(fokl_ctx *ctx, const double *G, int64_t ldg, const double *Xty, const int32_t *cols, int p,
                              const int32_t *cand_pos, const double *bv0, const double *bv1, int vm,
                              const fokl_hypers *hyp, const fokl_kill_params *kp, int32_t *out_i, double *out_ev)
{
    FOKL_CHECK_CTX(ctx);
    if (!G || !Xty || !cols || !hyp || !kp || !out_i || !out_ev || p < 1 || vm < 0 || ldg < p ||
        (vm > 0 && (!cand_pos || !bv0 || !bv1)))
        FOKL_FAIL(ctx, FOKL_EINVAL, "kill_loop: bad argument");
    if (kp->start < 0 || kp->start > vm) FOKL_FAIL(ctx, FOKL_EINVAL, "kill_loop: start outside the candidate list");
    for (int i = kp->start; i < vm; ++i)
        if (cand_pos[i] < 1 || cand_pos[i] >= p) FOKL_FAIL(ctx, FOKL_EINVAL, "kill_loop: candidate position out of range");
    int rc = fokl_bind_device(ctx);
    if (rc) return rc;
    fokl_hp_scope hp(ctx);
    if (hp.rc) return hp.rc;
    const size_t smem_cap = ctx->smem_optin ? ctx->smem_optin : 48 * 1024;
    const int head = 2 + ((p + 2) & ~1);                         // flags + pivot-row copy
    const int smem_t_cap = (int)(smem_cap / sizeof(double)) - head;
    const int64_t need_packed = (int64_t)(p + 1) * (p + 2) / 2;            // symmetric tableau, lower triangle
    const int64_t need_full = (int64_t)(p + 1) * (p + 1);
    const bool in_smem = need_packed <= smem_t_cap;
    const int64_t need = in_smem ? need_packed : need_full;

    // metadata: cols (p ints), cand_pos (vm ints), bv0, bv1 (vm doubles each)
    size_t off_pos = (size_t)p * sizeof(int32_t);
    size_t off_bv = (off_pos + (size_t)vm * sizeof(int32_t) + 15) & ~(size_t)15;
    size_t meta_bytes = off_bv + 2 * (size_t)vm * sizeof(double) + 16;
    char *dmeta = (char *)fokl_scratch(ctx, fokl_ctx::B_META, meta_bytes);
    if (!dmeta) return FOKL_ENOMEM;
    std::vector<char> h(meta_bytes, 0);
    memcpy(h.data(), cols, (size_t)p * sizeof(int32_t));
    if (vm) {
        memcpy(h.data() + off_pos, cand_pos, (size_t)vm * sizeof(int32_t));
        memcpy(h.data() + off_bv, bv0, (size_t)vm * sizeof(double));
        memcpy(h.data() + off_bv + (size_t)vm * sizeof(double), bv1, (size_t)vm * sizeof(double));
    }
    FOKL_CUDA(ctx, cudaMemcpyAsync(dmeta, h.data(), meta_bytes, cudaMemcpyHostToDevice, ctx->stream));
    // models whose packed tableau does not fit one SM's shared memory: whole-device kernel (killbig.cuh); the
    // environment knob moves the switch-over for tests and tools (0 = never)
    bool use_big = !in_smem;
    if (const char *e = getenv("FOKL_KILL_BIG_MIN_P")) use_big = atoi(e) > 0 && p >= atoi(e);
    // the model's eigendecomposition, if the caller has it: the tableau after the forward sweeps is formed from it
    // by every SM (kill_tableau_kernel) and the kill kernels start at their first round
    const bool from_eig = kp->lamb != nullptr && kp->Qt != nullptr && !getenv("FOKL_KILL_NO_EIG");
    const int ldt = (p + 1 + 15) & ~15;
    auto launch_tableau = [&](double *T0, double *w) -> int {
        KillTabParams K;
        K.G = G; K.ldg = ldg; K.Xty = Xty;
        K.cols = reinterpret_cast<const int32_t *>(dmeta);
        K.p = p; K.ldt = ldt; K.lamb = kp->lamb; K.Qt = kp->Qt;
        K.ybar = hyp->sum_y / (double)hyp->n;
        K.cc = hyp->yty - (double)hyp->n * K.ybar * K.ybar;
        K.w = w; K.T0 = T0;
        kill_w_kernel<<<(p + 7) / 8, 256, 0, ctx->stream>>>(K);
        FOKL_LAUNCH_CHECK(ctx);
        const int nt = (p + kTabTile - 1) / kTabTile;
        kill_tableau_kernel<<<nt * (nt + 1) / 2 + 1, 256, 0, ctx->stream>>>(K);
        FOKL_LAUNCH_CHECK(ctx);
        return FOKL_OK;
    };
    if (use_big) {
        // wide model: the tableau lives in L2 and its rows are dealt to one CTA per SM (killbig.cuh)
        const size_t ws = ((size_t)(p + 2) * ldt + 7 * (size_t)ldt) * sizeof(double) + 256;
        char *wcur = (char *)fokl_scratch(ctx, fokl_ctx::B_CAND_A, ws);
        if (!wcur) return FOKL_ENOMEM;
        killb::Params K;
        K.G = G; K.ldg = ldg; K.Xty = Xty;
        K.cols = reinterpret_cast<const int32_t *>(dmeta);
        K.cand_pos = reinterpret_cast<const int32_t *>(dmeta + off_pos);
        K.bv0 = reinterpret_cast<const double *>(dmeta + off_bv);
        K.bv1 = K.bv0 + vm;
        K.p = p; K.vm = vm; K.ldt = ldt;
        K.c.a = hyp->a; K.c.b = hyp->b; K.c.atau = hyp->atau; K.c.btau = hyp->btau;
        K.c.sigsqd0 = hyp->sigsqd0; K.c.tausqd0 = hyp->tausqd0; K.c.yty = hyp->yty; K.c.sum_y = hyp->sum_y;
        K.c.n = (double)hyp->n; K.c.draws = hyp->draws; K.c.from0 = hyp->stat_from0; K.c.from1 = hyp->stat_from1;
        K.in.threshav = kp->threshav; K.in.threshstda = kp->threshstda; K.in.threshstdb = kp->threshstdb;
        K.in.icpt = kp->icpt; K.in.evmin = kp->evmin; K.in.aic_adj = kp->aic_adj; K.in.start = kp->start;
        K.T = carve<double>(wcur, (size_t)(p + 2) * ldt);
        K.pre = from_eig ? 1 : 0;
        if (from_eig) {
            rc = launch_tableau(K.T, carve<double>(wcur, (size_t)ldt));
            if (rc) return rc;
        }
        K.dg = carve<double>(wcur, 2 * (size_t)ldt);
        K.last = carve<double>(wcur, 2 * (size_t)ldt);
        K.bcast = carve<double>(wcur, 2 * (size_t)ldt);
        K.bar = reinterpret_cast<unsigned *>(carve<int>(wcur, 16));
        K.out_i = out_i; K.out_ev = out_ev;
        FOKL_CUDA(ctx, cudaMemsetAsync(K.bar, 0, 16 * sizeof(int), ctx->stream));
        const size_t smem_big = (size_t)((p + 3) & ~1) * sizeof(double) + (size_t)(p + 1) + 16;
        if (smem_big > 48 * 1024)
            FOKL_CUDA(ctx, cudaFuncSetAttribute(killb::kill_loop_big_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_big));
        int occ = 0;
        FOKL_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, killb::kill_loop_big_kernel, killb::kThreads, smem_big));
        if (occ < 1) FOKL_FAIL(ctx, FOKL_ECUDA, "kill_loop: wide-model kernel does not fit an SM");
        const int sms = (ctx->sm_budget > 0 && ctx->sm_budget < ctx->num_sms) ? ctx->sm_budget : ctx->num_sms;
        int grid = std::max(1, std::min(sms, (p + 1 + killb::kWarps - 1) / killb::kWarps));
        if (const char *e = getenv("FOKL_KILL_BIG_GRID")) grid = std::max(1, std::min(sms, atoi(e)));
        void *args[] = {(void *)&K};
        FOKL_CUDA(ctx, cudaLaunchCooperativeKernel((const void *)killb::kill_loop_big_kernel, dim3((unsigned)grid),
                                                   dim3(killb::kThreads), args, smem_big, ctx->stream));
        FOKL_LAUNCH_CHECK(ctx);
        return FOKL_OK;
    }
    double *Tg = nullptr;
    if (!in_smem) {
        Tg = (double *)fokl_scratch(ctx, fokl_ctx::B_CAND_A, (size_t)need * sizeof(double));
        if (!Tg) return FOKL_ENOMEM;
    }
    KillLoopParams P;
    P.G = G; P.ldg = ldg; P.Xty = Xty;
    P.cols = reinterpret_cast<const int32_t *>(dmeta);
    P.cand_pos = reinterpret_cast<const int32_t *>(dmeta + off_pos);
    P.bv0 = reinterpret_cast<const double *>(dmeta + off_bv);
    P.bv1 = P.bv0 + vm;
    P.p = p; P.vm = vm;
    P.c.a = hyp->a; P.c.b = hyp->b; P.c.atau = hyp->atau; P.c.btau = hyp->btau;
    P.c.sigsqd0 = hyp->sigsqd0; P.c.tausqd0 = hyp->tausqd0; P.c.yty = hyp->yty; P.c.sum_y = hyp->sum_y;
    P.c.n = (double)hyp->n; P.c.draws = hyp->draws; P.c.from0 = hyp->stat_from0; P.c.from1 = hyp->stat_from1;
    P.in.threshav = kp->threshav; P.in.threshstda = kp->threshstda; P.in.threshstdb = kp->threshstdb;
    P.in.icpt = kp->icpt; P.in.evmin = kp->evmin; P.in.aic_adj = kp->aic_adj; P.in.start = kp->start;
    P.T_global = Tg; P.out_i = out_i; P.out_ev = out_ev;
    P.T0 = nullptr; P.ldt0 = ldt;
    if (from_eig) {
        char *tcur = (char *)fokl_scratch(ctx, fokl_ctx::B_CAND_B, ((size_t)(p + 2) * ldt + (size_t)ldt) * sizeof(double) + 256);
        if (!tcur) return FOKL_ENOMEM;
        double *T0 = carve<double>(tcur, (size_t)(p + 2) * ldt);
        rc = launch_tableau(T0, carve<double>(tcur, (size_t)ldt));
        if (rc) return rc;
        P.T0 = T0;
    }
    P.smem_doubles = in_smem ? (int)need : 0;
    size_t smem = (size_t)(head + (in_smem ? need : 0)) * sizeof(double);
    FOKL_CUDA(ctx, cudaFuncSetAttribute(kill_loop_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cap));
    kill_loop_kernel<<<1, kKillThreads, smem, ctx->stream>>>(P);
    FOKL_LAUNCH_CHECK(ctx);
    return FOKL_OK;
}
