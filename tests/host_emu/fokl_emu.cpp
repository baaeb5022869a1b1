// fokl_emu.cpp -- host emulation of the numerical core of the CUDA kernels (TEST INFRASTRUCTURE).
//
// Compiles fokl-gpy_b200/csrc/{fokl_math,cand_math}.cuh as plain C++ with a single-thread "Team"
// (nlane = nwarp = 1, barriers are no-ops) so the CPU test-suite can check the kernel math
// (basis evaluation, Jacobi eigensolver, betahat/BIC, eigenbasis Gibbs chain) against the oracle
// without a GPU.  Build: g++ -O2 -ffp-contract=off -shared -fPIC.
#include <cstdint>
#include <cstring>
#include <vector>
#include "../../fokl-gpy_b200/csrc/cand_math.cuh"
#include "../../fokl-gpy_b200/csrc/update_math.cuh"

using namespace fokl;

extern "C" {

// cubic factor values: out[i * n_ord + s] = phi_{orders[s]}(x[i]);  tab [n_orders][n_piece][4]
int emu_basis_cubic(const double *x, int64_t n, const int32_t *orders, int n_ord, const double *tab, int n_piece,
                    double *out)
{
    int bad = 0;
    for (int64_t i = 0; i < n; ++i) {
        int ph;
        double xs, x2, x3;
        if (!phind_xsm(x[i], n_piece, ph, xs)) bad = 1;
        square_cube(xs, x2, x3);
        for (int s = 0; s < n_ord; ++s) {
            const double *c = tab + ((size_t)(orders[s] - 1) * n_piece + ph) * 4;
            out[i * n_ord + s] = cubic_basis(c[0], c[1], c[2], c[3], xs, x2, x3);
        }
    }
    return bad;
}

int emu_phind(const double *x, int64_t n, int n_piece, int32_t *ph, double *xsm)
{
    int bad = 0;
    for (int64_t i = 0; i < n; ++i)
        if (!phind_xsm(x[i], n_piece, ph[i], xsm[i])) bad = 1;
    return bad;
}

// bernoulli factor values; tab [n_orders][row_len]
void emu_basis_bernoulli(const double *x, int64_t n, const int32_t *orders, int n_ord, const double *tab, int row_len,
                         double *out)
{
    std::vector<double> pw(row_len + 2);
    for (int64_t i = 0; i < n; ++i)
        for (int s = 0; s < n_ord; ++s) {
            int d = orders[s];
            powers_dd(x[i], d, pw.data());
            out[i * n_ord + s] = bernoulli_basis(tab + (size_t)(d - 1) * row_len, d + 1, pw.data());
        }
}

// bss_derivatives factor values (FR:770-781): out[i][s] = e-th derivative (e = 0, 1, 2) of the basis function of order
// orders[s] at the twice-normalised input (cubic) / at x (Bernoulli), divided by div when e > 0.
int emu_deriv_cubic(const double *x, int64_t n, const int32_t *orders, int n_ord, const double *tab, int n_piece, int e,
                    double div, double *out)
{
    int bad = 0;
    for (int64_t i = 0; i < n; ++i) {
        int ph;
        double xs, x2, x3;
        if (!phind_xsm(x[i], n_piece, ph, xs)) bad = 1;
        xs = twice_normalised(x[i], n_piece, ph);
        square_cube(xs, x2, x3);
        for (int s = 0; s < n_ord; ++s) {
            const double *c = tab + ((size_t)(orders[s] - 1) * n_piece + ph) * 4;
            double v = e == 0 ? cubic_basis(c[0], c[1], c[2], c[3], xs, x2, x3)
                     : e == 1 ? cubic_basis_d1(c[1], c[2], c[3], xs, x2) / div : cubic_basis_d2(c[2], c[3], xs) / div;
            out[i * n_ord + s] = v;
        }
    }
    return bad;
}

void emu_deriv_bernoulli(const double *x, int64_t n, const int32_t *orders, int n_ord, const double *tab, int row_len,
                         int e, double div, double *out)
{
    for (int64_t i = 0; i < n; ++i)
        for (int s = 0; s < n_ord; ++s) {
            int d = orders[s];
            if (e == 0) {
                std::vector<double> pw(row_len + 2);
                powers_dd(x[i], d, pw.data());
                out[i * n_ord + s] = bernoulli_basis(tab + (size_t)(d - 1) * row_len, d + 1, pw.data());
            } else {
                out[i * n_ord + s] = bernoulli_basis_deriv(tab + (size_t)(d - 1) * row_len, d + 1, x[i], e) / div;
            }
        }
}

struct emu_hypers {
    double a, b, atau, btau, sigsqd0, tausqd0, yty, sum_y;
    int64_t n;
    int32_t draws, from0, from1, reserved;
};

// One candidate, same stages as cand_eig_kernel + cand_chain_kernel + cand_betas_kernel.
// rng_mode 0: no chain; 1: injected variates [D][p+2]; 2: philox(seed, stream)
int emu_candidate(const double *G, int64_t ldg, const double *Xty, const int32_t *idx, int p, const emu_hypers *h,
                  int rng_mode, uint64_t seed, uint64_t stream, const double *variates, const double *sign_fix,
                  double *ev, double *betahat, double *lamb, double *Q, double *betas, double *sigs, double *taus,
                  int32_t *info)
{
    Team t;
    t.tid = 0; t.nthr = 1; t.lane = 0; t.nlane = 1; t.warp = 0; t.nwarp = 1;
    std::vector<double> W((size_t)p * p), V((size_t)p * p), lam_raw(p), ct(p), scratch(p), red(16);
    std::vector<int> perm(p);
    volatile int flag = 0;
    for (int e = 0; e < p * p; ++e) {
        int col = e / p, row = e - col * p;
        W[e] = G[(int64_t)idx[row] * ldg + idx[col]];
    }
    const double tol = 2.220446049250313e-16 * (2.0 * sqrt((double)p) + 6.0);
    // device order: Cholesky + Jacobi on the factor; the two-matrix Jacobi only if the Gram is not positive definite
    std::vector<double> L((size_t)p * p, 0.0);
    for (int e = 0; e < p * p; ++e) {
        int col = e / p, row = e - col * p;
        if (row >= col) L[e] = W[e];
    }
    int sweeps;
    int chol_failed = 0;
    if (cholesky_lower(t, L.data(), p)) {
        sweeps = jacobi_w_sweeps(t, L.data(), p, p, 40, tol, &flag);
        eig_finish_w(t, L.data(), p, p, lam_raw.data(), perm.data(), lamb, Q);
    } else {
        chol_failed = 2;
        sweeps = jacobi_eigh(t, W.data(), V.data(), p, p, 40, tol, &flag);
        eig_finish(t, W.data(), V.data(), p, p, lam_raw.data(), perm.data(), lamb, Q);
    }
    CandConst k;
    k.a = h->a; k.b = h->b; k.atau = h->atau; k.btau = h->btau; k.sigsqd0 = h->sigsqd0; k.tausqd0 = h->tausqd0;
    k.yty = h->yty; k.sum_y = h->sum_y; k.n = (double)h->n; k.draws = h->draws; k.from0 = h->from0; k.from1 = h->from1;
    *ev = ols_and_bic(t, G, ldg, Xty, idx, p, lamb, Q, k, ct.data(), betahat, scratch.data(), red.data());
    *info = (sweeps << 8) | chol_failed;
    if (rng_mode == 0) return 0;
    const int D = h->draws;
    std::vector<double> gam((size_t)D * p), table;
    const double *var = variates;
    if (rng_mode == 2) {
        Philox g;
        g.k0 = (uint32_t)seed; g.k1 = (uint32_t)(seed >> 32);
        table.resize((size_t)D * (p + 2));
        for (int d = 0; d < D; ++d)
            for (int e = 0; e < p + 2; ++e)
                table[(size_t)d * (p + 2) + e] = philox_variate(g, (uint32_t)stream, (uint32_t)(stream >> 32) & 0x7fffffffu, d, e,
                                                                p, chain_astar(k, p), chain_atau_star(k, p));
        var = table.data();
    }
    int bad = gibbs_chain(t, p, lamb, ct.data(), k, var, sign_fix, gam.data(), sigs, taus, red.data(), rng_mode == 2);
    if (bad) *info |= 1;
    for (int d = 0; d < D; ++d)
        for (int i = 0; i < p; ++i) {
            double s = 0.0;
            for (int r = 0; r < p; ++r) s += gam[(size_t)d * p + r] * Q[(size_t)r * p + i];
            betas[(size_t)d * p + i] = s;
        }
    return 0;
}

// kill_scores on the host: ev_out has k + 1 entries; returns the not-positive-definite flag
int emu_kill_scores(const double *G, int64_t ldg, const double *Xty, const int32_t *idx, int p, const int32_t *props,
                    int k, const emu_hypers *h, double *ev_out)
{
    Team t;
    t.tid = 0; t.nthr = 1; t.lane = 0; t.nlane = 1; t.warp = 0; t.nwarp = 1;
    std::vector<double> L((size_t)p * p), z(p), beta(p), wbuf(p), red(16);
    volatile int flag = 0;
    CandConst c;
    c.a = h->a; c.b = h->b; c.atau = h->atau; c.btau = h->btau; c.sigsqd0 = h->sigsqd0; c.tausqd0 = h->tausqd0;
    c.yty = h->yty; c.sum_y = h->sum_y; c.n = (double)h->n; c.draws = h->draws; c.from0 = h->from0; c.from1 = h->from1;
    return kill_scores(t, G, ldg, Xty, idx, p, props, k, c, L.data(), z.data(), beta.data(), wbuf.data(), ev_out, &flag,
                       red.data());
}

// kill_loop on the host: params = {threshav, threshstda, threshstdb, icpt, evmin, aic_adj}; returns the error flag
int emu_kill_loop(const double *G, int64_t ldg, const double *Xty, const int32_t *idx, int p, const int32_t *cand_pos,
                  const double *bv0, const double *bv1, int vm, const emu_hypers *h, const double *params, int start,
                  int packed, int32_t *out_i, double *out_ev)
{
    Team t;
    t.tid = 0; t.nthr = 1; t.lane = 0; t.nlane = 1; t.warp = 0; t.nwarp = 1;
    std::vector<double> T((size_t)(p + 1) * (p + 1));
    int sh[4];
    CandConst c;
    c.a = h->a; c.b = h->b; c.atau = h->atau; c.btau = h->btau; c.sigsqd0 = h->sigsqd0; c.tausqd0 = h->tausqd0;
    c.yty = h->yty; c.sum_y = h->sum_y; c.n = (double)h->n; c.draws = h->draws; c.from0 = h->from0; c.from1 = h->from1;
    KillLoopIn in;
    in.threshav = params[0]; in.threshstda = params[1]; in.threshstdb = params[2]; in.icpt = params[3];
    in.evmin = params[4]; in.aic_adj = params[5]; in.start = start;
    std::vector<double> rowbuf(p + 1);
    return kill_loop(t, G, ldg, Xty, idx, p, cand_pos, bv0, bv1, vm, c, in, T.data(), out_i, out_ev, sh, rowbuf.data(), packed != 0);
}

void emu_philox_normals(uint64_t seed, uint64_t stream, int draws, int p, double *out)
{
    Philox g;
    g.k0 = (uint32_t)seed; g.k1 = (uint32_t)(seed >> 32);
    for (int d = 0; d < draws; ++d)
        for (int e = 0; e < p; ++e)
            out[(size_t)d * p + e] = philox_normal(g, (uint32_t)stream, (uint32_t)(stream >> 32) & 0x7fffffffu, d, e);
}

void emu_philox_gammas(uint64_t seed, uint64_t stream, int draws, double shape, double *out)
{
    Philox g;
    g.k0 = (uint32_t)seed; g.k1 = (uint32_t)(seed >> 32);
    for (int d = 0; d < draws; ++d)
        out[d] = philox_gamma(g, (uint32_t)stream, (uint32_t)(stream >> 32) & 0x7fffffffu, d, 0u, shape);
}

// The update sampler (csrc/update_math.cuh) with one host thread.  mdl: [mode, po, pn, draws] ints; par: [astar,
// atau_star, b, btau, sigsqd0, yty, squerr, n].  variates: injected table or null (Philox seed / stream).
int emu_update_chain(const int32_t *mdl, const double *par, const double *lam_o, const double *c_o, const double *t_o,
                     const double *m_o, const double *lam_n, const double *c_n, const double *M, const double *Mt,
                     const double *K, const double *W, const double *variates, uint64_t seed, uint64_t stream,
                     double *gam_o, double *gam_n, double *sigs, double *taus, double *lik)
{
    Team t;
    t.tid = 0; t.nthr = 1; t.lane = 0; t.nlane = 1; t.warp = 0; t.nwarp = 1;
    UpdModel m;
    m.mode = mdl[0]; m.po = mdl[1]; m.pn = mdl[2]; m.draws = mdl[3];
    m.astar = par[0]; m.atau_star = par[1]; m.b = par[2]; m.btau = par[3]; m.sigsqd0 = par[4]; m.yty = par[5];
    m.squerr = par[6]; m.n = par[7];
    UpdArrays A;
    A.lam_o = lam_o; A.c_o = c_o; A.t_o = t_o; A.m_o = m_o; A.lam_n = lam_n; A.c_n = c_n; A.M = M; A.Mt = Mt; A.K = K; A.W = W;
    UpdVariates V;
    V.table = variates;
    V.g.k0 = (uint32_t)seed; V.g.k1 = (uint32_t)(seed >> 32);
    V.s_lo = (uint32_t)stream; V.s_hi = (uint32_t)(stream >> 32) & 0x7fffffffu;
    V.w = m.po + m.pn; V.astar = m.astar; V.atau_star = m.atau_star;
    std::vector<double> sh(update_scratch_doubles(m.po, m.pn, 1));
    return update_chain(t, m, A, V, gam_o, gam_n, sigs, taus, lik, sh.data());
}

}  // extern "C"

// ---- K2 work plan (csrc/gram_plan.h): host walk of tiles / blocks / fragments exactly as the Gram kernels +
// gram_reduce_kernel use them.  A is [n][p + gap + 1] row-major in the PHYSICAL column order of fokl_gram_update_ex
// (old columns, `gap` unused columns, new columns, y last) and may be null (plan checks and statistics only); out is
// (p + 1) x c in the logical order old | new | y and must be pre-filled by the caller; cover (same shape, int) counts
// how many times each entry was written.  pad_mode -1 / allow_loose 1 / force_r 0 are the defaults of gram_make_plan
// and gram_plan_place.
#include "../../fokl-gpy_b200/csrc/gram_plan.h"
extern "C" int emu_gram_plan(const double *A, int64_t n, int p_old, int c, int max_slots_cap, int warps, int kchunks, int mode,
                             int gap, int cross_only, int allow_loose, int pad_mode, int force_r, double *out, int32_t *cover,
                             int32_t *stats /* see kGramStats below */)
{
    // stats: 0 n_tiles, 1 max_slots, 2 total_blocks, 3 max_positions_per_tile, 4 max_ksplit, 5 sp_spread, 6 flex_late,
    // 7 pad layout, 8 loose items, 9-11 warps in FLEX form 0 / 1 / 2, 12 min_ksplit, 13-15 boxes of 8 / 32 / 128 columns,
    // 16 largest run count of the bulk-copy kernel's run table in one tile
    const int p = p_old + c;
    const int W = p + gap + 1;                       // columns of A
    auto logical = [&](int src) { return src < 0 ? -1 : (src >= p_old + gap ? src - gap : src); };
    GramPlan pl = gram_make_plan(p_old, c, max_slots_cap, warps, gap, cross_only != 0, pad_mode, allow_loose != 0);
    int pad_used = pad_mode;
    if (pad_used < 0) {
        // the layout the default chose: rebuild both and compare
        pad_used = 0;
        if (((c + 7) / 8) % 2 == 1) {
            GramPlan b = gram_make_plan(p_old, c, max_slots_cap, warps, gap, cross_only != 0, 1, allow_loose != 0);
            if (b.slot_src == pl.slot_src && b.blocks.size() == pl.blocks.size()) pad_used = 1;
        }
    }
    gram_plan_place(pl, warps, kchunks, mode, force_r);
    const int kTileBlocks = gram_tile_blocks(warps);
    for (int k = 0; k < 17; ++k) stats[k] = 0;
    stats[0] = (int32_t)pl.tiles.size();
    stats[1] = pl.max_slots;
    stats[7] = pad_used;
    stats[12] = 1 << 30;
    for (const GramTileMeta &tm : pl.tiles) {
        if (tm.n_blk > stats[3]) stats[3] = tm.n_blk;
        if (tm.ksplit > stats[4]) stats[4] = tm.ksplit;
        if (tm.ksplit < stats[12]) stats[12] = tm.ksplit;
        if (tm.n_blk > kTileBlocks || tm.n_slots > max_slots_cap || (tm.n_slots % 8) != 0) return -1;
        if (tm.ksplit < 1 || tm.ksplit > kchunks || (kchunks % tm.ksplit) != 0) return -5;
        for (int s = 0; s < tm.n_slots; ++s) {
            const int src = pl.slot_src[tm.slot_off + s];
            if (src < -1 || src >= W || (src >= p_old && src < p_old + gap)) return -10;     // never a gap column
            if (logical(src) != pl.slot_arow[tm.slot_off + s]) return -10;
        }
        // positions of a warp are filled from its first one (the kernel stops at the first hole)
        for (int w = 0; w < warps; ++w) {
            bool hole = false;
            int owned = 0;
            for (int q = w; q < tm.n_blk; q += warps) {
                const bool h = pl.blocks[tm.blk_off + q].mask == 0;
                if (hole && !h) return -6;
                hole = hole || h;
                owned += h ? 0 : 1;
            }
            if (owned > gram_warp_cap(warps, w)) return -8;
        }
        // placement statistics: items per SM sub-partition (warp & 3), loose / masked items outside a warp's first
        // position, the consumer form of every busy warp (gram_kernel_mb / gram_kernel_tma: FLEX)
        {
            int sl[4] = {0, 0, 0, 0}, busy = 0, flex_total = 0, flex_late = 0;
            for (int w = 0; w < warps; ++w) {
                int owned = 0, flex = 0;
                for (int q = w, b = 0; q < tm.n_blk && b < kGramBlocksPerWarp; q += warps, ++b) {
                    const GramBlockMeta &bm = pl.blocks[tm.blk_off + q];
                    if (bm.mask == 0) break;
                    ++owned;
                    if (bm.loose || bm.mask != 15) {
                        ++flex_total;
                        flex_late += b > 0;
                        flex = b == 0 ? (flex > 1 ? flex : 1) : 2;
                    }
                }
                sl[w & 3] += owned;
                busy += owned > 0;
                if (owned > 0) ++stats[9 + flex];
            }
            int mx = 0, mn = 1 << 30;
            for (int q = 0; q < 4; ++q) {
                int cap_q = 0;
                for (int w = q; w < warps; w += 4) cap_q += gram_warp_cap(warps, w);
                mx = sl[q] > mx ? sl[q] : mx;
                if (sl[q] < cap_q) mn = sl[q] < mn ? sl[q] : mn;       // a full sub-partition cannot take more
            }
            if (mn != (1 << 30) && mx - mn > stats[5]) stats[5] = mx - mn;
            if (flex_total <= busy) stats[6] += flex_late;
        }
        // the bulk-copy kernel's run table (gram_kernel_mb): same walk
        {
            int n_runs = 0, prev = -2;
            for (int sl = 0; sl < tm.n_slots; ++sl) {
                const int src = pl.slot_src[tm.slot_off + sl];
                if (src < 0) { prev = -2; continue; }
                if (!(src == prev + 1 && src != p + gap && n_runs > 0)) ++n_runs;
                prev = src;
            }
            if (n_runs > stats[16]) stats[16] = n_runs;
        }
        // TMA boxes: inside the tile, every non-padding slot fetched exactly once from its own column of [y | X]
        {
            auto xcol = [&](int src) { return src == p + gap ? 0 : src + 1; };
            std::vector<int> got(tm.n_slots, 0);
            for (int b = 0; b < tm.n_box; ++b) {
                const GramBoxMeta &bx = pl.boxes[tm.box_off + b];
                if (bx.kind < 0 || bx.kind >= kGramBoxKinds || bx.ncols != kGramBoxCols[bx.kind]) return -11;
                if (bx.slot0 < 0 || bx.slot0 % 8 != 0 || bx.slot0 + bx.ncols > tm.n_slots) return -11;
                ++stats[13 + bx.kind];
                for (int i = 0; i < bx.ncols; ++i) {
                    const int src = pl.slot_src[tm.slot_off + bx.slot0 + i];
                    if (src < 0) continue;
                    if (xcol(src) != bx.xcol0 + i) return -12;
                    ++got[bx.slot0 + i];
                }
            }
            for (int s = 0; s < tm.n_slots; ++s)
                if (got[s] != (pl.slot_src[tm.slot_off + s] >= 0 ? 1 : 0)) return -13;
        }
        // the kernels: every item accumulates its own chunks; gram_reduce_kernel: the head walks the chain
        std::vector<double> part((size_t)tm.n_blk * 256, 0.0);
        for (int q = 0; q < tm.n_blk; ++q) {
            const GramBlockMeta bm = pl.blocks[tm.blk_off + q];
            if (bm.mask == 0) continue;
            if (bm.loose) ++stats[8];
            if (bm.loose && !allow_loose) return -9;
            for (int f = 0; f < 4; ++f)
                if (bm.la[f] + 8 > tm.n_slots || bm.lb[f] + 8 > tm.n_slots) return -2;
            if (!bm.loose)
                for (int f = 0; f < 4; ++f)
                    if (bm.la[f] != bm.a_slot + 8 * (f >> 1) || bm.lb[f] != bm.b_slot + 8 * (f & 1)) return -9;
            if (bm.mask > 15 || bm.phase >= tm.ksplit) return -4;
            if (bm.next >= tm.n_blk || (bm.next >= 0 && pl.blocks[tm.blk_off + bm.next].phase != bm.phase + 1)) return -7;
            if ((bm.next < 0) != (bm.phase == tm.ksplit - 1)) return -7;
            if (!A) continue;
            for (int f = 0; f < 4; ++f)
                for (int idx = 0; idx < 64; ++idx) {
                    if (!(bm.mask >> f & 1)) continue;
                    const int ca = pl.slot_src[tm.slot_off + bm.la[f] + (idx >> 3)];
                    const int cb = pl.slot_src[tm.slot_off + bm.lb[f] + (idx & 7)];
                    if (ca < 0 || cb < 0) continue;
                    double s = 0.0;
                    for (int64_t i = 0; i < n; ++i)
                        if ((int)((i / 16) % tm.ksplit) == bm.phase) s += A[i * W + ca] * A[i * W + cb];
                    part[(size_t)q * 256 + f * 64 + idx] = s;
                }
        }
        for (int q = 0; q < tm.n_blk; ++q) {
            const GramBlockMeta bm = pl.blocks[tm.blk_off + q];
            if (bm.mask == 0 || bm.phase != 0) continue;
            ++stats[2];
            for (int f = 0; f < 4; ++f)
                for (int idx = 0; idx < 64; ++idx) {
                    if (!(bm.mask >> f & 1)) continue;
                    const int sa = tm.slot_off + bm.la[f] + (idx >> 3);
                    const int sb = tm.slot_off + bm.lb[f] + (idx & 7);
                    const int arow = pl.slot_arow[sa], bcol = pl.slot_bcol[sb];
                    if (arow < 0 || bcol < 0) continue;
                    const int ca = logical(pl.slot_src[sa]), cb = logical(pl.slot_src[sb]);
                    if (ca != arow || cb != p_old + bcol || cb >= p) return -3;
                    double s = 0.0;
                    int links = 0;
                    for (int qq = q; qq >= 0; qq = pl.blocks[tm.blk_off + qq].next) {
                        const GramBlockMeta it = pl.blocks[tm.blk_off + qq];
                        if (it.a_slot != bm.a_slot || it.b_slot != bm.b_slot || it.mask != bm.mask) return -8;
                        s += part[(size_t)qq * 256 + f * 64 + idx];
                        if (++links > tm.ksplit) return -8;
                    }
                    if (links != tm.ksplit) return -8;
                    out[(size_t)arow * c + bcol] = s;
                    cover[(size_t)arow * c + bcol] += 1;
                }
        }
    }
    return 0;
}
