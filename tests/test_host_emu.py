"""The numerical core of the CUDA kernels (fokl_math.cuh, cand_math.cuh) compiled for the host with a
single-thread team and checked against the oracle -- runs without a GPU."""
import numpy as np
import pytest

import emu
import fokl_oracle as fo
from conftest import load_golden


def test_cubic_basis_bit_exact(cubic_table, phis_cubic):
    g = load_golden('basis_values')
    out, bad = emu.basis_cubic(g['x'], np.arange(1, 49), cubic_table)
    assert bad == 0 and np.array_equal(out, g['cubic'])
    rng = np.random.default_rng(5)
    x = rng.random(50000)
    orders = np.array([1, 2, 3, 7, 20, 48])
    out, _ = emu.basis_cubic(x, orders, cubic_table)
    assert np.array_equal(out, fo.basis_columns(x[:, None], orders[:, None], phis_cubic, fo.CUBIC))


def test_phind_edges():
    x = np.array([0.0, -0.0, 1e-300, 1 / 499, 1.0, 0.999999999, 2 / 499 + 1e-18])
    ph, xs, bad = emu.phind(x)
    rph, rxs = fo.inputs_to_phind(x[:, None])
    assert bad == 0 and np.array_equal(ph, rph[:, 0]) and np.array_equal(xs, rxs[:, 0])
    for bad_x in (1.0001, -0.01, np.nan, 2.0):
        assert emu.phind(np.array([bad_x]))[2] == 1


def test_bernoulli_basis_tolerance(bern_table, phis_bern):
    rng = np.random.default_rng(6)
    x = rng.random(20000)
    orders = np.array([1, 2, 3, 5, 8, 10])
    out = emu.basis_bernoulli(x, orders, bern_table)
    ref = fo.basis_columns(x[:, None], orders[:, None], phis_bern, fo.BERNOULLI)
    scale = np.abs(ref).max(axis=0)
    assert np.all(np.abs(out - ref).max(axis=0) <= 1e-9 * scale)
    assert np.array_equal(out[:, 0], ref[:, 0])
    assert np.mean(out == ref) > 0.98


def bernoulli_order_tolerance(order):
    """Per-order tolerance (fraction of the column scale) for Bernoulli columns against the oracle's libm-`pow` path
    (FR:841-843).  The monomial sum c0 + sum c_k x^k cancels ~0.68 decimal digits per order, so the REFERENCE's own
    float64 result is only this accurate against the exact rational value (SURVEY appendix B: order 12 5e-9, order 16
    8e-6, order 20 1e-2); two correctly-implemented evaluations that round a single power differently cannot agree
    better.  tol(n) = 10^(-15.5 + 0.7 n): 3e-9 at order 10, 1.6e-8 at 11, 3e-2 at 20."""
    return 10.0 ** (-15.5 + 0.7 * order)


def test_bernoulli_all_orders_no_worse_than_the_reference(bern_table, phis_bern):
    """Orders 1-20 (the selection loop can reach ind = len(phis), FR:1747): the device arithmetic (host build of the
    same code) agrees with the oracle within the per-order tolerance, and against the EXACT rational value of the
    polynomial it is as accurate as the reference's own evaluation (within 2x) -- the bound that matters."""
    from fractions import Fraction
    rng = np.random.default_rng(2)
    x = rng.random(4000)
    orders = np.arange(1, 21)
    out = emu.basis_bernoulli(x, orders, bern_table)
    ref = fo.basis_columns(x[:, None], orders[:, None], phis_bern, fo.BERNOULLI)
    xs = [Fraction(float(v)) for v in x[:200]]
    for o in orders:
        scale = np.abs(ref[:, o - 1]).max()
        assert np.abs(out[:, o - 1] - ref[:, o - 1]).max() <= bernoulli_order_tolerance(o) * scale, o
        c = [Fraction(float(v)) for v in phis_bern[o - 1]]
        exact = np.array([float(sum(ck * xx ** k for k, ck in enumerate(c))) for xx in xs])
        err_ref = np.abs(ref[:200, o - 1] - exact).max()
        err_dev = np.abs(out[:200, o - 1] - exact).max()
        assert err_dev <= 2.0 * err_ref + 4e-16 * scale, (o, err_dev, err_ref)


def _problem(phis, n, m, seed):
    rng = np.random.default_rng(seed)
    x = rng.random((n, m))
    y = (np.sin(2 * np.pi * x[:, 0]) + x[:, 0] * x[:, 1] + 0.05 * rng.standard_normal(n))[:, None]
    terms = np.vstack([fo.distinct_perms(p).astype(int) for p in
                       ([1] + [0] * (m - 1), [1, 1] + [0] * (m - 2), [2] + [0] * (m - 1), [2, 1] + [0] * (m - 2))])
    X = np.hstack([np.ones((n, 1)), fo.basis_columns(x, terms, phis, fo.CUBIC)])
    return X, y


@pytest.mark.parametrize('n,m,seed', [(441, 2, 1), (3000, 3, 2)])
def test_candidate_math_matches_oracle(phis_cubic, n, m, seed):
    X, y = _problem(phis_cubic, n, m, seed)
    a = atau = 4
    b, btau = fo.default_b_btau(y, a, atau)
    D = 250
    dtd = y.T.dot(y)
    np.random.seed(seed)
    r = fo.gibbs_from_X(X, y, a, b, atau, btau, D, b / (1 + a), btau / (1 + atau), dtd, literal=True)
    p = X.shape[1]
    np.random.seed(seed)
    z, g1, g2 = fo.draw_variates(p, D, a + 1 + n / 2 + p / 2, atau + (p - 1) / 2)
    var = np.hstack([z, g1[:, None], g2[:, None]])
    hyp = dict(a=a, b=b, atau=atau, btau=btau, sigsqd0=b / (1 + a), tausqd0=btau / (1 + atau),
               yty=float(dtd[0, 0]), sum_y=float(y.sum()), n=n, draws=D)
    e0 = emu.candidate(r['XtX'], r['Xty'], np.arange(p), hyp, rng_mode=0)
    sign = np.sign(np.sum(e0['Q'] * r['Q'], axis=0))
    e = emu.candidate(r['XtX'], r['Xty'], np.arange(p), hyp, rng_mode=1, variates=var, sign_fix=sign)
    assert (e['info'] >> 8) < 40
    assert np.all(np.abs(e['lamb'] - r['Lamb']) <= 1e-12 * r['Lamb'][-1])
    assert abs(e['ev'] - r['ev']) <= 1e-10 * abs(r['ev'])
    assert np.max(np.abs(e['betahat'] - r['betahat'][:, 0])) <= 1e-8 * np.max(np.abs(r['betahat']))
    assert np.max(np.abs(e['betas'] - r['betas'])) <= 1e-8 * np.max(np.abs(r['betas']))
    assert np.allclose(e['sigs'], r['sigs'][:, 0], rtol=1e-9)
    assert np.allclose(e['taus'], r['taus'][:, 0], rtol=1e-8)
    # a sub-model addressed through an index list into the same master Gram
    idx = np.array([0, 2, 3, 5])
    es = emu.candidate(r['XtX'], r['Xty'], idx, hyp, rng_mode=0)
    rs = fo.gibbs_from_X(X[:, idx], y, a, b, atau, btau, 1, 1.0, 1.0, dtd, literal=False,
                         variates=(np.zeros((1, 4)), np.ones(1), np.ones(1)))
    assert abs(es['ev'] - rs['ev']) <= 1e-10 * abs(rs['ev'])


def test_philox_streams_are_standard():
    import ctypes
    L = emu.lib()
    out = np.zeros((4000, 8))
    L.emu_philox_normals(123, 7, 4000, 8, out.ctypes.data)
    assert abs(out.mean()) < 0.02 and abs(out.std() - 1) < 0.02
    out2 = np.zeros((4000, 8))
    L.emu_philox_normals(123, 8, 4000, 8, out2.ctypes.data)
    assert not np.array_equal(out, out2)
    for shape in (0.5, 1.0, 3.5, 5000.5):
        g = np.zeros(20000)
        L.emu_philox_gammas(99, 3, 20000, ctypes.c_double(shape), g.ctypes.data)
        assert abs(g.mean() - shape) < 5 * np.sqrt(shape / 20000) + 1e-12
        assert abs(g.var() - shape) < 0.1 * shape


def test_kill_scores_math_matches_oracle_bic(phis_cubic):
    X, y = _problem(phis_cubic, 2000, 3, 8)
    n, P = X.shape
    G, Xty = X.T @ X, (X.T @ y)[:, 0]
    hyp = dict(a=4, b=1, atau=4, btau=1, sigsqd0=1, tausqd0=1, yty=float((y.T @ y)[0, 0]), sum_y=float(y.sum()), n=n,
               draws=10)
    idx = np.array([0] + list(range(2, P)))
    props = np.arange(1, len(idx))
    ev, bad = emu.kill_scores(G, Xty, idx, props, hyp)
    assert bad == 0

    def bic(cols):
        r = fo.gibbs_from_X(X[:, cols], y, 4, 1, 4, 1, 1, 1.0, 1.0, y.T.dot(y), literal=False,
                            variates=(np.zeros((1, len(cols))), np.ones(1), np.ones(1)))
        return r['ev']
    ref = np.array([bic([c for j, c in enumerate(idx) if j != q]) for q in props] + [bic(list(idx))])
    assert np.max(np.abs(ev - ref) / np.abs(ref)) < 1e-12
    G2 = G.copy()
    G2[:, 2] = G2[:, 1]
    G2[2, :] = G2[1, :]
    assert emu.kill_scores(G2, Xty, np.arange(P), np.array([1]), hyp)[1] == 1


def _literal_kill_loop(X, y, idx, cand_cols, bv0, bv1, thr, evmin, aic_adj, threshstda=0.5, threshstdb=2.0):
    """FR:1666-1690 with one oracle `gibbs` BIC per proposal (no draws needed: BIC is draw-independent)."""
    def bic(cols):
        r = fo.gibbs_from_X(X[:, cols], y, 4, 1, 4, 1, 1, 1.0, 1.0, y.T.dot(y), literal=False,
                            variates=(np.zeros((1, len(cols))), np.ones(1), np.ones(1)))
        return r['ev'] + aic_adj * len(cols)
    killed, acc, calls, evs, tested = [], [], [], [], 0
    for i in range(len(cand_cols)):
        if bv1[i] > threshstdb or (bv1[i] > threshstda and bv0[i] < thr):
            tested += 1
            cols = [c for c in idx if c not in killed and c != cand_cols[i]]
            ev = bic(cols)
            if ev < evmin:
                killed.append(cand_cols[i]); acc.append(i); calls.append(tested); evs.append(ev); evmin = ev
    return acc, calls, evs, tested


@pytest.mark.parametrize('packed', [True, False])
@pytest.mark.parametrize('aic', [False, True])
def test_kill_loop_matches_sequential_oracle_loop(phis_cubic, aic, packed):
    rng = np.random.default_rng(11)
    n, m = 4000, 3
    x = rng.random((n, m))
    y = (np.sin(2 * np.pi * x[:, 0]) + x[:, 1] * x[:, 2] + 0.1 * rng.standard_normal(n))[:, None]
    terms = np.vstack([fo.distinct_perms(p).astype(int) for p in ([1, 0, 0], [1, 1, 0], [2, 0, 0], [2, 1, 0], [1, 1, 1])])
    X = np.hstack([np.ones((n, 1)), fo.basis_columns(x, terms, phis_cubic, fo.CUBIC)])
    P = X.shape[1]
    G, Xty = X.T @ X, (X.T @ y)[:, 0]
    hyp = dict(a=4, b=1, atau=4, btau=1, sigsqd0=1, tausqd0=1, yty=float((y.T @ y)[0, 0]), sum_y=float(y.sum()), n=n,
               draws=10)
    idx = list(range(P))
    vm = 10
    cand_cols = list(rng.permutation(np.arange(P - vm, P)))       # the new terms, in "ascending |mean|" order
    bv0 = np.sort(rng.random(vm))
    bv1 = rng.random(vm) * 3
    aic_adj = (2 - np.log(n)) if aic else 0.0
    full = fo.gibbs_from_X(X, y, 4, 1, 4, 1, 1, 1.0, 1.0, y.T.dot(y), literal=False,
                           variates=(np.zeros((1, P)), np.ones(1), np.ones(1)))['ev'] + aic_adj * P
    icpt, threshav = 2.0, 0.3
    acc, calls, evs, tested = _literal_kill_loop(X, y, idx, cand_cols, bv0, bv1, threshav * icpt, full, aic_adj)
    r = emu.kill_loop(G, Xty, idx, [idx.index(c) for c in cand_cols], bv0, bv1, hyp, threshav=threshav, icpt=icpt,
                      evmin=full, aic_adj=aic_adj, packed=packed)
    assert r['bad'] == 0 and len(acc) > 0
    assert list(r['acc']) == acc and list(r['calls']) == calls and r['tested'] == tested
    assert np.allclose(r['ev'], evs, rtol=1e-11, atol=0)
    # restart from the middle of the loop reproduces the tail
    k = len(acc) // 2
    if k:
        killed = [cand_cols[i] for i in acc[:k]]
        idx2 = [c for c in idx if c not in killed]
        pos2 = [idx2.index(c) if c in idx2 else -1 for c in cand_cols]
        r2 = emu.kill_loop(G, Xty, idx2, pos2, bv0, bv1, hyp, threshav=threshav, icpt=icpt, evmin=evs[k - 1],
                           aic_adj=aic_adj, start=acc[k - 1] + 1, packed=packed)
        assert list(r2['acc']) == acc[k:] and np.allclose(r2['ev'], evs[k:], rtol=1e-11)
    # a duplicated column is reported, not scored
    G2 = G.copy(); G2[:, 2] = G2[:, 1]; G2[2, :] = G2[1, :]
    assert emu.kill_loop(G2, Xty, idx, [idx.index(c) for c in cand_cols], bv0, bv1, hyp, evmin=full,
                         packed=packed)['bad'] == 1


@pytest.mark.parametrize('warps,kchunks,mode', [(16, 1, 1), (15, 4, 1), (15, 16, 1), (15, 8, 0), (16, 16, 0), (8, 8, 1), (15, 1, 2), (12, 1, 2), (15, 16, 2),
                                               (12, 4, 2)])
@pytest.mark.parametrize('p_old,c,cap', [(1, 1, 352), (1, 8, 352), (9, 28, 352), (37, 56, 352), (50, 168, 352),
                                          (71, 168, 352), (3, 5, 32), (130, 40, 64), (20, 300, 128), (400, 17, 352)])
def test_gram_work_plan_covers_the_block_exactly_once(p_old, c, cap, warps, kchunks, mode):
    """K2 plan (csrc/gram_plan.h): every entry of [X_old X_new y]' X_new that fokl_gram_scatter reads (all old / y rows,
    and the new x new part on or above the diagonal) is produced by exactly one fragment of one block of one tile, from
    the right pair of columns, as the sum of the block's k-split work items over disjoint 16-row chunks; tiles respect
    the position and shared-memory-slot budgets."""
    rng = np.random.default_rng(p_old * 1000 + c)
    n = 16 * 2 * kchunks + 5
    A = rng.standard_normal((n, p_old + c + 1))
    rc, out, cover, st = emu.gram_plan(A, p_old, c, cap, warps, kchunks, mode)
    assert rc == 0, rc
    ref = A.T @ A[:, p_old:p_old + c]
    a, j = np.meshgrid(np.arange(p_old + c + 1) - p_old, np.arange(c), indexing='ij')
    needed = ~((a > j) & (a < c))
    assert np.all(cover[needed] == 1)
    assert np.all(cover <= 1)
    got = cover == 1
    assert np.allclose(out[got], ref[got], rtol=1e-12, atol=1e-12)
    assert st['max_positions_per_tile'] <= 4 * warps and st['max_slots'] <= cap and st['max_ksplit'] <= kchunks
    # balanced: no tile is much smaller than the largest unless the slot cap forced a cut
    if p_old + c + 32 <= cap:
        # (every tile rounds its loose fragments up to whole blocks, which can cost one tile more than the quotient)
        assert -(-st['blocks'] // (4 * warps)) <= st['n_tiles'] <= -(-st['blocks'] // (4 * warps)) + 1


@pytest.mark.parametrize('p_old,c', [(28, 168), (51, 168), (58, 168), (64, 56), (37, 56), (14, 56), (8, 28), (400, 1680)])
@pytest.mark.parametrize('warps', [15, 12])
def test_gram_placement_is_even_over_the_sub_partitions(p_old, c, warps):
    """Placement mode 2 (the K2 default): the work items of a tile are dealt evenly over the four SM sub-partitions
    (warp & 3) -- the tensor pipe of a sub-partition is the shared resource -- and a loose / masked item sits in its
    warp's FIRST position whenever the tile has no more of them than busy warps (kernel form FLEX = 1: one 8-load item per
    warp at most)."""
    rng = np.random.default_rng(p_old + c)
    A = rng.random((40, p_old + c + 1))
    rc, out, cover, st = emu.gram_plan(A, p_old, c, cap=240, warps=warps, kchunks=1, mode=2)
    assert rc == 0
    assert st['sp_spread'] <= 1, st
    assert st['flex_late'] == 0, st


def test_gram_k_split_fills_the_cta():
    """A narrow substage (8 new columns against 50 old ones: 4 blocks) is split over the 16-row chunks of a slab so
    that more warps of the CTA have work (two items per block: one per SM sub-partition and block -- measured faster
    than four, profiles/r02_gram_round2.txt); a wide one (168 new columns) is left alone."""
    A = np.random.default_rng(0).standard_normal((300, 50 + 8 + 1))
    rc, _, _, st = emu.gram_plan(A, 50, 8, 352, 16, 16)
    assert rc == 0 and st['max_ksplit'] >= 2 and st['max_positions_per_tile'] >= 8
    A = np.random.default_rng(0).standard_normal((40, 50 + 168 + 1))
    rc, _, _, st = emu.gram_plan(A, 50, 168, 352, 16, 4)
    assert rc == 0 and st['max_ksplit'] == 1


GRAM_SHAPES = [(0, 1), (1, 1), (1, 7), (1, 8), (1, 9), (7, 16), (8, 17), (9, 24), (16, 33), (50, 8), (14, 56), (1, 146),
               (28, 168), (58, 168), (130, 40), (20, 300), (400, 17)]
# plan forms the kernels run: (consumer warps, kchunks, placement mode, loose items, forced pad layout, forced k-split)
GRAM_FORMS = {
    'mb15-place2': (15, 16, 2, True, -1, 0),
    'tma12-place2': (12, 16, 2, True, -1, 0),
    'cpasync16': (16, 1, 2, False, -1, 0),
    'place0-pad0-ks2': (15, 4, 0, True, 0, 2),
    'place1-pad1-ks16': (15, 16, 1, True, 1, 16),
}


@pytest.mark.parametrize('form', list(GRAM_FORMS))
@pytest.mark.parametrize('p_old,c', GRAM_SHAPES)
def test_gram_plan_forms_cover_the_block_exactly_once(p_old, c, form):
    """Every plan form of K2 -- the cp.async plan (no loose items), both pad layouts, forced k-splits, placements 0 / 1 /
    2, 12 and 15 warps -- contiguous, with the new block `gap` columns above the old ones (physical slot_src: the same
    logical block, the same bits) and cross-only (the new x new rows are not produced).  Inside emu_gram_plan: every
    tensor-map box lies inside its tile and fetches each non-padding slot exactly once from its own column of [y | X];
    the bulk-copy kernel's run table (max_slots * 8 bytes = max_slots / 2 runs) is never overrun."""
    warps, kchunks, mode, loose, pad, force_r = GRAM_FORMS[form]
    cap = 352
    rng = np.random.default_rng(p_old * 1000 + c)
    n = 16 * 2 * kchunks + 5
    p = p_old + c
    A = rng.standard_normal((n, p + 1))
    ref = A.T @ A[:, p_old:p]
    a, j = np.meshgrid(np.arange(p + 1) - p_old, np.arange(c), indexing='ij')
    new = (a >= 0) & (a < c)
    needed = ~(new & (a > j))
    base = None
    for gap in (0, 5):
        # physical layout: old | gap (NaN: never read) | new | y
        Ap = np.full((n, p + gap + 1), np.nan)
        Ap[:, :p_old] = A[:, :p_old]
        Ap[:, p_old + gap:] = A[:, p_old:]
        for cross in ((False, True) if p_old > 0 else (False,)):
            rc, out, cover, st = emu.gram_plan(Ap, p_old, c, cap, warps, kchunks, mode, gap=gap, cross_only=cross,
                                               allow_loose=loose, pad_mode=pad, force_r=force_r)
            assert rc == 0, (gap, cross, rc)
            want = needed & ~new if cross else needed
            skipped = new if cross else new & (a // 8 > j // 8)        # whole 8 x 8 fragments below the diagonal
            assert np.all(cover[want] == 1) and np.all(cover[skipped] == 0) and np.all(cover <= 1), (gap, cross)
            assert np.allclose(out[want], ref[want], rtol=1e-12, atol=1e-12)
            assert st['max_slots'] <= cap and st['max_positions_per_tile'] <= 4 * warps
            assert st['max_runs'] <= st['max_slots'] // 2
            assert 1 <= st['min_ksplit'] <= st['max_ksplit'] <= (min(force_r, kchunks) if force_r else kchunks)
            if not loose:
                assert st['loose'] == 0 and st['max_ksplit'] == 1
            if pad >= 0 and ((c + 7) // 8) % 2 == 1:
                assert st['pad'] == pad
            if not cross:
                if gap == 0:
                    base = (out, st)
                else:
                    # the same plan on physical columns: the same logical block, bit for bit
                    assert np.array_equal(out, base[0], equal_nan=True)
                    assert {k: v for k, v in st.items()} == base[1]


def test_gram_plan_reaches_every_kernel_form():
    """The forms the GPU reference tests name (tests/test_gpu_gram_ref.py) exist in the plans of their shapes: the
    all-loose warp form FLEX 2 (p_old = 1, c = 146 at 15 warps; 400 + 17 at 12), a k-split, both pad layouts, every
    box kind and multi-tile plans (the 352-slot cap)."""
    def st(p_old, c, warps=15, kchunks=1, **kw):
        rc, _, _, s = emu.gram_plan(None, p_old, c, 352, warps, kchunks, 2, **kw)
        assert rc == 0
        return s
    assert st(1, 146)['flex2'] > 0 and st(400, 17, warps=12)['flex2'] > 0
    assert st(28, 168)['flex2'] == 0 and st(28, 168)['flex0'] > 0 and st(28, 168)['flex1'] > 0
    assert st(50, 8, kchunks=4)['max_ksplit'] == 4 and st(58, 168)['max_ksplit'] == 1
    assert st(8, 17)['pad'] == 1 and st(16, 33)['pad'] == 0
    s = st(20, 300)
    assert s['box8'] > 0 and s['box32'] > 0 and s['box128'] > 0 and s['n_tiles'] > 1
    assert st(400, 1680)['n_tiles'] == 168
    # the cp.async plan of a wide tile: masked 2 x 2 blocks, no loose ones
    s = st(1, 146, warps=16, allow_loose=False)
    assert s['loose'] == 0 and s['flex1'] + s['flex2'] > 0


@pytest.mark.parametrize('e', [0, 1, 2])
def test_derivative_factor_math_matches_oracle(cubic_table, phis_cubic, bern_table, phis_bern, e):
    """The device's bss_derivatives factor math (fokl_math.cuh: twice_normalised, cubic_basis_d1/d2,
    bernoulli_basis_deriv) against the oracle's Python-scalar evaluation (FR:584-586, 834-847, 780-781)."""
    rng = np.random.default_rng(40 + e)
    x = np.concatenate([rng.random(3000), [0.0, 1.0, 1 / 499, 0.5, 2 / 499, 1 - 2 ** -53]])
    span = 3.7
    # cubic: bit-exact
    orders = np.array([1, 2, 5, 17, 48])
    xe, ph = fo.twice_normalised(x[:, None])
    div = [1, span / 499, (span / 499) ** 2][e]
    ref = np.zeros((len(x), len(orders)))
    for i in range(len(x)):
        for j, o in enumerate(orders):
            c = [phis_cubic[o - 1][q][int(ph[i, 0])] for q in range(4)]
            v = fo.eval_basis_d(c, xe[i, 0], fo.CUBIC, e)
            ref[i, j] = v / div if e else v
    out = emu.deriv_factors(x, orders, cubic_table, e, div, cubic=True)
    assert np.array_equal(out, ref)
    # Bernoulli: the running double-double power is correctly rounded, libm pow() is not always: tolerance
    orders = np.array([1, 2, 3, 5, 8, 10])
    div = [1, span, span ** 2][e]
    ref = np.zeros((300, len(orders)))
    for i in range(300):
        for j, o in enumerate(orders):
            v = fo.eval_basis_d(phis_bern[o - 1], np.float64(x[i]), fo.BERNOULLI, e)
            ref[i, j] = v / div
    out = emu.deriv_factors(x[:300], orders, bern_table, e, div, cubic=False)
    scale = np.max(np.abs(ref), axis=0) + 1e-300
    assert np.max(np.abs(out - ref) / scale) < 1e-9
    assert np.mean(out == ref) > 0.5
