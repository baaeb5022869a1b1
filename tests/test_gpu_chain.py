"""The sampling kernels of the candidate stage (csrc/candidates.cu: cand_variates_kernel, cand_chain_warp_kernel<2|4|8>,
cand_chain_kernel, cand_betas_kernel, cand_stats_kernel) against a long-double restatement of the eigenbasis draw loop
(FR:1519-1548), at every chain variant and width boundary, in mixed batches, at small and odd draw counts, and in the
bstar < 0 branch.

The reference takes the device's own eigenpairs (lamb, Q) of the same launch and forms ct = Q'X'y itself, so that what
is compared is the sampling stage alone; the eigensolvers are bounded by tests/test_gpu_candidates.py.  One comparison
per width against fokl_oracle.gibbs_from_X (LAPACK eigenpairs of the same Gram bits, signs aligned) ties the reference
to the pinned oracle, and free-running (Philox) chains are compared with the host emulation (tests/host_emu) that the
CPU suite's Philox-mode tests rest on.

Bounds.  Against the long-double reference on the device's own eigenpairs: sigs and taus rtol 1e-12, betas 1e-12 of
the largest |beta| (measured on a B200: at most 6e-14 and 4e-15 over every case of this file).  Where the eigenpairs
come from another solver (LAPACK in the oracle, the host Jacobi of the emulation) the suite's chain bounds: rtol 1e-9
and 1e-9 of the largest |beta| (measured: at most 4e-11, at p = 1100).  Column statistics: 1e-12 of the larger of the
statistic and the mean magnitude of the draws it sums (the scale of the rounding of a sum; measured 2e-15), NaN
exactly where numpy gives NaN.

The draw-loop kernel is chosen per launch from the widest chain of the batch (fokl_candidates_eval): one warp with
E = 2, 4, 8 elements per lane for p <= 64, 128, 256, above that the block kernel with 32 ceil(floor(p/2) / 32) threads
(at most 256), whose threads hold elements tid and tid + nthreads in registers and reach the rest through a strided
loop -- for p > 512, and for every p = 64 k + 1.  chain_variant() restates that choice; the test ids name the variant
a case runs in."""
import warnings

import numpy as np
import pytest

import fokl_oracle as fo
from FoKL import _lib

pytestmark = pytest.mark.gpu

A = ATAU = 4
REF_RTOL = 1e-12                 # sigs, taus; betas: x max |betas| -- same eigenpairs as the device
RTOL = 1e-9                      # the same against a chain on another solver's eigenpairs
STAT_RTOL = 1e-12
SEED = 20261020                  # Philox key of the free-running cases
LD = np.longdouble
WIDTHS = (1, 2, 31, 32, 33, 64, 65, 128, 129, 255, 256, 257, 511, 512, 513, 705, 1100)


def chain_variant(pmax):
    """The draw-loop kernel fokl_candidates_eval launches for a batch whose widest chain has pmax columns."""
    if pmax <= 64:
        return 'warpE2'
    if pmax <= 128:
        return 'warpE4'
    if pmax <= 256:
        return 'warpE8'
    nthr = max(32, min(256, 32 * ((pmax // 2 + 31) // 32)))
    return 'block%d%s' % (nthr, '-strided' if pmax > 2 * nthr else '')


def case_id(p):
    # p >= 705: the blocked eigensolver (eigbig.cuh) + cand_ols_kernel factorise the model
    return 'p%d-%s%s' % (p, chain_variant(p), '-eigb' if p >= 705 else '')


def load_problem(engine, pmax, seed):
    """Gaussian design with scaled columns (column 0 = intercept, n = 3 pmax + 50 rows); its Gram goes straight into
    the engine, no basis build, so that any width can be reached."""
    import torch
    rng = np.random.default_rng(seed)
    n = 3 * pmax + 50
    X = rng.standard_normal((n, pmax)) * (1.0 + 3.0 * rng.random(pmax))
    X[:, 0] = 1.0
    k = min(5, pmax)
    y = 2.0 + X[:, :k] @ rng.standard_normal(k) + 0.5 * rng.standard_normal(n)
    G, Xty = X.T @ X, X.T @ y
    cap = max(pmax, 64)
    engine.G = torch.zeros((cap, cap), dtype=torch.float64, device=engine.device)
    engine.Xty = torch.zeros(cap, dtype=torch.float64, device=engine.device)
    engine.G[:pmax, :pmax] = torch.from_numpy(G).to(engine.device)
    engine.Xty[:pmax] = torch.from_numpy(Xty).to(engine.device)
    engine.Gcap = cap
    engine.n_global, engine.sum_y, engine.yty = n, float(y.sum()), float(y @ y)
    return X, y, G, Xty


def hypers(engine, y, D):
    """Device hypers (from the engine's yty / sum_y / n) and the same values as a dict for the references."""
    b, btau = fo.default_b_btau(y, A, ATAU)
    hd = dict(a=A, b=b, atau=ATAU, btau=btau, sigsqd0=b / (1 + A), tausqd0=btau / (1 + ATAU), yty=engine.yty,
              sum_y=engine.sum_y, n=engine.n_global, draws=D)
    return engine.make_hypers(A, b, ATAU, btau, hd['sigsqd0'], hd['tausqd0'], D), hd


def variate_table(rng, p, D, n):
    """D rows of [z_0 .. z_{p-1}, G1, G2]: normal(p), standard_gamma(astar), standard_gamma(atau_star)."""
    astar = A + 1 + n / 2 + p / 2
    atau_star = ATAU + (p - 1) / 2
    return np.hstack([rng.standard_normal((D, p)), rng.standard_gamma(astar, (D, 1)),
                      rng.standard_gamma(atau_star, (D, 1))])


def run(engine, sets, hyp, tables=None, run_chain=None, stream_ids=None):
    """One launch: injected variates if `tables` (one D x (p + 2) table per candidate, idle ones included), else
    Philox streams `stream_ids` of SEED."""
    mode = _lib.RNG_INJECTED if tables is not None else _lib.RNG_PHILOX
    var = None if tables is None else np.concatenate([np.asarray(t).reshape(-1) for t in tables])
    return engine.evaluate(sets, hyp, rng_mode=mode, run_chain=run_chain, seed=SEED, stream_ids=stream_ids,
                           variates=var, want_betas=True, want_eig=True, refine_tol=None)


def device_out(res, c):
    p, D = int(res.p[c]), res.draws
    return dict(
        lamb=res.lamb[res.vec_off[c]:res.vec_off[c] + p].cpu().numpy(),
        Q=res.Q[res.mat_off[c]:res.mat_off[c] + p * p].view(p, p).cpu().numpy().T,      # columns = eigenvectors
        sigs=res.sigs[D * c:D * (c + 1)].cpu().numpy(), taus=res.taus[D * c:D * (c + 1)].cpu().numpy(),
        betas=res.betas_of(c).cpu().numpy(), stats=res.stats_of(c).cpu().numpy(), info=int(res.info[c]),
        ev=float(res.ev[c]))


def ref_chain(lamb, Q, xty, hd, table):
    """FR:1519-1548 in the eigenbasis, in long double and in the reference's operation order (fokl_oracle.gibbs_from_X,
    literal=False), on the given eigenpairs (Q: columns = eigenvectors) with injected variates.
    Returns float64 (betas, sigs, taus)."""
    p, D = len(lamb), table.shape[0]
    lam = np.asarray(lamb, dtype=LD)
    Ql = np.asarray(Q, dtype=LD)
    ct = Ql.T @ np.asarray(xty, dtype=LD)
    z = np.asarray(table[:, :p], dtype=LD)
    g1, g2 = np.asarray(table[:, p], dtype=LD), np.asarray(table[:, p + 1], dtype=LD)
    one, two, half = LD(1), LD(2), LD(0.5)
    b, btau, yty = LD(hd['b']), LD(hd['btau']), LD(hd['yty'])
    sig, tau = LD(hd['sigsqd0']), LD(hd['tausqd0'])
    gam = np.zeros((D, p), dtype=LD)
    sigs = np.zeros(D, dtype=LD)
    taus = np.zeros(D, dtype=LD)
    for k in range(D):
        d = one / (lam + one / tau)
        g = d * ct + np.sqrt(sig) * np.sqrt(d) * z[k]
        gam[k] = g
        s1 = np.sum(lam * g * g)
        s2 = np.sum(g * ct)
        s3 = np.sum(g * g)
        bstar = b + half * (s1 - two * s2 + yty + s3 / tau)
        sig = LD(np.nan) if bstar < 0 else one / ((one / bstar) * g1[k])
        sigs[k] = sig
        btau_star = (one / (two * sig)) * s3 + btau
        tau = one / ((one / btau_star) * g2[k])
        taus[k] = tau
    return (gam @ Ql.T).astype(np.float64), sigs.astype(np.float64), taus.astype(np.float64)


def chain_errors(dev, ref):
    b_ref, s_ref, t_ref = ref
    es = np.max(np.abs(dev['sigs'] - s_ref) / np.abs(s_ref))
    et = np.max(np.abs(dev['taus'] - t_ref) / np.abs(t_ref))
    eb = np.max(np.abs(dev['betas'] - b_ref)) / np.max(np.abs(b_ref))
    return es, et, eb


def check_chain(dev, ref, what, rtol=REF_RTOL):
    es, et, eb = chain_errors(dev, ref)
    print('%s: sigs %.2e taus %.2e betas %.2e' % (what, es, et, eb))
    assert es <= rtol and et <= rtol and eb <= rtol, (what, es, et, eb)


def numpy_stats(bt, D):
    """Rows of stats_of(c) restated with numpy on the returned draws (FR:1656-1658)."""
    h0, h1 = int(np.ceil(D / 2)), int(np.ceil(D / 2 + 1))
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)            # mean / std of an empty slice: NaN
        with np.errstate(all='ignore'):
            want = np.vstack([bt[h1:].mean(axis=0), bt[h1:].std(axis=0), bt[h0:].mean(axis=0)])
            scale = np.vstack([np.abs(bt[h1:]).mean(axis=0)] * 2 + [np.abs(bt[h0:]).mean(axis=0)])
    return want, scale


def check_stats(st, bt, D, what):
    want, scale = numpy_stats(bt, D)
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(st), nan), (what, 'NaN pattern', st[:, :4], want[:, :4])
    if nan.all():
        return
    err = np.abs(st - want)[~nan] / np.maximum(np.abs(want), scale)[~nan]
    print('%s: stats %.2e' % (what, err.max()))
    assert err.max() <= STAT_RTOL, (what, err.max())


def oracle_chain(X, y, cols, G, Xty, hd, table, Q_dev):
    """fokl_oracle.gibbs_from_X (eigenbasis form) on the same Gram bits and variates, its LAPACK eigenvectors' signs
    carried to the normals (z_j -> s_j z_j pairs them with the device's eigenvectors)."""
    from scipy.linalg import eigh
    p, D = len(cols), table.shape[0]
    Gs, xs = G[np.ix_(cols, cols)], Xty[cols]
    _, Qo = eigh(Gs)
    s = np.sign(np.sum(Q_dev * Qo, axis=0))
    r = fo.gibbs_from_X(X[:, cols], y[:, None], hd['a'], hd['b'], hd['atau'], hd['btau'], D, hd['sigsqd0'],
                        hd['tausqd0'], np.array([[hd['yty']]]), literal=False,
                        variates=(table[:, :p] * s, table[:, p], table[:, p + 1]), gram=(Gs, xs))
    return r['betas'], r['sigs'][:, 0], r['taus'][:, 0]


# ---- 1. every chain variant and width boundary ----------------------------------------------------------------------
@pytest.mark.parametrize('p', WIDTHS, ids=case_id)
def test_chain_at_every_variant_matches_long_double_reference(engine, p):
    D = 67
    X, y, G, Xty = load_problem(engine, p, seed=p)
    hyp, hd = hypers(engine, y, D)
    table = variate_table(np.random.default_rng(1000 + p), p, D, hd['n'])
    cols = list(range(p))
    dev = device_out(run(engine, [cols], hyp, tables=[table]), 0)
    assert dev['info'] & 0xff == 0, dev['info']
    check_chain(dev, ref_chain(dev['lamb'], dev['Q'], Xty, hd, table), case_id(p))
    check_chain(dev, oracle_chain(X, y, cols, G, Xty, hd, table, dev['Q']), case_id(p) + ' vs oracle', RTOL)
    check_stats(dev['stats'], dev['betas'], D, case_id(p))


# ---- 2. mixed batches -----------------------------------------------------------------------------------------------
def _column_sets(rng, sizes, pmax):
    """Prefixes, and for every other model a scattered column list (intercept first)."""
    sets = []
    for j, p in enumerate(sizes):
        if j % 2 and 1 < p < pmax:
            sets.append([0] + sorted(int(c) for c in rng.choice(np.arange(1, pmax), size=p - 1, replace=False)))
        else:
            sets.append(list(range(p)))
    return sets


@pytest.mark.parametrize('sizes', [(1, 33, 200), (1, 64, 65, 300, 600)],
                         ids=lambda s: '-'.join(map(str, s)) + '-' + chain_variant(max(s)))
def test_mixed_batch_matches_reference(engine, sizes):
    D = 67
    pmax = max(sizes)
    X, y, G, Xty = load_problem(engine, pmax, seed=sum(sizes))
    hyp, hd = hypers(engine, y, D)
    rng = np.random.default_rng(7)
    sets = _column_sets(rng, sizes, pmax)
    tables = [variate_table(rng, len(s), D, hd['n']) for s in sets]
    res = run(engine, sets, hyp, tables=tables)
    for c, cols in enumerate(sets):
        dev = device_out(res, c)
        what = 'batch %s, model %d (p %d)' % (chain_variant(pmax), c, len(cols))
        assert dev['info'] & 0xff == 0, (what, dev['info'])
        check_chain(dev, ref_chain(dev['lamb'], dev['Q'], Xty[cols], hd, tables[c]), what)
        check_stats(dev['stats'], dev['betas'], D, what)


@pytest.mark.parametrize('mode', ['injected', 'philox'])
def test_batch_with_idle_candidates(engine, mode):
    """run_chain = [1, 0, 1, 0, 1]: injected tables are addressed per candidate (D (vec_off + 2 c)), Philox tables per
    chain (D (gam_off + 2 chain_idx)).  The idle candidates' injected tables are NaN, so a chain that read one would
    show it; their statistics stay unwritten."""
    import emu
    D = 67
    sizes = (40, 120, 90, 3, 20)
    run_chain = [1, 0, 1, 0, 1]
    X, y, G, Xty = load_problem(engine, max(sizes), seed=41)
    hyp, hd = hypers(engine, y, D)
    rng = np.random.default_rng(43)
    sets = _column_sets(rng, sizes, max(sizes))
    if mode == 'injected':
        tables = [variate_table(rng, len(s), D, hd['n']) if on else np.full((D, len(s) + 2), np.nan)
                  for s, on in zip(sets, run_chain)]
        res = run(engine, sets, hyp, tables=tables, run_chain=run_chain)
    else:
        sids = [101, 102, 103, 104, 105]
        res = run(engine, sets, hyp, run_chain=run_chain, stream_ids=sids)
    for c, cols in enumerate(sets):
        dev = device_out(res, c)
        what = '%s, model %d (p %d)' % (mode, c, len(cols))
        if not run_chain[c]:
            assert np.all(dev['stats'] == 0.0), what
            continue
        if mode == 'injected':
            ref = ref_chain(dev['lamb'], dev['Q'], Xty[cols], hd, tables[c])
        else:
            want = emu.candidate(G, Xty, cols, hd, rng_mode=_lib.RNG_PHILOX, seed=SEED, stream=sids[c])
            ref = (want['betas'], want['sigs'], want['taus'])
        assert dev['info'] & 0xff == 0, (what, dev['info'])
        check_chain(dev, ref, what, REF_RTOL if mode == 'injected' else RTOL)
        check_stats(dev['stats'], dev['betas'], D, what)


def test_warp_kernel_draws_do_not_depend_on_the_batch(engine, monkeypatch):
    """A model's chain, betas and statistics are the same bits alone (E = 2) and inside wider warp-kernel batches
    (E = 4, 8): lanes past p add exact zeros to the same two partial sums.  The block kernel (a batch with a chain wider
    than 256) rounds differently -- another reduction tree and other reciprocal / square-root instructions -- so there
    only the reference bound holds: a model's draws are batch-invariant among warp-kernel batches only.
    FOKL_EIGJ_CS=1 keeps the model's eigensolver launch the same in every batch (p = 40 alone in its cluster class,
    512 threads), so that the eigenpairs are the same bits too."""
    monkeypatch.setenv('FOKL_EIGJ_CS', '1')
    D = 67
    X, y, G, Xty = load_problem(engine, 300, seed=3)
    hyp, hd = hypers(engine, y, D)
    rng = np.random.default_rng(5)
    tab = {p: variate_table(rng, p, D, hd['n']) for p in (40, 100, 230, 300)}
    outs = {}
    for batch in ((40,), (40, 100), (40, 100, 230), (40, 300)):
        res = run(engine, [list(range(p)) for p in batch], hyp, tables=[tab[p] for p in batch])
        outs[chain_variant(max(batch))] = device_out(res, 0)
    alone = outs['warpE2']
    for name in ('warpE4', 'warpE8'):
        got = outs[name]
        assert np.array_equal(got['lamb'], alone['lamb']) and np.array_equal(got['Q'], alone['Q']), name
        for key in ('sigs', 'taus', 'betas', 'stats'):
            assert np.array_equal(got[key], alone[key]), (name, key)
    for name, dev in outs.items():
        check_chain(dev, ref_chain(dev['lamb'], dev['Q'], Xty[:40], hd, tab[40]), 'p 40 in a %s batch' % name)


# ---- 3. draw counts -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('D', [1, 2, 3, 4, 63, 64, 65])
@pytest.mark.parametrize('p', [5, 70, 300], ids=case_id)
def test_draw_counts(engine, p, D):
    """D = 1, 2, 3: the two-row variate prefetch runs past the chain, and one or both statistic windows
    (rows ceil(D/2) .. and ceil(D/2 + 1) ..) are empty -- their statistics are NaN, as numpy's; D = 63 ... 65: the
    64-row tiles of the betas kernel."""
    X, y, G, Xty = load_problem(engine, p, seed=500 + p)
    hyp, hd = hypers(engine, y, D)
    table = variate_table(np.random.default_rng(D), p, D, hd['n'])
    dev = device_out(run(engine, [list(range(p))], hyp, tables=[table]), 0)
    what = '%s D %d' % (case_id(p), D)
    assert dev['info'] & 0xff == 0, (what, dev['info'])
    check_chain(dev, ref_chain(dev['lamb'], dev['Q'], Xty, hd, table), what)
    check_stats(dev['stats'], dev['betas'], D, what)


# ---- 4. statistics at every column-CTA edge -------------------------------------------------------------------------
@pytest.mark.parametrize('sizes', [(31,), (32,), (33,), (95,), (257,), (31, 32, 33, 95, 257)],
                         ids=lambda s: 'p' + '-'.join(map(str, s)))
def test_stats_at_column_block_edges(engine, sizes):
    """cand_stats_kernel: 32 columns per CTA, 16 row lanes; an odd draw count leaves the lanes unequal rows."""
    D = 1001
    X, y, G, Xty = load_problem(engine, max(sizes), seed=900 + max(sizes))
    hyp, hd = hypers(engine, y, D)
    res = run(engine, [list(range(p)) for p in sizes], hyp, stream_ids=list(range(len(sizes))))
    for c, p in enumerate(sizes):
        dev = device_out(res, c)
        assert dev['info'] & 0xff == 0
        check_stats(dev['stats'], dev['betas'], D, 'p %d in %s' % (p, sizes))


# ---- 5. Philox mode against the host emulation ----------------------------------------------------------------------
@pytest.mark.parametrize('p', [w for w in WIDTHS if w <= 513], ids=case_id)
def test_philox_chain_equals_host_emulation(engine, p):
    """Same seed, same stream ids, canonical eigenvector signs: the device's free-running chain is the host emulation's
    (emu_candidate: the same cand_math.cuh on one thread) -- the link that carries the CPU suite's Philox-mode tests
    over to the device.  Two streams of one seed give different draws."""
    import emu
    D = 67
    X, y, G, Xty = load_problem(engine, p, seed=p)
    hyp, hd = hypers(engine, y, D)
    cols = list(range(p))
    sids = [7, (1 << 40) + 8]                  # the high word of a stream id selects a stream as well
    res = run(engine, [cols, cols], hyp, stream_ids=sids)
    devs = [device_out(res, c) for c in range(2)]
    assert not np.array_equal(devs[0]['betas'], devs[1]['betas'])
    assert not np.array_equal(devs[0]['sigs'], devs[1]['sigs'])
    for c, sid in enumerate(sids):
        want = emu.candidate(G, Xty, cols, hd, rng_mode=_lib.RNG_PHILOX, seed=SEED, stream=sid)
        dev = devs[c]
        assert dev['info'] & 0xff == 0 and want['info'] & 0xff == 0
        check_chain(dev, (want['betas'], want['sigs'], want['taus']), '%s stream %d' % (case_id(p), sid), RTOL)
        assert abs(dev['ev'] - want['ev']) <= 1e-9 * abs(want['ev'])


# ---- 6. bstar < 0 ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('p', [20, 100, 200, 300, 513], ids=case_id)
def test_negative_bstar_gives_nan_from_that_draw_on(engine, p):
    """yty below Xty' G^-1 Xty drives the bracket of FR:1538 negative: sig^2 is NaN from the first such draw on, and so
    is everything after it, as in the oracle's eigenbasis branch (fokl_oracle.py:443-447); bit 0 of info is set.  The
    draws before it still match the reference.  The offset keeps the first draw's bracket positive (its sig^2 = sigsqd0
    noise term outweighs it) so that the switch happens inside the chain."""
    D = 20
    X, y, G, Xty = load_problem(engine, p, seed=600 + p)
    b, _ = fo.default_b_btau(y, A, ATAU)
    engine.yty = float(Xty @ np.linalg.solve(G, Xty)) - 2 * b - 0.25 * p * b / (1 + A)
    hyp, hd = hypers(engine, y, D)
    table = variate_table(np.random.default_rng(p), p, D, hd['n'])
    dev = device_out(run(engine, [list(range(p))], hyp, tables=[table]), 0)
    b_ref, s_ref, t_ref = ref_chain(dev['lamb'], dev['Q'], Xty, hd, table)
    bad = np.flatnonzero(np.isnan(s_ref))
    assert len(bad) and 0 < bad[0] < D - 1, bad                  # the case reaches the branch inside the chain
    k = int(bad[0])
    assert dev['info'] & 1, dev['info']
    assert np.all(np.isnan(dev['sigs'][k:])) and np.all(np.isnan(dev['taus'][k:]))
    assert np.all(np.isnan(dev['betas'][k + 1:]))
    assert not np.any(np.isnan(dev['betas'][:k + 1]))
    check_chain(dict(sigs=dev['sigs'][:k], taus=dev['taus'][:k], betas=dev['betas'][:k + 1]),
                (b_ref[:k + 1], s_ref[:k], t_ref[:k]), '%s first bad draw %d' % (case_id(p), k))
