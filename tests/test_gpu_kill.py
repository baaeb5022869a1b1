"""The kill-loop kernels (csrc/cand_math.cuh kill_loop_t in kill_loop_kernel, csrc/killbig.cuh kill_loop_big_kernel,
csrc/candidates.cu kill_w_kernel + kill_tableau_kernel, kill_scores_kernel) against a long-double restatement of the
loop (FR:1666-1690) on the same inputs, at every tableau form, width boundary and grid shape.

ref_kill_loop() builds the centred tableau [G x; x' s] of fokl::kill_loop_t from the float64 Gram bits G[cols][cols],
Xty, yty, sum_y and n, runs the p forward sweeps and then the proposal scan of each round (proposal rule, strict
evt < evmin, the BIC with aic_adj (pa - 1)), one reverse sweep per accepted kill -- all in np.longdouble and following
its own decisions.  The unmarked tests tie it to the literal one-BIC-per-proposal loop of the oracle
(test_host_emu._literal_kill_loop) and to least squares solved from scratch; they run without a GPU.

Forms (kill_form() restates the dispatch of fokl_kill_loop; the test ids name the form a case runs in):
  packed   one CTA, lower-triangle tableau in shared memory: (p+1)(p+2)/2 + 2 + ((p+2)&~1) doubles fit the opt-in
           shared memory (p <= 238 on a B200);
  full     one CTA, full tableau in global memory (L2): FOKL_KILL_BIG_MIN_P=0 and p >= 239;
  big-gN   kill_loop_big_kernel on N CTAs (min(SMs, ceil((p+1)/16)), or FOKL_KILL_BIG_GRID); '-xR' when a warp owns up
           to R rows of the tableau (p + 1 > 16 N);
  -eig     the tableau after the forward sweeps formed from the model's eigendecomposition (kill_w_kernel,
           kill_tableau_kernel), which every full model of a fit uses.

Bounds.  BIC crosses zero, so the bound is on the SSE behind each BIC: |SSE_dev - SSE_ref| <= 1e-12 s_c, s_c = yty -
n ybar^2, checked as |ev_dev - ev_ref| SSE_ref / (n s_c) (first order in the error of log SSE).  Graded designs:
GRADED_C cond(A) eps s_c, cond(A) the 2-norm condition number of G[cols][cols].  Decisions (acc, calls, tested, n_acc,
bad) exactly.  Every fixture asserts that no proposal's BIC lies within 1e-6 of the threshold it is compared with (for
the graded designs: within 10x what the bound allows), so that the decisions are well defined in float64.
Measured on a B200 (1000 W power limit) over every case of this file: packed 1.3e-15, full 6.5e-16, big 1.3e-15 of
s_c; from the eigendecomposition at most 2.3e-14 up to p = 400, 1.6e-13 at p = 705 and 2.8e-13 at p = 1100 (the
eigenpairs' own rounding, which grows with p, dominates there); graded designs (cond 1e7, and 5e9 / 2e10 next to
the usable flag's threshold) 2.2e-4 cond eps s_c, whence GRADED_C = 1e-3; kill_scores 4.4e-16."""
import functools

import numpy as np
import pytest

LD = np.longdouble
EPS = np.finfo(np.float64).eps
SSE_RTOL = 1e-12                 # x s_c
GRADED_C = 1e-3                  # x cond(A) eps s_c
MARGIN = 1e-6
THRESHAV, THRESHSTDA, THRESHSTDB, ICPT = 0.3, 0.5, 2.0, 2.0
B200_SMEM_OPTIN, B200_SMS = 232448, 148       # what the test ids assume; test_dispatch_* checks the device
WIDTHS = (2, 3, 31, 32, 33, 63, 64, 65, 127, 128, 129, 226, 237, 238, 239, 255, 256, 257, 400, 705, 1100)
FORCED_P = (33, 129, 238, 257, 705)


# ---- the long-double reference ----------------------------------------------------------------------------------------
def _sweep(T, k, sign, blk=128):
    """One pivot of the sweep operator on the lower triangle of the symmetric tableau T (long double): off the pivot
    cross T_ij -= c_i c_j / d, on it sign c_i / d, at the pivot -1 / d (c = row k, d = T_kk)."""
    ld = T.shape[0]
    ck = np.concatenate([T[k, :k + 1], T[k + 1:, k]])
    inv = 1 / ck[k]
    v = ck * inv
    for r0 in range(0, ld, blk):
        r1 = min(ld, r0 + blk)
        T[r0:r1, :r1] -= np.multiply.outer(v[r0:r1], ck[:r1])
    T[k, :k + 1] = sign * v[:k + 1]
    T[k + 1:, k] = sign * v[k + 1:]
    T[k, k] = -inv


def bic(sse, n, pa, aic_adj):
    """The kernels' BIC of a model of pa columns with residual sum of squares sse, in long double."""
    n = LD(n)
    return LD(pa) * np.log(n) - 2 * (-(n / 2) * np.log(sse / n) - (n - 1) / 2) + LD(aic_adj) * LD(pa)


def proposed(bv0, bv1, threshav=THRESHAV, threshstda=THRESHSTDA, threshstdb=THRESHSTDB, icpt=ICPT):
    """The proposal rule in float64, as the kernels evaluate it."""
    bv0, bv1 = np.asarray(bv0, dtype=np.float64), np.asarray(bv1, dtype=np.float64)
    return (bv1 > threshstdb) | ((bv1 > threshstda) & (bv0 < threshav * icpt))


def forward_tableau(G, Xty, cols, yty, sum_y, n):
    """(tableau after the p forward sweeps, bad): the centred tableau of fokl::kill_loop_t, swept in long double; bad = 1
    if a pivot fails the kernels' test d > 1e-11 G_kk."""
    cols = np.asarray(cols)
    p = len(cols)
    ybar = LD(sum_y) / LD(n)
    T = np.zeros((p + 1, p + 1), dtype=LD)
    T[:p, :p] = np.asarray(G[np.ix_(cols, cols)], dtype=LD)
    T[p, :p] = np.asarray(Xty[cols], dtype=LD) - ybar * np.asarray(G[cols[0], cols], dtype=LD)
    T[p, p] = LD(yty) - LD(n) * ybar * ybar
    for k in range(p):
        if not T[k, k] > LD(1e-11) * LD(G[cols[k], cols[k]]):
            return T, 1
        _sweep(T, k, 1)
    return T, 0


def ref_kill_loop(G, Xty, cols, yty, sum_y, n, cand_pos, bv0, bv1, evmin=None, aic_adj=0.0, start=0,
                  threshav=THRESHAV, threshstda=THRESHSTDA, threshstdb=THRESHSTDB, icpt=ICPT, T=None):
    """FR:1666-1690 on the sweep tableau in long double.  evmin None: the full model's own BIC (with aic_adj p),
    rounded to float64 as the kernels get it.  Returns dict(n_acc, tested, bad, acc, calls, ev, sse, evmin, s_c,
    sse_full, sse0 (SSE of the model without position q, q = 0 .. p - 1, before any kill), margin (smallest
    |evt - evmin| of every comparison made))."""
    p = len(cols)
    if T is None:
        T, bad = forward_tableau(G, Xty, cols, yty, sum_y, n)
    else:
        T, bad = T.copy(), 0
    ybar = LD(sum_y) / LD(n)
    out = dict(n_acc=0, tested=0, bad=bad, acc=[], calls=[], ev=[], sse=[], margin=np.inf,
               s_c=float(LD(yty) - LD(n) * ybar * ybar))
    if bad:
        return out
    out['sse_full'] = T[p, p]
    with np.errstate(divide='ignore', invalid='ignore'):
        out['sse0'] = T[p, p] + T[p, :p] ** 2 / -np.diagonal(T)[:p]
    if evmin is None:
        evmin = float(bic(T[p, p], n, p, aic_adj))
    out['evmin'] = evmin
    prop = proposed(bv0, bv1, threshav, threshstda, threshstdb, icpt)
    cand_pos = np.asarray(cand_pos)
    vm = len(cand_pos)
    evmin_l, pa, cur = LD(evmin), p, start
    while cur < vm:
        ii = np.flatnonzero(prop[cur:vm]) + cur
        q = cand_pos[ii]
        tqq, tqy = T[q, q], T[p, q]
        if not np.all(tqq < 0):
            out['bad'] = 2
            break
        sse = T[p, p] + tqy * tqy / -tqq
        evt = bic(sse, n, pa - 1, aic_adj)
        below = np.flatnonzero(evt < evmin_l)
        upto = len(ii) if len(below) == 0 else below[0] + 1
        if upto:
            out['margin'] = min(out['margin'], float(np.min(np.abs(evt[:upto] - evmin_l))))
        out['tested'] += int(upto)
        if len(below) == 0:
            break
        h = below[0]
        out['acc'].append(int(ii[h]))
        out['calls'].append(out['tested'])
        out['ev'].append(evt[h])
        out['sse'].append(sse[h])
        evmin_l = evt[h]
        _sweep(T, int(q[h]), -1)
        pa -= 1
        cur = int(ii[h]) + 1
    out['n_acc'] = len(out['acc'])
    return out


# ---- fixtures ---------------------------------------------------------------------------------------------------------
class Problem:
    """A Gaussian design with scaled columns (column 0 = intercept, n = 3 p + 50 rows) of gcap columns, a model `cols`
    of p of them (the intercept first; 'scattered': gcap = 1.5 p and cols a sorted sample), y depending on every 7th
    model column, and candidates at vm = 3 (p - 1) / 4 model positions (1 and p - 1 among them) in a random order,
    with bv0 ascending and bv1 in [0, 3): both branches of the proposal rule and neither.
    kind 'graded': the non-intercept model columns are W = U S V' (U orthonormal and orthogonal to the intercept, V a
    random rotation), so G[cols][cols] = diag(n, V S^2 V') has eigenvalues n and n geomspace(1, 1 / cond)."""

    def __init__(self, p, seed, layout='scattered', kind='gauss', cond=None, n=None, signal=7, vm=None, bv='mixed'):
        rng = np.random.default_rng(seed)
        self.p = p
        gcap = max(p, (3 * p + 1) // 2) if layout == 'scattered' else p
        n = 3 * p + 50 if n is None else n
        X = rng.standard_normal((n, gcap)) * (1.0 + 3.0 * rng.random(gcap))
        X[:, 0] = 1.0
        if layout == 'scattered' and p > 1:
            cols = [0] + sorted(int(c) for c in rng.choice(np.arange(1, gcap), size=p - 1, replace=False))
        else:
            cols = list(range(p))
        if kind == 'graded' and p > 1:
            Z = rng.standard_normal((n, p - 1))
            Z -= Z.mean(axis=0)
            U, _ = np.linalg.qr(Z)
            V, _ = np.linalg.qr(rng.standard_normal((p - 1, p - 1)))
            s = np.sqrt(n * np.geomspace(1.0, 1.0 / cond, p - 1))
            X[:, cols[1:]] = (U * s) @ V.T
        self.cols = cols
        sig = cols[signal::signal] if signal else []
        coef = rng.choice([-1.0, 1.0], size=len(sig)) * (0.5 + rng.random(len(sig)))
        y = 2.0 + X[:, sig] @ coef + 0.5 * rng.standard_normal(n)
        self.X, self.y, self.n = X, y, n
        self.G, self.Xty = X.T @ X, X.T @ y
        self.yty, self.sum_y = float(y @ y), float(y.sum())
        vm = max(min(p - 1, 2), (3 * (p - 1)) // 4) if vm is None else min(vm, p - 1)
        if vm >= 2:
            mid = rng.choice(np.arange(2, p - 1), size=vm - 2, replace=False) if vm > 2 else np.array([], int)
            pos = np.concatenate([[1, p - 1], mid])
        else:
            pos = np.array([1, p - 1][:vm])
        self.cand_pos = [int(c) for c in rng.permutation(pos)]
        self.bv0 = np.sort(rng.random(vm))
        self.bv1 = rng.random(vm) * 3.0 if bv == 'mixed' and vm > 2 else np.full(vm, 2.5)     # (tiny lists: all proposed)
        self.cond = np.linalg.cond(self.G[np.ix_(cols, cols)]) if kind == 'graded' else None

    def ref(self, **kw):
        return ref_kill_loop(self.G, self.Xty, self.cols, self.yty, self.sum_y, self.n, self.cand_pos, self.bv0,
                             self.bv1, **kw)


@functools.lru_cache(maxsize=None)
def problem(p, seed, layout='scattered', kind='gauss', cond=None, n=None, signal=7, vm=None, bv='mixed'):
    return Problem(p, seed, layout, kind, cond, n, signal, vm, bv)


@functools.lru_cache(maxsize=None)
def reference(key, aic=False, start=0):
    """The reference of problem(*key) (computed once per fixture, reused by every form it runs in)."""
    pr = problem(*key)
    aic_adj = (2.0 - np.log(pr.n)) if aic else 0.0
    return pr.ref(aic_adj=aic_adj, start=start)


def sse_error(ev_dev, ref, n):
    """Largest |SSE_dev - SSE_ref| / s_c behind the device's BICs after each kill (first order in the log)."""
    if not len(ref['ev']):
        return 0.0
    ev_ref = np.asarray(ref['ev'], dtype=LD)
    sse = np.asarray(ref['sse'], dtype=LD)
    err = np.abs(np.asarray(ev_dev, dtype=LD) - ev_ref) * sse / (LD(n) * LD(ref['s_c']))
    return float(np.max(err))


def check_decisions(got, ref, what):
    assert got['bad'] == ref['bad'], (what, got['bad'], ref['bad'])
    assert got['n_acc'] == ref['n_acc'], (what, got['n_acc'], ref['n_acc'])
    assert got['tested'] == ref['tested'], (what, got['tested'], ref['tested'])
    assert list(got['acc']) == ref['acc'], what
    assert list(got['calls']) == ref['calls'], what


def check_against_reference(got, ref, pr, what, bound=SSE_RTOL):
    check_decisions(got, ref, what)
    err = sse_error(got['ev'], ref, pr.n)
    print('%s: %d kills, %d tested, SSE error %.2e s_c' % (what, ref['n_acc'], ref['tested'], err))
    assert err <= bound, (what, err, bound)
    return err


def check_margin(ref, what, margin=MARGIN):
    assert ref['margin'] >= margin, (what, 'near tie: change the seed', ref['margin'])


# ---- dispatch -----------------------------------------------------------------------------------------------------------
def kill_form(p, smem_optin=B200_SMEM_OPTIN, sms=B200_SMS, big_min_p=None, grid=None, eig=False):
    """The kernel fokl_kill_loop runs for a p-column model (FOKL_KILL_BIG_MIN_P = big_min_p, FOKL_KILL_BIG_GRID =
    grid)."""
    packed = (p + 1) * (p + 2) // 2 <= smem_optin // 8 - (2 + ((p + 2) & ~1))
    use_big = not packed if big_min_p is None else (big_min_p > 0 and p >= big_min_p)
    if use_big:
        g = max(1, min(sms, -(-(p + 1) // 16)))
        if grid is not None:
            g = max(1, min(sms, grid))
        rows = -(-(p + 1) // (16 * g))
        name = 'big-g%d' % g + ('-x%d' % rows if rows > 1 else '')
    else:
        name = 'packed' if packed else 'full'
    return name + ('-eig' if eig else '')


def device_form(p, **kw):
    import torch
    pr = torch.cuda.get_device_properties(0)
    return kill_form(p, pr.shared_memory_per_block_optin, pr.multi_processor_count, **kw)


# ---- CPU: the reference against the oracle's literal loop and least squares ------------------------------------------
@pytest.mark.parametrize('aic', [False, True], ids=['bic', 'aic'])
@pytest.mark.parametrize('start', [0, 3])
@pytest.mark.parametrize('seed', [1, 2, 3])
def test_reference_equals_literal_oracle_loop(seed, start, aic):
    """Decisions, calls, tested and BICs of the reference equal the oracle's one-`gibbs`-BIC-per-proposal loop;
    start > 0 is the literal loop over the candidates from `start` on."""
    from test_host_emu import _literal_kill_loop
    pr = Problem(14, seed, layout='scattered', signal=3, vm=13)
    aic_adj = (2.0 - np.log(pr.n)) if aic else 0.0
    ref = pr.ref(aic_adj=aic_adj, start=start)
    prop = proposed(pr.bv0, pr.bv1)
    branch_b = pr.bv1 > THRESHSTDB
    assert np.any(prop & ~branch_b) and np.any(branch_b) and np.any(~prop)      # each branch, and neither
    cand_cols = [pr.cols[q] for q in pr.cand_pos]
    acc, calls, evs, tested = _literal_kill_loop(pr.X, pr.y[:, None], pr.cols, cand_cols[start:], pr.bv0[start:],
                                                 pr.bv1[start:], THRESHAV * ICPT, ref['evmin'], aic_adj)
    assert ref['bad'] == 0 and ref['n_acc'] > 0
    assert ref['acc'] == [a + start for a in acc] and ref['calls'] == calls and ref['tested'] == tested
    assert ref['n_acc'] < len(prop[start:].nonzero()[0])                       # some proposals were rejected
    np.testing.assert_allclose(np.asarray(ref['ev'], dtype=np.float64), evs, rtol=1e-11, atol=0)
    check_margin(ref, 'seed %d' % seed)


@pytest.mark.parametrize('p,layout', [(60, 'scattered'), (129, 'contiguous')])
def test_reference_bic_equals_least_squares_from_scratch(p, layout):
    """After every kill the reference's SSE and BIC are those of the reduced model solved from scratch."""
    pr = problem(p, p, layout)
    ref = reference((p, p, layout))
    assert ref['bad'] == 0 and ref['n_acc'] > 2
    killed = []
    yc = pr.y - pr.y.mean()
    s_c = float(yc @ yc)
    for k, i in enumerate(ref['acc']):
        killed.append(pr.cols[pr.cand_pos[i]])
        cols = [c for c in pr.cols if c not in killed]
        beta = np.linalg.lstsq(pr.X[:, cols], pr.y, rcond=None)[0]
        r = pr.y - pr.X[:, cols] @ beta
        sse = float(r @ r)
        assert abs(float(ref['sse'][k]) - sse) <= 1e-11 * s_c, (k, float(ref['sse'][k]), sse)
        ev = float(bic(LD(sse), pr.n, len(cols), 0.0))
        assert abs(float(ref['ev'][k]) - ev) <= 1e-11 * max(abs(ev), pr.n), (k, float(ref['ev'][k]), ev)


def test_reference_restart_reproduces_the_tail():
    """start = acc[k-1] + 1 on the reduced model (killed candidates at position -1) continues the loop."""
    pr = problem(90, 5)
    ref = reference((90, 5))
    k = ref['n_acc'] // 2
    assert k >= 2
    r2 = restart_reference(pr, ref, k)
    assert r2['acc'] == ref['acc'][k:]
    assert r2['calls'] == [c - ref['calls'][k - 1] for c in ref['calls'][k:]]
    np.testing.assert_allclose(np.asarray(r2['sse'], dtype=np.float64), np.asarray(ref['sse'][k:], dtype=np.float64),
                               rtol=1e-14)


@pytest.mark.parametrize('p,packed', [(33, True), (129, True), (129, False)])
def test_host_build_of_the_kernel_math_matches_reference(p, packed):
    """fokl::kill_loop_t compiled for the host (one thread, tests/host_emu) against the reference: the shared
    per-entry arithmetic of every device form, without a GPU."""
    import emu
    pr = problem(p, p)
    ref = reference((p, p))
    hd = dict(a=4, b=1, atau=4, btau=1, sigsqd0=1, tausqd0=1, yty=pr.yty, sum_y=pr.sum_y, n=pr.n, draws=10)
    got = emu.kill_loop(pr.G, pr.Xty, pr.cols, pr.cand_pos, pr.bv0, pr.bv1, hd, threshav=THRESHAV, icpt=ICPT,
                        evmin=ref['evmin'], packed=packed)
    check_against_reference(got, ref, pr, 'host p%d %s' % (p, 'packed' if packed else 'full'))


def restart_reference(pr, ref, k):
    cols2, pos2 = restart_inputs(pr, ref, k)
    return ref_kill_loop(pr.G, pr.Xty, cols2, pr.yty, pr.sum_y, pr.n, pos2, pr.bv0, pr.bv1,
                         evmin=float(ref['ev'][k - 1]), start=ref['acc'][k - 1] + 1)


def restart_inputs(pr, ref, k):
    killed = {pr.cols[pr.cand_pos[i]] for i in ref['acc'][:k]}
    cols2 = [c for c in pr.cols if c not in killed]
    pos2 = [cols2.index(pr.cols[q]) if pr.cols[q] in cols2 else -1 for q in pr.cand_pos]
    return cols2, pos2


# ---- GPU ----------------------------------------------------------------------------------------------------------------
def load(engine, pr):
    import torch
    cap = max(pr.G.shape[0], 64)
    engine.G = torch.zeros((cap, cap), dtype=torch.float64, device=engine.device)
    engine.Xty = torch.zeros(cap, dtype=torch.float64, device=engine.device)
    engine.G[:pr.G.shape[0], :pr.G.shape[0]] = torch.from_numpy(pr.G).to(engine.device)
    engine.Xty[:pr.G.shape[0]] = torch.from_numpy(pr.Xty).to(engine.device)
    engine.Gcap = cap
    engine.n_global, engine.sum_y, engine.yty = pr.n, pr.sum_y, pr.yty
    return engine.make_hypers(4, 1, 4, 1, 1, 1, 10)


def run_kill(engine, monkeypatch, pr, hyp, ref, eig=None, big_min_p=None, grid=None, no_eig=False, cols=None,
             cand_pos=None, start=0, aic_adj=0.0, evmin=None):
    for name, val in (('FOKL_KILL_BIG_MIN_P', big_min_p), ('FOKL_KILL_BIG_GRID', grid),
                      ('FOKL_KILL_NO_EIG', 1 if no_eig else None)):
        if val is None:
            monkeypatch.delenv(name, raising=False)
        else:
            monkeypatch.setenv(name, str(val))
    try:
        return engine.kill_loop_launch(pr.cols if cols is None else cols,
                                       pr.cand_pos if cand_pos is None else cand_pos, pr.bv0, pr.bv1, hyp, THRESHAV,
                                       THRESHSTDA, THRESHSTDB, ICPT, ref['evmin'] if evmin is None else evmin,
                                       aic_adj, start, eig=eig).finish()
    finally:
        for name in ('FOKL_KILL_BIG_MIN_P', 'FOKL_KILL_BIG_GRID', 'FOKL_KILL_NO_EIG'):
            monkeypatch.delenv(name, raising=False)


def eigen(engine, cols, hyp):
    res = engine.evaluate([list(cols)], hyp, want_eig=True, refine_tol=None)
    assert int(res.info[0]) & 6 == 0, int(res.info[0])
    return res.lamb, res.Q


def same_bits(a, b, what):
    for key in ('bad', 'n_acc', 'tested'):
        assert a[key] == b[key], (what, key, a[key], b[key])
    for key in ('acc', 'calls', 'ev'):
        assert np.array_equal(a[key], b[key]), (what, key)


def width_id(p):
    return 'p%d-%s' % (p, kill_form(p))


@pytest.mark.gpu
def test_dispatch_switches_at_238_on_a_b200():
    """The forms the test ids name are the ones a B200 runs: packed up to p = 238, the big kernel from 239 on."""
    import torch
    pr = torch.cuda.get_device_properties(0)
    if 'B200' not in pr.name:
        pytest.skip('the ids name the forms of a B200; this device is a %s' % pr.name)
    assert pr.shared_memory_per_block_optin == B200_SMEM_OPTIN and pr.multi_processor_count == B200_SMS
    assert device_form(238) == 'packed' and device_form(239) == 'big-g15'
    assert device_form(238, big_min_p=0) == 'packed' and device_form(239, big_min_p=0) == 'full'
    for p in WIDTHS:
        assert device_form(p) == kill_form(p)


@pytest.mark.gpu
@pytest.mark.parametrize('p', WIDTHS, ids=width_id)
def test_kill_loop_at_every_width_matches_reference(engine, monkeypatch, p):
    """Default form, sequential and from the eigendecomposition, on a scattered column list of a Gram 1.5 p wide;
    the other tableau form (big below the switch, the single-CTA full form above it) gives the same bits."""
    pr = problem(p, p)
    ref = reference((p, p))
    check_margin(ref, width_id(p))
    hyp = load(engine, pr)
    seq = run_kill(engine, monkeypatch, pr, hyp, ref)
    check_against_reference(seq, ref, pr, width_id(p))
    eig = run_kill(engine, monkeypatch, pr, hyp, ref, eig=eigen(engine, pr.cols, hyp))
    check_against_reference(eig, ref, pr, width_id(p) + '-eig')
    other = dict(big_min_p=2) if kill_form(p) == 'packed' else dict(big_min_p=0)
    same_bits(run_kill(engine, monkeypatch, pr, hyp, ref, **other), seq, '%s vs %s' % (width_id(p), kill_form(p, **other)))


@pytest.mark.gpu
@pytest.mark.parametrize('p', (33, 238, 257, 705), ids=lambda p: 'p%d-%s-contiguous' % (p, kill_form(p)))
def test_contiguous_model_matches_reference(engine, monkeypatch, p):
    pr = problem(p, 50 + p, 'contiguous')
    ref = reference((p, 50 + p, 'contiguous'))
    check_margin(ref, 'p%d contiguous' % p)
    hyp = load(engine, pr)
    check_against_reference(run_kill(engine, monkeypatch, pr, hyp, ref), ref, pr, 'p%d contiguous' % p)


def _forced_cases():
    cases = []
    for p in FORCED_P:
        if p >= 239:
            cases.append((p, dict(big_min_p=0)))
        else:
            cases.append((p, dict(big_min_p=2)))
        cases.append((p, dict(no_eig=True)))
        for g in (1, 2, 3, 5):
            cases.append((p, dict(big_min_p=2, grid=g)))
        cases.append((p, dict(big_min_p=2, grid=3, eig=True)))
    ids = [_forced_id(c) for c in cases]
    return [c for j, c in enumerate(cases) if ids.index(ids[j]) == j]      # (big below the switch may be a knob grid)


def _forced_id(case):
    p, kw = case
    if kw.get('no_eig'):
        return 'p%d-%s-eig-off' % (p, kill_form(p))
    return 'p%d-%s' % (p, kill_form(p, big_min_p=kw.get('big_min_p'), grid=kw.get('grid'), eig=kw.get('eig', False)))


@pytest.mark.gpu
@pytest.mark.parametrize('case', _forced_cases(), ids=_forced_id)
def test_forced_forms_match_reference(engine, monkeypatch, case):
    """FOKL_KILL_BIG_MIN_P / FOKL_KILL_BIG_GRID / FOKL_KILL_NO_EIG: the full single-CTA form, the big kernel below the
    switch and on 1, 2, 3, 5 CTAs (several rows per warp, the look-ahead owner wrapping), the eigendecomposition
    switched off.  Each matches the reference and gives the default form's bits (the per-entry arithmetic is the
    same; from the eigendecomposition, both start from the same tableau), and with FOKL_KILL_NO_EIG the
    eigendecomposition passed in is ignored."""
    p, kw = case
    what = _forced_id(case)
    pr = problem(p, p)
    ref = reference((p, p))
    hyp = load(engine, pr)
    eig = eigen(engine, pr.cols, hyp) if (kw.get('eig') or kw.get('no_eig')) else None
    got = run_kill(engine, monkeypatch, pr, hyp, ref, eig=eig, big_min_p=kw.get('big_min_p'), grid=kw.get('grid'),
                   no_eig=kw.get('no_eig', False))
    check_against_reference(got, ref, pr, what)
    default = run_kill(engine, monkeypatch, pr, hyp, ref, eig=eig if kw.get('eig') else None)
    same_bits(got, default, what + ' vs ' + kill_form(p, eig=kw.get('eig', False)))


EDGES = ('vm0', 'start-vm', 'none-proposed', 'none-improves', 'all-accepted', 'restart', 'aic')


@pytest.mark.gpu
@pytest.mark.parametrize('form', ['packed', 'big'])
@pytest.mark.parametrize('edge', EDGES)
def test_loop_edges(engine, monkeypatch, edge, form):
    p = 90
    kw = dict(big_min_p=2) if form == 'big' else {}
    what = 'p%d-%s %s' % (p, kill_form(p, **kw), edge)
    key = {'none-improves': (p, 11, 'scattered', 'gauss', None, None, 1),
           'all-accepted': (p, 13, 'scattered', 'gauss', None, 40000, 0, p - 1, 'all')}.get(edge, (p, 10))
    pr = problem(*key)
    hyp = load(engine, pr)
    if edge == 'vm0':
        ref = reference(key)
        ref0 = ref_kill_loop(pr.G, pr.Xty, pr.cols, pr.yty, pr.sum_y, pr.n, [], [], [], evmin=ref['evmin'])
        got = run_kill(engine, monkeypatch, pr, hyp, ref, cand_pos=[], **kw)
        check_decisions(got, ref0, what)
        assert got['n_acc'] == 0 and got['tested'] == 0
        return
    if edge == 'start-vm':
        ref = reference(key, start=len(pr.cand_pos))
        got = run_kill(engine, monkeypatch, pr, hyp, ref, start=len(pr.cand_pos), **kw)
        check_decisions(got, ref, what)
        assert got['n_acc'] == 0 and got['tested'] == 0
        return
    if edge == 'none-proposed':
        # bv1 <= threshstda everywhere, or in (threshstda, threshstdb] with bv0 >= threshav icpt
        bv1 = np.where(np.arange(len(pr.bv1)) % 2, 0.4, 1.5)
        bv0 = np.full(len(pr.bv0), THRESHAV * ICPT)
        assert not np.any(proposed(bv0, bv1))
        monkeypatch.setattr(pr, 'bv0', bv0)
        monkeypatch.setattr(pr, 'bv1', bv1)
        ref = pr.ref()
        got = run_kill(engine, monkeypatch, pr, hyp, ref, **kw)
        check_decisions(got, ref, what)
        assert got['n_acc'] == 0 and got['tested'] == 0
        return
    if edge == 'aic':
        ref = reference(key, aic=True)
        aic_adj = 2.0 - np.log(pr.n)
        check_margin(ref, what)
        got = run_kill(engine, monkeypatch, pr, hyp, ref, aic_adj=aic_adj, **kw)
        check_against_reference(got, ref, pr, what)
        assert ref['n_acc'] != reference(key)['n_acc']            # aic changes the outcome
        return
    ref = reference(key)
    check_margin(ref, what)
    if edge == 'restart':
        k = ref['n_acc'] // 2
        assert k >= 2
        cols2, pos2 = restart_inputs(pr, ref, k)
        r2 = restart_reference(pr, ref, k)
        check_margin(r2, what)
        assert r2['acc'] == ref['acc'][k:]
        got = run_kill(engine, monkeypatch, pr, hyp, ref, cols=cols2, cand_pos=pos2, start=ref['acc'][k - 1] + 1,
                       evmin=float(ref['ev'][k - 1]), **kw)
        check_decisions(got, r2, what)
        err = sse_error(got['ev'], dict(ev=ref['ev'][k:], sse=ref['sse'][k:], s_c=ref['s_c']), pr.n)
        assert err <= SSE_RTOL, (what, err)
        return
    got = run_kill(engine, monkeypatch, pr, hyp, ref, **kw)
    check_against_reference(got, ref, pr, what)
    if edge == 'none-improves':
        assert ref['n_acc'] == 0 and ref['tested'] == int(proposed(pr.bv0, pr.bv1).sum()) > 0
    elif edge == 'all-accepted':
        assert ref['n_acc'] == len(pr.cand_pos) == ref['tested']


GRADED = [(100, {}), (100, dict(big_min_p=2)), (300, {}), (300, dict(big_min_p=0))]


@pytest.mark.gpu
@pytest.mark.parametrize('eig', [False, True], ids=['seq', 'eig'])
@pytest.mark.parametrize('case', GRADED, ids=lambda c: 'p%d-%s' % (c[0], kill_form(c[0], **c[1])))
def test_graded_design_within_condition_scaled_bound(engine, monkeypatch, case, eig):
    """cond(G[cols][cols]) = 1e7: the SSE within GRADED_C cond eps s_c in every form."""
    p, kw = case
    key = (p, 300 + p, 'scattered', 'graded', 1e7)
    pr = problem(*key)
    ref = reference(key)
    bound = GRADED_C * pr.cond * EPS
    what = 'p%d-%s%s graded cond %.1e' % (p, kill_form(p, **kw), '-eig' if eig else '', pr.cond)
    check_margin(ref, what, max(MARGIN, 10 * pr.n * bound * ref['s_c'] / float(ref['sse_full'])))
    hyp = load(engine, pr)
    got = run_kill(engine, monkeypatch, pr, hyp, ref, eig=eigen(engine, pr.cols, hyp) if eig else None, **kw)
    check_against_reference(got, ref, pr, what, bound)


@pytest.mark.gpu
@pytest.mark.parametrize('form', ['packed', 'big'])
@pytest.mark.parametrize('side', ['below', 'above'])
def test_usable_flag_threshold(engine, monkeypatch, side, form):
    """lam_min = 0.5 / 2 x 1e-10 max_k A_kk (max diag = n, the intercept's): just below the usable flag's threshold the
    tableau from the eigendecomposition is not used -- the result is the sequential form's, bit for bit; just above it
    is used and stays within the condition-scaled bound of the reference."""
    p = 80
    kw = dict(big_min_p=2) if form == 'big' else {}
    f = 0.5 if side == 'below' else 2.0
    key = (p, 400 + p, 'scattered', 'graded', 1.0 / (f * 1e-10))
    pr = problem(*key)
    ref = reference(key)
    bound = GRADED_C * pr.cond * EPS
    what = 'p%d-%s-eig flag %s cond %.1e' % (p, kill_form(p, **kw), side, pr.cond)
    check_margin(ref, what, max(MARGIN, 10 * pr.n * bound * ref['s_c'] / float(ref['sse_full'])))
    hyp = load(engine, pr)
    lamb, Q = eigen(engine, pr.cols, hyp)
    lam_min = float(lamb[0])
    assert (lam_min > 1e-10 * pr.n) == (side == 'above'), (lam_min, pr.n)
    seq = run_kill(engine, monkeypatch, pr, hyp, ref, **kw)
    got = run_kill(engine, monkeypatch, pr, hyp, ref, eig=(lamb, Q), **kw)
    if side == 'below':
        same_bits(got, seq, what)
    check_against_reference(seq, ref, pr, what.replace('-eig', ''), bound)
    check_against_reference(got, ref, pr, what, bound)


@pytest.mark.gpu
@pytest.mark.parametrize('case', [(90, {}), (90, dict(big_min_p=2)), (300, {}), (300, dict(big_min_p=0)),
                                  (90, dict(eig=True)), (300, dict(eig=True))],
                         ids=lambda c: 'p%d-%s' % (c[0], kill_form(c[0], big_min_p=c[1].get('big_min_p'),
                                                                     eig=c[1].get('eig', False))))
def test_singular_gram_is_reported(engine, monkeypatch, case):
    """Two equal model columns (scattered list): the forward sweeps' pivot test fails in every form (bad = 1); with an
    eigendecomposition passed in, lam_min ~ 0 keeps the usable flag off and the sequential test runs."""
    p, kw = case
    pr = Problem(p, 700 + p)
    a, b = pr.cols[2], pr.cols[p // 2]
    pr.G[:, b] = pr.G[:, a]
    pr.G[b, :] = pr.G[a, :]
    pr.Xty[b] = pr.Xty[a]
    ref = pr.ref()
    assert ref['bad'] == 1
    hyp = load(engine, pr)
    eig = None
    if kw.get('eig'):
        res = engine.evaluate([pr.cols], hyp, want_eig=True, refine_tol=None)
        eig = (res.lamb, res.Q)
    got = run_kill(engine, monkeypatch, pr, hyp, ref, eig=eig, big_min_p=kw.get('big_min_p'), evmin=0.0)
    assert got['bad'] == 1 and got['n_acc'] == 0, got


@pytest.mark.gpu
@pytest.mark.parametrize('p', [60, 169, 170, 300], ids=lambda p: 'p%d-L-%s' % (p, 'smem' if p * p <= B200_SMEM_OPTIN // 8 - 194 else 'global'))
def test_kill_scores_match_reference_first_round(engine, p):
    """fokl_kill_scores (Cholesky; L in shared memory for p <= 169 on a B200, else in global memory; one warp per
    proposal, p - 1 > 32 proposals so that warps take several) against the reference's SSE of every single-column
    deletion before the first kill, and of the model itself."""
    pr = problem(p, p)
    ref = reference((p, p))
    hyp = load(engine, pr)
    props = list(range(1, p))
    ev, ok = engine.kill_scores(pr.cols, props, hyp)
    assert ok
    sse = np.concatenate([ref['sse0'][1:], [ref['sse_full']]])
    pa = np.array([p - 1] * len(props) + [p])
    ev_ref = bic(sse, pr.n, pa, 0.0)
    err = float(np.max(np.abs(np.asarray(ev, dtype=LD) - ev_ref) * sse / (LD(pr.n) * LD(ref['s_c']))))
    print('kill_scores p%d: SSE error %.2e s_c' % (p, err))
    assert err <= SSE_RTOL, (p, err)
