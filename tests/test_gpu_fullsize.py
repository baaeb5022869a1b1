"""BASELINE.json's full-size synthetic workloads (cfg3: N = 1e6, M = 4, Bernoulli; cfg4: N = 1e7, M = 8, 3-way cubic)
on the device, checked through size-independent properties -- the oracle cannot run these sizes (SURVEY section 0.8):

  * design-matrix columns on a row sample against the oracle's literal loop (bit-exact for cubic splines);
  * Gram entries of a column sample against a float64 numpy product over all N rows;
  * BIC from Gram quantities alone against the explicit N-length residual pass (FR:1551-1554);
  * the planted structure of the synthetic target is selected;
  * same seed -> bit-identical fit; a row permutation of the dataset gives the same Gram and the same BIC.
"""
import os
import sys

import numpy as np
import pytest

import fokl_oracle as fo
from conftest import ROOT

sys.path.insert(0, ROOT)
import bench_data  # noqa: E402

pytestmark = pytest.mark.gpu


def _fit(FR, cfg, phis, x, y, seed, **kw):
    np.random.seed(seed)
    model = bench_data.make_model(FR, cfg, phis=phis, **kw)
    betas, mtx, evs = model.fit(x, y, clean=True)
    return model, betas, mtx, evs


def _supports(mtx):
    return {tuple(np.nonzero(r)[0].tolist()) for r in np.asarray(mtx)}


def _device_checks(FR, model, mtx_last, phis, kernel, y, cubic):
    """Checks on the engine's state after a gimmie=True fit (its X / G hold the returned model)."""
    import torch
    from FoKL import _lib
    eng = FR._engine()
    P = eng.P
    n = eng.ds.n
    assert P == mtx_last.shape[0] + 1 and n == len(y)
    rng = np.random.default_rng(99)
    # (a) K1 columns on a row sample
    rows = np.sort(rng.choice(n, 1500, replace=False))
    rows_t = torch.as_tensor(rows, device=eng.device)
    xs = eng.ds.x[:, rows_t].cpu().numpy().T
    got = eng.X[:P].index_select(1, rows_t).cpu().numpy().T
    want = np.hstack([np.ones((len(rows), 1)), fo.basis_columns(xs, mtx_last.astype(int), phis, kernel)])
    if cubic:
        assert np.array_equal(got, want)
    else:
        scale = np.max(np.abs(want), axis=0) + 1e-300
        assert np.max(np.abs(got - want) / scale) < 1e-9
    # (b) Gram / projection entries of a column sample over all N rows
    idx = np.sort(rng.choice(P, min(5, P), replace=False))
    cols = eng.X[torch.as_tensor(idx, device=eng.device), :n].cpu().numpy()
    g_np = cols @ cols.T
    g_dev = eng.G[:P, :P].cpu().numpy()[np.ix_(idx, idx)]
    d = np.sqrt(np.diag(g_np))
    assert np.max(np.abs(g_dev - g_np) / np.outer(d, d)) < 1e-11
    xty_dev = eng.Xty[:P].cpu().numpy()[idx]
    assert np.allclose(xty_dev, cols @ y, rtol=1e-10, atol=1e-10 * np.sqrt(n))
    # (c) Gram-only BIC == explicit residual pass
    hyp = eng.make_hypers(4, 1.0, 4, 1.0, 0.2, 0.2, 10)
    full = list(range(P))
    res = eng.evaluate([full], hyp, rng_mode=_lib.RNG_NONE, refine_tol=None)
    ev_res = eng.residual_bic(full, res.betahat)
    assert np.isclose(res.ev[0], ev_res, rtol=1e-9, atol=0)


def test_cfg4_full_size_properties(phis_cubic):
    from FoKL import FoKLRoutines as FR
    c = bench_data.CONFIGS['cfg4']
    n = c['n']
    x, y = bench_data.make_rows('cfg4', 0, n)
    model, betas, mtx_last, evs = _fit(FR, 'cfg4', phis_cubic, x, y, seed=4, gimmie=True)
    info = dict(FR.LAST_FIT_INFO)
    assert info['n'] == n and betas.shape == (1000, mtx_last.shape[0] + 1)
    _device_checks(FR, model, mtx_last, phis_cubic, fo.CUBIC, y, cubic=True)
    # (d) planted structure: sin(2 pi x0) + x1 x2 + x3 x4 x5 + x6^2 / 2, x7 inert
    _, betas2, mtx, evs2 = _fit(FR, 'cfg4', phis_cubic, x, y, seed=4)
    sup = _supports(mtx)
    for need in [(0,), (1, 2), (3, 4, 5), (6,)]:
        assert need in sup, (need, sorted(sup))
    # (terms of the inert input x7 can survive: the reference only proposes a term for deletion when its relative
    # posterior std exceeds threshstda, FR:1669-1671, and with N = 1e7 a chance 2-sigma coefficient never is)
    assert len(np.unique(mtx, axis=0)) == len(mtx), 'duplicate terms'
    # (e) determinism: the same seed gives the same chain bit for bit
    assert np.array_equal(evs, evs2)
    _, betas3, mtx3, evs3 = _fit(FR, 'cfg4', phis_cubic, x, y, seed=4)
    assert np.array_equal(mtx, mtx3) and np.array_equal(evs2, evs3) and np.array_equal(betas2, betas3)
    # (e') the pipelined selection loop (side context next to the main one: stream-ordering bugs show up at this size,
    # where the full-model evaluation is long) == the sequential loop, bit for bit
    FR.B200_CONFIG['pipeline'] = False
    try:
        _, betas4, mtx4, evs4 = _fit(FR, 'cfg4', phis_cubic, x, y, seed=4)
    finally:
        FR.B200_CONFIG['pipeline'] = True
    assert np.array_equal(mtx, mtx4) and np.array_equal(evs2, evs4) and np.array_equal(betas2, betas4)
    # (f) row order does not matter: the same terms built in one go on a row-permuted copy of the dataset give the
    # same Gram (different summation order and a different K2 work plan: all columns in one launch) and the same BIC.
    import torch
    from FoKL import _lib
    model, _, mtx_last, _ = _fit(FR, 'cfg4', phis_cubic, x, y, seed=4, gimmie=True)
    eng = FR._engine()
    P = eng.P
    G = eng.G[:P, :P].cpu().numpy()
    xty = eng.Xty[:P].cpu().numpy()
    hyp = eng.make_hypers(4, 1.0, 4, 1.0, 0.2, 0.2, 10)
    ev = eng.evaluate([list(range(P))], hyp, rng_mode=_lib.RNG_NONE, refine_tol=None).ev[0]
    xn = eng.ds.x[:, :n].cpu().numpy().T
    perm = np.random.default_rng(5).permutation(n)
    ds_p = eng.upload(xn[perm], y[perm])
    eng.begin_fit(ds_p)
    eng.append_terms(mtx_last.astype(np.int16))
    assert eng.P == P
    G_p = eng.G[:P, :P].cpu().numpy()
    d = np.sqrt(np.diag(G))
    assert np.max(np.abs(G_p - G) / np.outer(d, d)) < 1e-11
    assert np.allclose(eng.Xty[:P].cpu().numpy(), xty, rtol=1e-10, atol=1e-10 * np.sqrt(n))
    ev_p = eng.evaluate([list(range(P))], hyp, rng_mode=_lib.RNG_NONE, refine_tol=None).ev[0]
    assert np.isclose(ev, ev_p, rtol=1e-9, atol=0)
    # (g) ... and, because the free-running chain orients every eigenvector by its projection on X'y (cand_math.cuh,
    # gibbs_chain `canon`), the whole row-permuted fit walks the same path: same terms, same BIC trace
    _, _, mtx_p, evs_p = _fit(FR, 'cfg4', phis_cubic, x[perm], y[perm], seed=4)
    assert np.array_equal(mtx, mtx_p)
    assert np.allclose(evs2, evs_p, rtol=1e-9, atol=0)
    FR._engine().release()


def test_cfg3_full_size_properties(phis_bern):
    from FoKL import FoKLRoutines as FR
    c = bench_data.CONFIGS['cfg3']
    n = c['n']
    x, y = bench_data.make_rows('cfg3', 0, n)
    model, betas, mtx_last, evs = _fit(FR, 'cfg3', None, x, y, seed=3, gimmie=True)
    assert betas.shape == (1000, mtx_last.shape[0] + 1) and mtx_last.shape[1] == 4
    _device_checks(FR, model, mtx_last, model.phis, fo.BERNOULLI, y, cubic=False)
    _, _, mtx, evs2 = _fit(FR, 'cfg3', None, x, y, seed=3)
    sup = _supports(mtx)
    for need in [(0,), (1,), (2, 3)]:        # sin(2 pi x0) + 2 (x1 - 1/2)^2 + x2 x3
        assert need in sup, (need, sorted(sup))
    assert np.array_equal(evs, evs2)
    FR._engine().release()


_DIRECT_FIT = """
import sys, numpy as np
sys.path[:0] = [%r, %r]
import bench_data
from FoKL import FoKLRoutines as FR, getKernels
n, draws, out = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3]
x, y = bench_data.make_rows('cfg4', 0, n, n_total=n)
phis = getKernels._to_phis(getKernels.regenerate_spline_table(500))
ds = FR._engine().upload(x, y)
np.random.seed(bench_data.CONFIGS['cfg4']['seed'])
betas, mtx, evs = bench_data.make_model(FR, 'cfg4', draws=draws, phis=phis).fit(ds, None)
np.savez(out, betas=betas, mtx=mtx, evs=evs)
"""


def test_bench_dump_outputs_are_the_last_timed_fit(tmp_path):
    """bench.py --dump-outputs on a reduced cfg4: the dumped betas / mtx / evs are float64 and equal, bit for bit, to what
    a direct resident fit of the same seeded data and model returns (in its own process).  --steps 1 and --steps 3 dump
    the same arrays, and the timed loop really runs that many fits: three times the device launches, the same
    candidate models per step."""
    import json
    import subprocess
    n, draws = 200000, 200
    lines, dumps = [], []
    for steps in (1, 3):
        d = tmp_path / ('steps%d' % steps)
        r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '1', '--steps', str(steps),
                            '--warmup', '1', '--n', str(n), '--draws', str(draws), '--no-cpu-baseline', '--no-e2e',
                            '--dump-outputs', str(d)], capture_output=True, text=True, timeout=900, cwd=str(tmp_path))
        assert r.returncode == 0, r.stderr[-3000:]
        lines.append(json.loads(r.stdout.strip().splitlines()[-1]))
        dumps.append({k: np.load(str(d / (k + '.npy'))) for k in ('betas', 'mtx', 'evs')})
    assert lines[1]['gpu_launches'] == 3 * lines[0]['gpu_launches'] > 0
    assert lines[1]['candidate_models_per_step'] == lines[0]['candidate_models_per_step'] > 0
    direct = tmp_path / 'direct.npz'
    r = subprocess.run([sys.executable, '-c', _DIRECT_FIT % (os.path.join(ROOT, 'fokl-gpy_b200'), ROOT), str(n),
                        str(draws), str(direct)], capture_output=True, text=True, timeout=900, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-3000:]
    want = np.load(str(direct))
    for k in ('betas', 'mtx', 'evs'):
        for got in dumps:
            assert got[k].dtype == np.float64 and np.array_equal(got[k], want[k]), k
    assert want['betas'].shape == (draws, want['mtx'].shape[0] + 1) and want['mtx'].shape[1] == 8
