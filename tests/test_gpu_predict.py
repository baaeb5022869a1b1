"""fokl_predict_summary on the device: the per-row mean and 95 % bounds of evaluate / coverage3 and the mean over
draws of bss_derivatives, reduced on the chip.

* The summary equals the existing path (fokl_predict_draws, then np.mean / np.sort on the host) on the same device,
  bit for bit up to NaN payloads and the sign of a zero: p in {1, 2, 52, 320, 700} x every draws count of the issue's
  grid x n at the L2-chunk edges, plus NaN / inf betas, duplicated draws and all-zero rows.
* evaluate / coverage3 / bss_derivatives through the summary path (threshold 0): the golden cases, the old path's bits,
  `setnos` and numpy RNG state.
* cfg4's shape (N = 1e7, 8 inputs, 52 cubic 3-way terms, 1000 draws) at the default threshold: completes, matches the
  old path on sampled rows, and the device memory it adds does not depend on N.
* After fit(clean=True) the device-resident inputs are read in place."""
import pickle
import tempfile
import warnings

import numpy as np
import pytest

from conftest import load_golden

pytestmark = pytest.mark.gpu

P_GRID = [1, 2, 52, 320, 700]
DRAWS_GRID = [2, 3, 39, 40, 41, 127, 128, 129, 1000, 1001, 4097, 10000]
CHUNK_BYTES, TILE_ROWS, MAX_CHUNK_ROWS = 32 << 20, 128, 1 << 16     # csrc/predict.cu


def chunk_rows(draws):
    r = CHUNK_BYTES // (8 * draws) // TILE_ROWS * TILE_ROWS
    return min(max(r, TILE_ROWS), MAX_CHUNK_ROWS)


def same(got, want):
    got, want = np.asarray(got), np.asarray(want)
    if not np.array_equal(got, want, equal_nan=True):
        return False
    fin = ~np.isnan(want) & (want != 0)
    return np.array_equal(got[fin].view(np.uint64), want[fin].view(np.uint64))


@pytest.fixture(scope='module')
def FR():
    from FoKL import FoKLRoutines
    return FoKLRoutines


def _summary(eng, X, ld, n, p, b, draws, rlo, rhi):
    import torch
    out = torch.full((3, n), 12345.0, dtype=torch.float64, device=eng.device)
    eng._ck(eng.lib.fokl_predict_summary(eng.ctx, X.data_ptr(), ld, n, p, b.data_ptr(), draws, rlo, rhi,
                                         out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr()))
    eng.synchronize()
    return out.cpu().numpy()


def _old(eng, X, ld, n, p, b, draws):
    import torch
    out = torch.empty((n, draws), dtype=torch.float64, device=eng.device)
    eng._ck(eng.lib.fokl_predict_draws(eng.ctx, X.data_ptr(), ld, n, p, b.data_ptr(), draws, out.data_ptr()))
    eng.synchronize()
    return out.cpu().numpy()


def _check_against_old(eng, X, ld, ns, p, b, draws):
    old = _old(eng, X, ld, max(ns), p, b, draws)
    cut = int(np.floor(draws * 0.025) + 1)
    mean_all = np.mean(old, 1)
    srt = np.sort(old, axis=1)
    for n in ns:
        got = _summary(eng, X, ld, n, p, b, draws, cut, draws - cut)
        assert np.array_equal(got[0].view(np.uint64), mean_all[:n].view(np.uint64)) or same(got[0], mean_all[:n]), n
        assert same(got[1], srt[:n, cut]) and same(got[2], srt[:n, draws - cut]), (n, p, draws)
        m_only = _summary(eng, X, ld, n, p, b, draws, -1, -1)
        assert same(m_only[0], got[0]) and np.all(m_only[1:] == 12345.0)


@pytest.mark.parametrize('draws', DRAWS_GRID)
@pytest.mark.parametrize('p', P_GRID)
def test_summary_equals_the_existing_path(FR, p, draws):
    import torch
    eng = FR._engine()
    c = chunk_rows(draws)
    ns = sorted({1, 17, c - 1, c, c + 1, 3 * c + 5})
    n_max = max(ns)
    g = torch.Generator(device=eng.device).manual_seed(p * 100003 + draws)
    ld = (n_max + 15) // 16 * 16 + 16
    X = torch.rand((p, ld), dtype=torch.float64, device=eng.device, generator=g)
    X[0] = 1.0
    b = torch.randn((draws, p), dtype=torch.float64, device=eng.device, generator=g) * 3.0
    _check_against_old(eng, X, ld, ns, p, b, draws)


@pytest.mark.parametrize('draws', [40, 1000, 4097])
def test_nan_inf_betas_duplicated_draws_and_zero_rows(FR, draws):
    import torch
    eng = FR._engine()
    p, c = 52, chunk_rows(draws)
    n = c + 37
    g = torch.Generator(device=eng.device).manual_seed(draws)
    X = torch.rand((p, n), dtype=torch.float64, device=eng.device, generator=g)
    X[:, 5] = 0.0                       # all-zero rows: every draw gives +0.0
    X[:, c] = 0.0
    b = torch.randn((draws, p), dtype=torch.float64, device=eng.device, generator=g)
    b[3, 7] = float('nan')
    b[11, 0] = float('inf')
    b[12, 1] = -float('inf')
    b[20:30] = b[19]                    # duplicated draws: ties at every row
    b[-1, -1] = -float('nan')
    _check_against_old(eng, X, n, [n, c, 17], p, b, draws)
    b2 = b.clone()
    b2[:] = b[0]                        # every draw the same: all-equal rows
    _check_against_old(eng, X, n, [n], p, b2, draws)


def test_bad_arguments_are_rejected(FR):
    import torch
    eng = FR._engine()
    X = torch.ones((2, 16), dtype=torch.float64, device=eng.device)
    b = torch.ones((4, 2), dtype=torch.float64, device=eng.device)
    out = torch.zeros((3, 16), dtype=torch.float64, device=eng.device)
    args = lambda rlo, rhi, hi_ptr: (eng.ctx, X.data_ptr(), 16, 16, 2, b.data_ptr(), 4, rlo, rhi, out[0].data_ptr(),
                                     out[1].data_ptr(), hi_ptr)
    for rlo, rhi, hi_ptr in ((4, 1, out[2].data_ptr()), (-1, 2, out[2].data_ptr()), (1, 2, None), (-2, -2, None)):
        assert eng.lib.fokl_predict_summary(*args(rlo, rhi, hi_ptr)) != 0
    assert np.all(out.cpu().numpy() == 0.0)


@pytest.mark.parametrize('name', ['cubic', 'bern'])
def test_golden_evaluate_coverage3_and_bss_derivatives_through_the_summary_path(name, FR, phis_cubic, phis_bern,
                                                                                monkeypatch):
    g = load_golden('evaluate')
    gd = load_golden('bss_derivatives')
    phis, kernel = (phis_cubic, 'Cubic Splines') if name == 'cubic' else (phis_bern, 'Bernoulli Polynomials')

    def run(min_cells):
        monkeypatch.setattr(FR, '_PREDICT_SUMMARY_MIN_CELLS', min_cells)
        model = FR.FoKL(phis=phis, kernel=kernel, UserWarnings=False)
        model.mtx, model.minmax, model.draws, model.betas = g['mtx'], g['minmax'].tolist(), 100, g['betas']
        model.inputs, model.data = g['x'], g['data']
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            np.random.seed(int(g['seed']))
            out = [*model.evaluate(g['x'], ReturnBounds=1), model.evaluate(g['x']), model.evaluate(draws=20),
                   *model.coverage3(inputs=g['x'], data=g['data'], draws=100)]
            setnos, state = model.setnos, np.random.get_state()
            dm = FR.FoKL(phis=phis, kernel=kernel, UserWarnings=False)
            dm.mtx, dm.minmax, dm.draws, dm.betas = gd['mtx'], gd['minmax'].tolist(), int(gd['draws']), gd['betas']
            kw = dict(inputs=gd['x'], betas=gd['betas'], mtx=gd['mtx'], minmax=gd['minmax'].tolist(),
                      draws=int(gd['draws']))
            out += [dm.bss_derivatives(**kw), dm.bss_derivatives(d1=[1, 0, 1], d2=[0, 1, 1], **kw),
                    dm.bss_derivatives(d1=False, d2=1, **kw)]
        return out, setnos, state

    new, setnos, state = run(0)
    old, setnos_old, state_old = run(1 << 62)
    scale = np.max(np.abs(g[name + '_mean'])) + 1e-300
    assert np.max(np.abs(new[0] - g[name + '_mean'])) < 1e-9 * scale
    assert np.max(np.abs(new[1] - g[name + '_bounds'])) < 1e-9 * scale
    assert np.max(np.abs(new[4] - g[name + '_cov_mean'])) < 1e-9 * scale
    assert abs(float(new[6]) - float(g[name + '_cov_rmse'])) < 1e-9 * scale
    for got, key in zip(new[7:], ('grad', 'd1d2', 'd2_only')):
        want = gd[name + '_' + key]
        assert np.max(np.abs(got - want) / (np.max(np.abs(want), axis=0, keepdims=True) + 1e-300)) < 1e-9
    assert np.array_equal(setnos, setnos_old)
    assert state[0] == state_old[0] and all(np.array_equal(a, b) for a, b in zip(state[1:], state_old[1:]))
    for a, b in zip(new, old):
        assert np.shape(a) == np.shape(b) and same(np.ravel(a), np.ravel(b))
    for a, b in zip(new[7:], old[7:]):           # bss_derivatives: the very bits of np.mean(dy, axis=3)
        assert np.array_equal(np.asarray(a).view(np.uint64), np.asarray(b).view(np.uint64))


def _cfg4_model(FR, phis, n_terms=52, draws=1000, seed=44):
    rng = np.random.default_rng(seed)
    mtx = np.zeros((n_terms, 8), dtype=np.int64)
    for t in range(n_terms):
        k = 1 + t % 3
        mtx[t, rng.choice(8, k, replace=False)] = rng.integers(1, 6, k)
    model = FR.FoKL(phis=phis, draws=draws, UserWarnings=False)
    model.mtx, model.minmax = mtx.astype(np.float64), [[0.0, 1.0]] * 8
    model.betas = rng.standard_normal((draws, n_terms + 1)) * np.geomspace(1, 1e-3, n_terms + 1)
    return model


def test_cfg4_shape_completes_matches_sampled_rows_and_memory_does_not_grow_with_n(FR, phis_cubic, monkeypatch):
    import torch
    n = 10_000_000
    rng = np.random.default_rng(5)
    x = rng.random((n, 8))
    data = rng.standard_normal(n)
    model = _cfg4_model(FR, phis_cubic)
    # data as a flat vector: with an (N, 1) column, coverage3's 'rmse' keeps the reference's (N,) - (N, 1) broadcast
    # (FR:1193), an N x N host array
    model.inputs, model.data = x, data
    FR._engine()
    torch.cuda.synchronize()
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        np.random.seed(9)
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        mean, bounds = model.evaluate(x, ReturnBounds=1)
        grew = torch.cuda.max_memory_allocated() - base
        cm, cb, rmse = model.coverage3()
        assert same(cm, mean) and same(cb, bounds) and np.isfinite(rmse)
        assert grew < 2 * 1024 ** 3, grew        # the uploaded inputs and the three output columns, no N x draws block
        assert mean.shape == (n,) and bounds.shape == (n, 2) and mean.dtype == np.float64
        idx = np.sort(rng.choice(n, 4096, replace=False))
        monkeypatch.setattr(FR, '_PREDICT_SUMMARY_MIN_CELLS', 1 << 62)
        om, ob = model.evaluate(x[idx], ReturnBounds=1)
    assert same(mean[idx], om) and same(bounds[idx], ob)


def test_fit_clean_device_inputs_are_read_in_place(FR, phis_cubic):
    n = 200_000
    rng = np.random.default_rng(6)
    x = rng.random((n, 8)) * 3.0 - 1.0
    y = np.sin(2 * np.pi * (x[:, 0] + 1) / 3) + 0.05 * rng.standard_normal(n)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        np.random.seed(3)
        model = FR.FoKL(phis=phis_cubic, draws=100, burnin=100, UserWarnings=False, ConsoleOutput=False)
        model.fit(x, y, clean=True)
        assert isinstance(model.__dict__['inputs'], FR._DeviceInputs)
        assert n * model.draws >= FR._PREDICT_SUMMARY_MIN_CELLS
        mean, bounds = model.evaluate(ReturnBounds=1)
        cm, cb, _ = model.coverage3(data=False)     # no 'rmse': the reference's form of it is N x N here
        assert isinstance(model.__dict__['inputs'], FR._DeviceInputs)
        assert same(cm, mean) and same(cb, bounds)
        rm, rb = model.evaluate(model.inputs, ReturnBounds=1)
    assert isinstance(model.__dict__['inputs'], np.ndarray)
    assert same(mean, rm) and same(bounds, rb)
    with tempfile.TemporaryDirectory() as d:
        path = model.save('m', directory=d)
        back = FR.load(path)
    assert isinstance(back.__dict__['inputs'], np.ndarray) and np.array_equal(back.inputs, model.inputs)
    st = pickle.loads(pickle.dumps(model)).__dict__
    assert isinstance(st['inputs'], np.ndarray)
