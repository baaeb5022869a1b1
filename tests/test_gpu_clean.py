"""`clean` in HBM on the device: fokl_rows_compact against numpy boolean indexing bit for bit (every mask shape, tile
edges, up to 40 inputs, NaN-poisoned outputs so the padding is checked, rejected arguments), fokl_normalize past 32
inputs, and each form a user reaches the device path by against the host path (forced by raising
_CLEAN_ON_DEVICE_MIN_CELLS): attributes, warnings, numpy RNG state, fit and evaluate outputs, bit for bit."""
import copy
import ctypes
import os
import sys
import warnings

import numpy as np
import pandas as pd
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TILE = 4096        # rows per block of the compaction kernel (csrc/ctx.cu kCompactTile)
HOST, DEVICE = 1 << 62, 0


@pytest.fixture(scope='module')
def eng():
    import torch
    from FoKL._engine import Engine
    e = Engine(torch.device('cuda', 0))
    yield e
    e.close()


def _masks(n, rng):
    out = {'all': np.ones(n, bool), 'first': np.zeros(n, bool), 'last': np.zeros(n, bool),
           'alternating': np.arange(n) % 2 == 0}
    out['first'][0] = True
    out['last'][-1] = True
    for p in (0.5, 0.8, 0.999):
        out['rand%g' % p] = rng.random(n) < p
    return out


def _compact(eng, x, y, keep, ldx_out):
    import torch
    m, n = x.shape
    ldx = (n + 15) // 16 * 16
    xd = torch.zeros((m, ldx), dtype=torch.float64, device=eng.device)
    xd[:, :n] = torch.from_numpy(x).to(eng.device)
    yd = torch.zeros(ldx, dtype=torch.float64, device=eng.device)
    yd[:n] = torch.from_numpy(y).to(eng.device)
    kd = torch.from_numpy(keep.view(np.uint8)).to(eng.device)
    xo = torch.full((m, max(ldx_out, 1)), float('nan'), dtype=torch.float64, device=eng.device)
    yo = torch.full((max(ldx_out, 1),), float('nan'), dtype=torch.float64, device=eng.device)
    n_out = ctypes.c_int64(-7)
    rc = eng.lib.fokl_rows_compact(eng.ctx, xd.data_ptr(), yd.data_ptr(), n, ldx, m, kd.data_ptr(), xo.data_ptr(),
                                   yo.data_ptr(), ldx_out, ctypes.byref(n_out))
    eng.synchronize()
    return rc, n_out.value, xo.cpu().numpy(), yo.cpu().numpy()


@pytest.mark.parametrize('n', [1, 15, 16, 17, TILE - 1, TILE, TILE + 1, 2 * TILE - 1, 2 * TILE + 1, 1024 * TILE + 17])
@pytest.mark.parametrize('m', [1, 3, 8, 33, 40])
def test_rows_compact_equals_boolean_indexing(eng, n, m):
    rng = np.random.default_rng(n * 41 + m)
    x = rng.standard_normal((m, n))
    y = rng.standard_normal(n)
    for name, keep in _masks(n, rng).items():
        kept = int(keep.sum())
        ldx_out = (kept + 15) // 16 * 16 + (16 if name == 'alternating' else 0)      # also a wider padding
        rc, n_out, xo, yo = _compact(eng, x, y, keep, ldx_out)
        assert rc == 0 and n_out == kept, name
        assert np.array_equal(xo[:, :kept].view(np.uint64), x[:, keep].view(np.uint64)), name
        assert np.array_equal(yo[:kept].view(np.uint64), y[keep].view(np.uint64)), name
        assert np.all(xo[:, kept:ldx_out] == 0.0) and np.all(yo[kept:ldx_out] == 0.0), name


def test_rows_compact_at_ten_million_rows(eng):
    n, rng = 10 ** 7, np.random.default_rng(5)
    x = rng.standard_normal((2, n))
    y = rng.standard_normal(n)
    keep = rng.random(n) < 0.8
    kept = int(keep.sum())
    rc, n_out, xo, yo = _compact(eng, x, y, keep, (kept + 15) // 16 * 16)
    assert rc == 0 and n_out == kept
    assert np.array_equal(xo[:, :kept], x[:, keep]) and np.array_equal(yo[:kept], y[keep])


def test_rows_compact_rejects_bad_arguments_and_leaves_the_output_untouched(eng):
    import torch
    n, m = 100, 3
    x = torch.zeros((m, 112), dtype=torch.float64, device=eng.device)
    y = torch.zeros(112, dtype=torch.float64, device=eng.device)
    keep = torch.ones(n, dtype=torch.uint8, device=eng.device)
    xo = torch.full((m, 112), float('nan'), dtype=torch.float64, device=eng.device)
    yo = torch.full((112,), float('nan'), dtype=torch.float64, device=eng.device)
    n_out = ctypes.c_int64(-7)
    good = [eng.ctx, x.data_ptr(), y.data_ptr(), n, 112, m, keep.data_ptr(), xo.data_ptr(), yo.data_ptr(), 112,
            ctypes.byref(n_out)]
    bad = [(1, None), (2, None), (6, None), (7, None), (8, None), (10, None), (5, 0), (4, 99), (3, 0), (9, 99)]
    for pos, val in bad:
        args = list(good)
        args[pos] = val
        assert eng.lib.fokl_rows_compact(*args) == -1, pos
    eng.synchronize()
    assert n_out.value == -7 and torch.isnan(xo).all() and torch.isnan(yo).all()
    assert eng.lib.fokl_rows_compact(*good) == 0 and n_out.value == n


def test_normalize_past_32_inputs_matches_the_host_expression(eng):
    rng = np.random.default_rng(9)
    for m in (31, 32, 33, 40, 70):
        raw = rng.random((5000, m)) * 7 - 3
        bounds = [[raw[:, k].min() - 0.1, raw[:, k].max() + 0.2] for k in range(m)]
        ds = eng.upload_clean(raw, np.zeros(5000), lambda column_minmax: bounds)
        host = raw.copy()
        for k in range(m):
            host[:, k] = (host[:, k] - bounds[k][0]) / (bounds[k][1] - bounds[k][0])
        got = ds.x[:, :5000].t().cpu().numpy()
        assert np.array_equal(got, host), m


# ---- each routed form, host path against device path, on the real engine ------------------------------------------------
def _raw(n, m, seed):
    rng = np.random.default_rng(seed)
    x = rng.random((n, m)) * (1.0 + np.arange(m)) - 0.5 * np.arange(m)
    u = (x - x.min(axis=0)) / (x.max(axis=0) - x.min(axis=0))
    y = np.sin(2 * np.pi * u[:, 0]) + u[:, 1] * u[:, -1] + 0.05 * rng.standard_normal(n)
    return x, y


X, Y = _raw(20000, 4, 1)
X40, Y40 = _raw(6000, 40, 2)
FORMS = {
    'numpy_f64_split': (lambda: (X.copy(), Y.copy()), dict(train=0.8)),
    'numpy_f32': (lambda: (X.astype(np.float32), Y.astype(np.float32)), {}),
    'pandas_f64': (lambda: (pd.DataFrame(X, columns=list('abcd')), pd.Series(Y)), {}),
    'pandas_f32_split': (lambda: (pd.DataFrame(X.astype(np.float32)), pd.DataFrame(Y[:, None])), dict(train=0.7)),
    'transposed': (lambda: (np.ascontiguousarray(X.T), Y[None, :].copy()), {}),
    'bounds_pillow_split': (lambda: (X.copy(), Y.copy()),
                            dict(train=0.5, minmax=[[-1.0, 2.0], [-1.5, 2.5], [-2.0, 3.0], [-2.0, 3.0]], pillow=0.1)),
    'wide_40': (lambda: (X40.copy(), Y40.copy()), {}),
    'wide_40_split': (lambda: (X40.copy(), Y40.copy()), dict(train=0.9)),
}


def _same(a, b):
    a, b = np.ascontiguousarray(np.atleast_1d(a)), np.ascontiguousarray(np.atleast_1d(b))
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def _user_warnings(rec):
    return [(w.category, str(w.message)) for w in rec if issubclass(w.category, UserWarning)]


def _fit(FR, cells, form, phis):
    make, kw = FORMS[form]
    FR._CLEAN_ON_DEVICE_MIN_CELLS = cells
    x, y = make()
    with warnings.catch_warnings(record=True) as rec:
        model = FR.FoKL(phis=phis, draws=100, burnin=100, tolerance=1, ConsoleOutput=False)
        warnings.simplefilter('always')
        np.random.seed(11)
        out = model.fit(x, y, clean=True, **kw)
    return model, out, _user_warnings(rec), np.random.get_state()


@pytest.fixture
def FR(monkeypatch):
    from FoKL import FoKLRoutines
    monkeypatch.setattr(FoKLRoutines, '_CLEAN_ON_DEVICE_MIN_CELLS', FoKLRoutines._CLEAN_ON_DEVICE_MIN_CELLS)
    return FoKLRoutines


@pytest.mark.parametrize('form', sorted(FORMS))
def test_fit_clean_on_device_equals_host_path(form, FR, phis_cubic):
    dev, dev_out, dev_warn, dev_state = _fit(FR, DEVICE, form, phis_cubic)
    assert isinstance(dev.__dict__['inputs'], FR._DeviceInputs)
    host, host_out, host_warn, host_state = _fit(FR, HOST, form, phis_cubic)
    assert isinstance(host.__dict__['inputs'], np.ndarray)
    assert dev_warn == host_warn
    assert dev_state[0] == host_state[0] and np.array_equal(dev_state[1], host_state[1]) and dev_state[2:] == host_state[2:]
    for a, b in zip(dev_out, host_out):
        assert _same(a, b)
    assert _same(dev.inputs, host.inputs) and _same(dev.data, host.data) and dev.minmax == host.minmax
    assert (dev.trainlog is None and host.trainlog is None) or _same(dev.trainlog, host.trainlog)
    assert _same(dev.b, host.b) and _same(dev.btau, host.btau)


@pytest.mark.parametrize('kernel', ['Cubic Splines', 'Bernoulli Polynomials'])
@pytest.mark.parametrize('form', ['numpy_f64', 'numpy_f32', 'pandas_f32', 'transposed'])
def test_evaluate_clean_on_device_equals_host_path(form, kernel, FR, phis_cubic, phis_bern):
    phis = phis_cubic if kernel == 'Cubic Splines' else phis_bern
    x3 = X[:3000].astype(np.float32).astype(np.float64)        # float32-exact, so every form stays in the bounds
    xr = x3[np.random.default_rng(6).integers(0, 3000, 40000)]     # of the fit below (the cubic kernel checks them)
    raw = {'numpy_f64': lambda: xr.copy(), 'numpy_f32': lambda: xr.astype(np.float32),
           'pandas_f32': lambda: pd.DataFrame(xr.astype(np.float32)), 'transposed': lambda: np.ascontiguousarray(xr.T)}[form]
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        FR._CLEAN_ON_DEVICE_MIN_CELLS = HOST
        np.random.seed(3)
        base = FR.FoKL(phis=phis, kernel=kernel, draws=500, burnin=500, tolerance=1, ConsoleOutput=False)
        base.fit(x3, Y[:3000], clean=True)
    res = {}
    for cells in (DEVICE, HOST):
        FR._CLEAN_ON_DEVICE_MIN_CELLS = cells
        model = copy.deepcopy(base)
        with warnings.catch_warnings(record=True) as rec:
            model.UserWarnings = True
            warnings.simplefilter('always')
            np.random.seed(4)
            outs = [model.evaluate(raw(), clean=True, ReturnBounds=1), model.evaluate(raw(), clean=True),
                    model.evaluate(raw(), clean=True, ReturnBounds=1, minmax=[[-1.0, 2.0], [-1.0, 2.5], [-2.0, 3.0],
                                                                               [-2.0, 3.0]]),
                    model.evaluate(raw(), clean=True, pillow=[0.05, 0.1] * 4, pillow_type='absolute')]
        res[cells] = (outs, _user_warnings(rec), np.random.get_state(), model.minmax, model.setnos)
    d, h = res[DEVICE], res[HOST]
    assert d[1] == h[1] and np.array_equal(d[2][1], h[2][1]) and d[3] == h[3] and _same(d[4], h[4])
    for a, b in zip(d[0], h[0]):
        for u, v in zip(a if isinstance(a, tuple) else (a,), b if isinstance(b, tuple) else (b,)):
            assert _same(u, v)


def test_cfg4_shape_split_at_ten_million_rows(FR, phis_cubic):
    """cfg4's shape (N = 10^7, 8 inputs, 3-way) with train=0.8 on the device path: it completes, and the training rows
    it holds are the host formula's -- (raw[trainlog] - min) / (max - min) -- at sampled rows, with data[trainlog]."""
    sys.path.insert(0, ROOT)
    import bench_data
    x, y = bench_data.make_rows('cfg4', 0, 10 ** 7, n_total=10 ** 7)
    raw = x * np.arange(1.0, 9.0) - 2.0
    del x
    np.random.seed(21)
    model = FR.FoKL(phis=phis_cubic, way3=True, UserWarnings=False, ConsoleOutput=False)
    betas, mtx, evs = model.fit(raw, y, clean=True, train=0.8)
    assert isinstance(model.__dict__['inputs'], FR._DeviceInputs) and mtx.shape[0] >= 1
    np.random.seed(21)
    trainlog = FR.FoKL().generate_trainlog(0.8, 10 ** 7)
    assert _same(trainlog, model.trainlog)
    rows = np.nonzero(trainlog)[0]
    ds = model.__dict__['inputs'].ds
    assert ds.n == len(rows) == int(10 ** 7 * 0.8)
    pick = np.random.default_rng(0).choice(len(rows), 4096, replace=False)
    pick = np.concatenate([pick, [0, len(rows) - 1]])
    got = ds.x[:, :ds.n].t()[pick].cpu().numpy()
    want = np.empty((len(pick), 8))
    for k in range(8):
        lo, hi = raw[:, k].min(), raw[:, k].max()
        assert model.minmax[k] == [lo, hi]
        want[:, k] = (raw[rows[pick], k] - lo) / (hi - lo)
    assert np.array_equal(got, want)
    assert np.array_equal(model.data[pick, 0], y[rows[pick]])
