"""`clean` in HBM (FoKL._clean_on_device, FoKL._evaluate_clean) against the host path, through the product's own
plumbing (Engine.upload / upload_clean / rows_compact and the ctypes argument lists) on the host stand-in of
tests/clean_stand_in.py.  For every form a user reaches the device path by -- pandas frames, float32 arrays, a train
split, more than 32 inputs, transposed inputs, user bounds and pillow, evaluate(raw_inputs, clean=True) -- the two
paths must leave the same attributes, warnings (category and text, in order), numpy RNG state and fit, bit for bit.
The host path is forced by raising _CLEAN_ON_DEVICE_MIN_CELLS."""
import warnings

import numpy as np
import pandas as pd
import pytest

from clean_stand_in import CleanStandIn

HOST, DEVICE = 1 << 62, 0


def _raw(n, m, seed):
    rng = np.random.default_rng(seed)
    x = rng.random((n, m)) * (1.0 + np.arange(m)) - 0.5 * np.arange(m)
    u = (x - x.min(axis=0)) / (x.max(axis=0) - x.min(axis=0))
    y = np.sin(2 * np.pi * u[:, 0]) + u[:, 1] * u[:, -1] + 0.05 * rng.standard_normal(n)
    return x, y


def _forms():
    x, y = _raw(240, 3, 1)
    x40, y40 = _raw(200, 40, 2)
    return {
        'numpy_f64_split': (lambda: (x.copy(), y.copy()), dict(train=0.8)),
        'numpy_f32': (lambda: (x.astype(np.float32), y.astype(np.float32)), {}),
        'numpy_f32_split': (lambda: (x.astype(np.float32), y.copy()), dict(train=0.6)),
        'pandas_f64': (lambda: (pd.DataFrame(x, columns=list('abc')), pd.Series(y)), {}),
        'pandas_f32_split': (lambda: (pd.DataFrame(x.astype(np.float32)), pd.DataFrame(y[:, None])), dict(train=0.7)),
        'transposed': (lambda: (np.ascontiguousarray(x.T), y[None, :].copy()), {}),
        'bounds_pillow_split': (lambda: (x.copy(), y.copy()),
                                dict(train=0.5, minmax=[[-1.0, 2.0], [-1.5, 2.5], [-2.0, 3.0]], pillow=0.1)),
    }


FORMS = _forms()


@pytest.fixture
def stand_in(monkeypatch):
    from FoKL import FoKLRoutines as FR
    eng = CleanStandIn()
    monkeypatch.setattr(FR, '_engine', lambda device=None: eng)
    monkeypatch.setitem(FR.B200_CONFIG, 'rng', 'numpy')
    return FR, eng, monkeypatch


def _fit(FR, eng, mp, cells, form, phis, **extra):
    make, kw = FORMS[form]
    mp.setattr(FR, '_CLEAN_ON_DEVICE_MIN_CELLS', cells)
    eng.log.clear()
    x, y = make()
    with warnings.catch_warnings(record=True) as rec:
        model = FR.FoKL(phis=phis, draws=30, burnin=30, tolerance=1, ConsoleOutput=False)
        warnings.simplefilter('always')
        np.random.seed(11)
        out = model.fit(x, y, clean=True, **kw, **extra)
    return model, out, [(w.category, str(w.message)) for w in rec if issubclass(w.category, UserWarning)], np.random.get_state(), list(eng.log)


def _same(a, b):
    a, b = np.ascontiguousarray(np.atleast_1d(a)), np.ascontiguousarray(np.atleast_1d(b))
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def _same_state(s, t):
    return s[0] == t[0] and np.array_equal(s[1], t[1]) and s[2:] == t[2:]


@pytest.mark.parametrize('form', sorted(FORMS))
def test_fit_clean_on_device_equals_host_path(form, stand_in, phis_cubic):
    FR, eng, mp = stand_in
    dev, dev_out, dev_warn, dev_state, dev_log = _fit(FR, eng, mp, DEVICE, form, phis_cubic)
    assert 'normalize' in [c[0] for c in dev_log]
    assert ('rows_compact' in [c[0] for c in dev_log]) == ('train' in FORMS[form][1])
    assert isinstance(dev.__dict__['inputs'], FR._DeviceInputs)
    host, host_out, host_warn, host_state, host_log = _fit(FR, eng, mp, HOST, form, phis_cubic)
    assert not [c for c in host_log if c[0] in ('normalize', 'rows_compact', 'column_minmax')]
    assert dev_warn == host_warn
    assert _same_state(dev_state, host_state)
    for a, b in zip(dev_out, host_out):
        assert _same(a, b)
    assert _same(dev.inputs, host.inputs) and _same(dev.data, host.data)
    assert (dev.trainlog is None and host.trainlog is None) or _same(dev.trainlog, host.trainlog)
    assert dev.minmax == host.minmax
    for k in ('b', 'btau'):
        assert _same(getattr(dev, k), getattr(host, k)), k


def test_mixed_and_object_frames_and_series_keep_the_host_path(stand_in, phis_cubic):
    FR, eng, mp = stand_in
    mp.setattr(FR, '_CLEAN_ON_DEVICE_MIN_CELLS', DEVICE)
    x, y = _raw(120, 2, 3)
    frames = [pd.DataFrame({'a': x[:, 0], 'b': x[:, 1].astype(np.float32)}), pd.DataFrame(x.astype(object)),
              pd.Series(x[:, 0])]
    for frame in frames:
        eng.log.clear()
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            model = FR.FoKL(phis=phis_cubic, draws=20, burnin=20, tolerance=1, ConsoleOutput=False)
            model.fit(frame, y, clean=True)
        assert not [c for c in eng.log if c[0] in ('normalize', 'rows_compact')]
        assert isinstance(model.__dict__['inputs'], np.ndarray)
    for kw in (dict(bit=32), dict(normalize=False)):
        assert FR.FoKL()._device_raw_inputs(x, dict(FR._CLEAN_DEFAULTS, **kw)) is None


def _evaluate_runs(FR, eng, mp, cells, phis, kernel, raw):
    mp.setattr(FR, '_CLEAN_ON_DEVICE_MIN_CELLS', cells)
    mp.setattr(FR, '_PREDICT_SUMMARY_MIN_CELLS', 0)
    x, y = _raw(150, 3, 5)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        model = FR.FoKL(phis=phis, kernel=kernel, draws=40, burnin=40, tolerance=1, ConsoleOutput=False)
        mp.setattr(FR, '_CLEAN_ON_DEVICE_MIN_CELLS', HOST)
        np.random.seed(3)
        model.fit(x, y, clean=True)
        mp.setattr(FR, '_CLEAN_ON_DEVICE_MIN_CELLS', cells)
    eng.log.clear()
    with warnings.catch_warnings(record=True) as rec:
        model.UserWarnings = True
        warnings.simplefilter('always')
        np.random.seed(4)
        outs = [model.evaluate(raw(), clean=True, ReturnBounds=1), model.evaluate(raw(), clean=True),
                model.evaluate(raw(), clean=True, ReturnBounds=1, minmax=[[-1.0, 2.0], [-1.0, 2.5], [-2.0, 3.0]]),
                model.evaluate(raw(), clean=True, pillow=[0.05, 0.1] * 3, pillow_type='absolute'),
                model.evaluate(raw(), clean=True, draws=1)]
    return outs, [(w.category, str(w.message)) for w in rec if issubclass(w.category, UserWarning)], np.random.get_state(), model, list(eng.log)


@pytest.mark.parametrize('kernel', ['Cubic Splines', 'Bernoulli Polynomials'])
@pytest.mark.parametrize('form', ['numpy_f64', 'numpy_f32', 'pandas_f32', 'transposed'])
def test_evaluate_clean_on_device_equals_host_path(form, kernel, stand_in, phis_cubic, phis_bern):
    FR, eng, mp = stand_in
    phis = phis_cubic if kernel == 'Cubic Splines' else phis_bern
    xr = _raw(90, 3, 6)[0] * 1.2 - 0.1
    raw = {'numpy_f64': lambda: xr.copy(), 'numpy_f32': lambda: xr.astype(np.float32),
           'pandas_f32': lambda: pd.DataFrame(xr.astype(np.float32)), 'transposed': lambda: np.ascontiguousarray(xr.T)}[form]
    dev = _evaluate_runs(FR, eng, mp, DEVICE, phis, kernel, raw)
    assert [c[0] for c in dev[4]].count('normalize') == 4       # draws=1 is reduced on the host: clean stays there
    host = _evaluate_runs(FR, eng, mp, HOST, phis, kernel, raw)
    assert 'normalize' not in [c[0] for c in host[4]]
    assert dev[1] == host[1] and _same_state(dev[2], host[2])
    for a, b in zip(dev[0], host[0]):
        for u, v in zip(a if isinstance(a, tuple) else (a,), b if isinstance(b, tuple) else (b,)):
            assert _same(u, v)
    assert dev[3].minmax == host[3].minmax and _same(dev[3].setnos, host[3].setnos)


def test_rows_compact_plumbing_rejects_a_mask_of_the_wrong_length(stand_in):
    FR, eng, _ = stand_in
    ds = eng.upload(np.arange(12.0).reshape(6, 2), np.arange(6.0))
    with pytest.raises(ValueError):
        eng.rows_compact(ds, np.ones(5, dtype=bool))
    sub = eng.rows_compact(ds, np.array([0, 1, 1, 0, 0, 1], dtype=bool))
    assert sub.n == 3 and sub.ldx == 16
    assert np.array_equal(sub.x[:, :3].t().numpy(), np.arange(12.0).reshape(6, 2)[[1, 2, 5]])
    assert np.array_equal(sub.y[:3].numpy(), [1.0, 2.0, 5.0]) and not sub.x[:, 3:].any() and not sub.y[3:].any()
