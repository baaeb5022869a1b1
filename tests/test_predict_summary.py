"""The per-row prediction summary (csrc/predict_math.cuh) and its host wiring (FoKL.FoKLRoutines.eng_predict_summary),
without a GPU.

* The header's math compiled for the host (tests/host_emu/predict_emu.cpp) against `np.mean(a, 1)` and
  `np.sort(a, 1)[:, k]`, bit for bit: every row length 1 .. 4200 at its `cut` / `draws - cut`, every rank of short
  rows, and rows with NaN, +-inf, ties, all-equal values and +-0.0.
* evaluate / coverage3 / bss_derivatives through the summary path (threshold forced to 0) on a host "device" built like
  tests/fake_device.py with fokl_predict_summary added: the reference's golden outputs, and the same bits, RNG use
  and `setnos` as the existing path."""
import ctypes
import hashlib
import os
import subprocess
import tempfile
import warnings

import numpy as np
import pytest

from conftest import ROOT

_SRC = os.path.join(ROOT, 'tests', 'host_emu', 'predict_emu.cpp')
_HDR = os.path.join(ROOT, 'fokl-gpy_b200', 'csrc', 'predict_math.cuh')
_HDR2 = os.path.join(ROOT, 'fokl-gpy_b200', 'csrc', 'fokl_math.cuh')
_lib = None


def emu():
    """Build the host emulation into a temporary directory (the tree may be read-only) keyed by its sources."""
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for f in (_SRC, _HDR, _HDR2):
            h.update(open(f, 'rb').read())
        so = os.path.join(tempfile.gettempdir(), 'fokl_predict_emu_%s_%d.so' % (h.hexdigest()[:16], os.getuid()))
        if not os.path.exists(so):
            tmp = so + '.%d.tmp' % os.getpid()
            subprocess.check_call(['g++', '-O2', '-ffp-contract=off', '-std=c++17', '-shared', '-fPIC', '-o', tmp, _SRC])
            os.replace(tmp, so)
        L = ctypes.CDLL(so)
        vp = ctypes.c_void_p
        L.emu_predict_summary.argtypes = [vp, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp, vp]
        L.emu_predict_summary.restype = None
        L.emu_pw_leaf_count.argtypes = [ctypes.c_int]
        L.emu_pw_leaf_count.restype = ctypes.c_int
        _lib = L
    return _lib


def summary(a, rank_lo=-1, rank_hi=-1):
    a = np.ascontiguousarray(a, dtype=np.float64)
    n, d = a.shape
    mean, lo, hi = np.empty(n), np.empty(n), np.empty(n)
    emu().emu_predict_summary(a.ctypes.data, n, d, rank_lo, rank_hi, mean.ctypes.data, lo.ctypes.data, hi.ctypes.data)
    return mean, lo, hi


def cut_of(d):
    return int(np.floor(d * 0.025) + 1)


def same(got, want):
    """Identical bits, except that NaN payloads and the sign of a zero are free (np.sort treats -0.0 == 0.0)."""
    got, want = np.asarray(got), np.asarray(want)
    if not np.array_equal(got, want, equal_nan=True):
        return False
    fin = ~np.isnan(want) & (want != 0)
    return np.array_equal(got[fin].view(np.uint64), want[fin].view(np.uint64))


def test_mean_and_ranks_match_numpy_at_every_row_length_up_to_4200():
    rng = np.random.default_rng(7)
    for d in range(1, 4201):
        rows = 3 if d > 600 else 6
        a = np.exp(rng.uniform(-20, 20, (rows, d))) * rng.choice([-1.0, 1.0], (rows, d))
        if d % 3 == 0:
            a = rng.standard_normal((rows, d)) + 1e3         # one exponent: the select starts deep in the mantissa
        if d >= 2:
            c = cut_of(d)
            rl, rh = c, d - c
        else:
            rl = rh = 0
        mean, lo, hi = summary(a, rl, rh)
        assert np.array_equal(mean.view(np.uint64), np.mean(a, 1).view(np.uint64)), d
        srt = np.sort(a, 1)
        assert same(lo, srt[:, rl]) and same(hi, srt[:, rh]), d


def test_every_rank_of_short_rows():
    rng = np.random.default_rng(8)
    for d in range(1, 70):
        a = np.round(rng.standard_normal((5, d)) * 4) / 4           # many ties
        srt = np.sort(a, 1)
        for k in range(d):
            _, lo, hi = summary(a, k, d - 1 - k)
            assert same(lo, srt[:, k]) and same(hi, srt[:, d - 1 - k]), (d, k)


@pytest.mark.parametrize('d', [2, 3, 8, 39, 40, 41, 127, 128, 129, 1000, 1001])
def test_special_values(d):
    rng = np.random.default_rng(d)
    base = rng.standard_normal((12, d))
    base[0] = 0.0
    base[1] = -0.0
    base[2] = rng.choice([0.0, -0.0], d)
    base[3] = 2.5
    base[4, ::3] = np.nan
    base[5, ::2] = np.inf
    base[5, 1::4] = -np.inf
    base[6, 0] = np.nan                                  # one NaN poisons the mean, sorts last
    base[7] = -np.nan
    base[8] = np.round(base[8])                          # ties
    base[9, : d // 2] = np.inf
    base[9, d // 2:] = -np.inf                           # mean inf - inf = NaN
    base[10] = rng.choice([np.nan, -np.inf, np.inf, 0.0, -0.0, 1.0], d)
    base[11] = 5e-324 * rng.integers(-3, 4, d)          # subnormals
    for k in sorted({0, cut_of(d) % d, (d - cut_of(d)) % d, d - 1}):
        mean, lo, hi = summary(base, k, d - 1 - k)
        want = np.mean(base, 1)
        assert np.array_equal(mean, want, equal_nan=True)
        fin = ~np.isnan(want)
        assert np.array_equal(mean[fin].view(np.uint64), want[fin].view(np.uint64))
        srt = np.sort(base, 1)
        assert same(lo, srt[:, k]) and same(hi, srt[:, d - 1 - k]), (d, k)


def test_mean_only_mode_leaves_rank_outputs_alone():
    a = np.random.default_rng(3).standard_normal((4, 300))
    mean, lo, hi = np.empty(4), np.full(4, 7.0), np.full(4, 7.0)
    emu().emu_predict_summary(a.ctypes.data, 4, 300, -1, -1, mean.ctypes.data, lo.ctypes.data, hi.ctypes.data)
    assert np.array_equal(mean, np.mean(a, 1)) and np.all(lo == 7.0) and np.all(hi == 7.0)


def test_leaf_count_bounds_the_shared_memory_of_a_row():
    for d in (1, 128, 129, 1000, 10000, 100000):
        assert emu().emu_pw_leaf_count(d) <= d // 64 + 1


# ---- host wiring on a host "device" --------------------------------------------------------------------------------

def _product(Xv, b):
    """v[i, d] = sum_j X[i, j] b[d, j] in j order from 0.0 (the kernels' order; the host rounds the product apart)."""
    v = np.zeros((Xv.shape[1], b.shape[0]))
    for j in range(Xv.shape[0]):
        v = v + Xv[j][:, None] * b[:, j][None, :]
    return v


@pytest.fixture
def fake(monkeypatch):
    from FoKL import FoKLRoutines as FR
    from fake_device import FakeDeviceEngine, _view

    class SummaryEngine(FakeDeviceEngine):
        world = 1

        def __init__(self):
            super().__init__()
            self.lib.fokl_predict_draws = self._predict_draws_ordered
            self.lib.fokl_predict_summary = self._predict_summary

        def _predict_draws_ordered(self, ctx, X, ld, n, p, betas, draws, out):
            self.calls.append(('predict_draws', p, draws))
            v = _product(_view(X, (p, ld), np.float64)[:, :n], _view(betas, (draws, p), np.float64))
            _view(out, (n, draws), np.float64)[:] = v
            return 0

        def _predict_summary(self, ctx, X, ld, n, p, betas, draws, rank_lo, rank_hi, mean, lo, hi):
            self.calls.append(('predict_summary', p, draws, n))
            assert ld >= n and draws >= 1 and (rank_lo == rank_hi == -1 or 0 <= min(rank_lo, rank_hi))
            v = _product(_view(X, (p, ld), np.float64)[:, :n], _view(betas, (draws, p), np.float64))
            m, l, h = summary(v, rank_lo, rank_hi)
            _view(mean, (n,), np.float64)[:] = m
            if rank_lo >= 0:
                _view(lo, (n,), np.float64)[:] = l
                _view(hi, (n,), np.float64)[:] = h
            else:
                assert lo is None and hi is None
            return 0

    eng = SummaryEngine()
    monkeypatch.setattr(FR, '_engine', lambda device=None: eng)
    monkeypatch.setattr(FR, '_PREDICT_CHUNK_ROWS', 16)      # several K1 / summary chunks even at the golden sizes
    return FR, eng, monkeypatch


def _golden(name):
    return dict(np.load(os.path.join(ROOT, 'tests', 'golden', name + '.npz'), allow_pickle=True))


@pytest.fixture
def phis_of(phis_cubic, phis_bern):
    return lambda name: (phis_cubic, 'Cubic Splines') if name == 'cubic' else (phis_bern, 'Bernoulli Polynomials')


@pytest.mark.parametrize('name', ['cubic', 'bern'])
def test_evaluate_and_coverage3_through_the_summary_path(name, fake, phis_of):
    FR, eng, mp = fake
    g = _golden('evaluate')
    phis, kernel = phis_of(name)

    def run(min_cells):
        mp.setattr(FR, '_PREDICT_SUMMARY_MIN_CELLS', min_cells)
        eng.calls.clear()
        model = FR.FoKL(phis=phis, kernel=kernel, UserWarnings=False)
        model.mtx, model.minmax, model.draws, model.betas = g['mtx'], g['minmax'].tolist(), 100, g['betas']
        model.inputs, model.data = g['x'], g['data']
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            np.random.seed(int(g['seed']))
            out = [*model.evaluate(g['x'], ReturnBounds=1), model.evaluate(g['x']), model.evaluate(draws=20),
                   *model.coverage3(inputs=g['x'], data=g['data'], draws=100),
                   *model.coverage3(ReturnBounds=False)]
            state = np.random.get_state()
        return out, model.setnos, state, list(eng.calls)

    new, setnos_new, state_new, calls = run(0)
    assert [c[0] for c in calls[:2]] == ['basis_build', 'predict_summary']
    assert 'predict_draws' not in [c[0] for c in calls]
    assert [c[3] for c in calls if c[0] == 'predict_summary'][:4] == [16, 16, 16, 5]      # 53 rows in chunks of 16
    scale = np.max(np.abs(g[name + '_mean'])) + 1e-300
    assert np.max(np.abs(new[0] - g[name + '_mean'])) < 1e-9 * scale
    assert np.max(np.abs(new[1] - g[name + '_bounds'])) < 1e-9 * scale
    assert np.max(np.abs(new[4] - g[name + '_cov_mean'])) < 1e-9 * scale
    assert abs(float(new[6]) - float(g[name + '_cov_rmse'])) < 1e-9 * scale
    old, setnos_old, state_old, calls_old = run(1 << 62)
    assert 'predict_summary' not in [c[0] for c in calls_old]
    assert np.array_equal(setnos_new, setnos_old) and np.array_equal(setnos_new, g[name + '_setnos'])
    assert all(np.array_equal(a, b) for a, b in zip(state_new[1:], state_old[1:])) and state_new[0] == state_old[0]
    assert len(new) == len(old)
    for a, b in zip(new, old):
        assert np.shape(a) == np.shape(b) and np.asarray(a).dtype == np.asarray(b).dtype
        assert same(np.ravel(a), np.ravel(b))


def test_evaluate_draws_one_and_short_setnos_keep_the_existing_path(fake, phis_of):
    FR, eng, mp = fake
    mp.setattr(FR, '_PREDICT_SUMMARY_MIN_CELLS', 0)
    g = _golden('evaluate')
    phis, kernel = phis_of('cubic')
    model = FR.FoKL(phis=phis, kernel=kernel, UserWarnings=False)
    model.mtx, model.minmax, model.draws, model.betas = g['mtx'], g['minmax'].tolist(), 100, g['betas']
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        model.evaluate(g['x'], draws=1)
        assert [c[0] for c in eng.calls] == ['basis_build', 'predict_draws']
        eng.calls.clear()
        model.setnos = model.setnos[:10]            # fewer stored draws than asked for: numpy's behaviour is kept
        model.evaluate(g['x'], draws=30)
        assert [c[0] for c in eng.calls] == ['basis_build', 'predict_draws']


@pytest.mark.parametrize('name', ['cubic', 'bern'])
def test_bss_derivatives_mean_over_draws_through_the_summary_path(name, fake, phis_of):
    FR, eng, mp = fake
    g = _golden('bss_derivatives')
    phis, kernel = phis_of(name)
    model = FR.FoKL(phis=phis, kernel=kernel, UserWarnings=False)
    model.mtx, model.minmax, model.draws, model.betas = g['mtx'], g['minmax'].tolist(), int(g['draws']), g['betas']
    kw = dict(inputs=g['x'], betas=g['betas'], mtx=g['mtx'], minmax=g['minmax'].tolist(), draws=int(g['draws']))
    cases = [({}, 'grad'), (dict(d1=[1, 0, 1], d2=[0, 1, 1]), 'd1d2'), (dict(d1=False, d2=1), 'd2_only'),
             (dict(d1=True, d2=True, ReturnFullArray=True), None)]
    out = {}
    for min_cells in (0, 1 << 62):
        mp.setattr(FR, '_PREDICT_SUMMARY_MIN_CELLS', min_cells)
        eng.calls.clear()
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            out[min_cells] = [model.bss_derivatives(**kw, **extra) for extra, _ in cases]
        kinds = {c[0] for c in eng.calls}
        assert ('predict_summary' in kinds) == (min_cells == 0) and ('predict_draws' in kinds) == (min_cells != 0)
    for (extra, key), got, old in zip(cases, out[0], out[1 << 62]):
        assert np.shape(got) == np.shape(old)
        assert np.array_equal(got.view(np.uint64), old.view(np.uint64)), extra
        if key is not None:
            want = g[name + '_' + key]
            scale = np.max(np.abs(want), axis=0, keepdims=True) + 1e-300
            assert np.max(np.abs(got - want) / scale) < 1e-9
    with pytest.raises(ValueError, match='fewer than draws'):
        mp.setattr(FR, '_PREDICT_SUMMARY_MIN_CELLS', 0)
        model.bss_derivatives(**dict(kw, draws=g['betas'].shape[0] + 1))


def test_device_resident_inputs_are_read_in_place(fake, phis_of):
    """fit(clean=True) on a large dataset leaves `inputs` in HBM (_DeviceInputs): evaluate() and coverage3() read them
    there and leave the attribute un-materialised, with the bits of evaluate(model.inputs)."""
    import pickle
    FR, eng, mp = fake
    mp.setattr(FR, '_PREDICT_SUMMARY_MIN_CELLS', 0)
    g = _golden('evaluate')
    phis, kernel = phis_of('cubic')
    model = FR.FoKL(phis=phis, kernel=kernel, UserWarnings=False)
    model.mtx, model.minmax, model.draws, model.betas = g['mtx'], g['minmax'].tolist(), 100, g['betas']
    model.data = g['data'][:, None]
    model.__dict__['inputs'] = FR._DeviceInputs(eng.upload(g['x'], g['data']))
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        np.random.seed(4)
        mean, bounds = model.evaluate(ReturnBounds=1)
        cm, cb, rmse = model.coverage3()
        assert isinstance(model.__dict__['inputs'], FR._DeviceInputs)
        assert same(cm, mean) and same(cb, bounds)
        ref_mean, ref_bounds = model.evaluate(model.inputs, ReturnBounds=1)
    assert isinstance(model.__dict__['inputs'], np.ndarray)
    assert same(mean, ref_mean) and same(bounds, ref_bounds)
    state = pickle.loads(pickle.dumps(model)).__dict__
    assert isinstance(state['inputs'], np.ndarray) and np.array_equal(state['inputs'], g['x'])
