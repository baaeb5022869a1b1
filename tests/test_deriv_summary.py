"""bss_derivatives streamed through fokl_deriv_summary (FoKL.FoKLRoutines.eng_derivative_summary), and coverage3's
'rmse' without the N x N broadcast, without a GPU.

* A host stand-in for fokl_deriv_summary (argument order, pair table, dy layout, zeros in the slots no pair writes),
  built on tests/fake_device.py: the derivative columns of each row chunk by the stand-in's K1 formulas, each pair's
  values in the kernels' FMA order, the mean over the draws by the host build of csrc/predict_math.cuh.
* bss_derivatives through it (threshold forced to 0, rows in chunks of 16) equals the existing path bit for bit, and
  the reference's golden outputs, for cubic and Bernoulli, d1 / d2 given as int, list, bool and str, an input that no
  term contains, ReturnFullArray on and off, and both IndividualDraws modes.
* Device-resident default inputs are read in place.
* coverage3's 'rmse' with an (N, 1) data column: the literal expression's bits up to N = 4096, within 1e-12 of the
  data's scale above."""
import os
import warnings

import numpy as np
import pytest

from conftest import ROOT
from test_predict_summary import _product, summary


def same(got, want):
    """Identical bits, except that NaN payloads and the sign of a zero are free."""
    got, want = np.asarray(got), np.asarray(want)
    if not np.array_equal(got, want, equal_nan=True):
        return False
    fin = ~np.isnan(want) & (want != 0)
    return np.array_equal(got[fin].view(np.uint64), want[fin].view(np.uint64))


@pytest.fixture
def fake(monkeypatch):
    from FoKL import FoKLRoutines as FR
    from fake_device import FakeDeviceEngine, _view

    class DerivEngine(FakeDeviceEngine):
        world = 1

        def __init__(self):
            super().__init__()
            self.lib.fokl_predict_draws = self._predict_draws_ordered
            self.lib.fokl_predict_summary = self._predict_summary
            self.lib.fokl_deriv_summary = self._deriv_summary

        def _predict_draws_ordered(self, ctx, X, ld, n, p, betas, draws, out):
            self.calls.append(('predict_draws', p, draws))
            v = _product(_view(X, (p, ld), np.float64)[:, :n], _view(betas, (draws, p), np.float64))
            _view(out, (n, draws), np.float64)[:] = v
            return 0

        def _predict_summary(self, ctx, X, ld, n, p, betas, draws, rank_lo, rank_hi, mean, lo, hi):
            self.calls.append(('predict_summary', p, draws, n))
            v = _product(_view(X, (p, ld), np.float64)[:, :n], _view(betas, (draws, p), np.float64))
            _view(mean, (n,), np.float64)[:] = summary(v)[0]
            return 0

        def _deriv_summary(self, ctx, kernel, x, ldx, m, r0, rows, terms, deriv, divisors, c, pairs, n_pairs, betas,
                           draws, mean_only, out):
            """include/fokl_b200.h: pairs n_pairs x {column offset, width, betas offset, input, order - 1}; out the
            C-order slice dy[r0:r0 + rows], [rows][m][2][draws] or (mean_only) [rows][m][2]."""
            assert kernel == self.kernel_id and 0 <= r0 and rows >= 1 and ldx >= r0 + rows and mean_only in (0, 1)
            self.calls.append(('deriv_summary', r0, rows, n_pairs, mean_only))
            xs = np.ascontiguousarray(_view(x, (m, ldx), np.float64)[:, r0:r0 + rows])
            W = np.zeros((c, rows))
            self._columns(xs.ctypes.data, rows, rows, m, terms, deriv, divisors, c, W.ctypes.data, rows)
            table = _view(pairs, (n_pairs, 5), np.int64)
            total = int(max((t[2] + draws * t[1] for t in table), default=0))
            b = _view(betas, (total,), np.float64)
            dst = _view(out, (rows, m, 2, 1 if mean_only else draws), np.float64)
            dst[:] = 0.0
            assert len({(int(t[3]), int(t[4])) for t in table}) == n_pairs
            for off, w, boff, pm, di in table:
                assert 0 <= off and off + w <= c and 0 <= pm < m and di in (0, 1)
                if w == 0:
                    continue
                v = _product(W[off:off + w], b[boff:boff + draws * w].reshape(draws, w))
                dst[:, pm, di, :] = summary(v)[0][:, None] if mean_only else v
            return 0

    eng = DerivEngine()
    monkeypatch.setattr(FR, '_engine', lambda device=None: eng)
    monkeypatch.setattr(FR, '_PREDICT_CHUNK_ROWS', 16)      # several row chunks even at the golden sizes
    return FR, eng, monkeypatch


def _golden(name):
    return dict(np.load(os.path.join(ROOT, 'tests', 'golden', name + '.npz'), allow_pickle=True))


@pytest.fixture
def phis_of(phis_cubic, phis_bern):
    return lambda name: (phis_cubic, 'Cubic Splines') if name == 'cubic' else (phis_bern, 'Bernoulli Polynomials')


def _run(FR, eng, mp, model, kw, cases, new):
    mp.setattr(FR, '_DERIV_SUMMARY_MIN_CELLS', 0 if new else 1 << 62)
    mp.setattr(FR, '_PREDICT_SUMMARY_MIN_CELLS', 1 << 62)
    eng.calls.clear()
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        out = [model.bss_derivatives(**kw, **extra) for extra in cases]
    kinds = {c[0] for c in eng.calls}
    assert ('deriv_summary' in kinds) == new and ('predict_draws' in kinds) == (not new)
    return out


CASES = [{}, dict(d1=[1, 0, 1], d2=[0, 1, 1]), dict(d1=False, d2=1),
         dict(d1=True, d2=True, IndividualDraws=True, ReturnFullArray=True),
         dict(d1=2, d2='on'), dict(d1='off', d2=[True, False, True]), dict(d1=[2], d2=True),
         dict(d1=True, d2=True, ReturnFullArray=True), dict(d1=1, IndividualDraws=True),
         dict(d1=[0, 1, 1], IndividualDraws=True, ReturnFullArray=False)]
GOLDEN_KEYS = ['grad', 'd1d2', 'd2_only', 'full_draws']


@pytest.mark.parametrize('name', ['cubic', 'bern'])
def test_streamed_derivatives_equal_the_existing_path_and_the_golden_outputs(name, fake, phis_of):
    FR, eng, mp = fake
    g = _golden('bss_derivatives')
    phis, kernel = phis_of(name)
    model = FR.FoKL(phis=phis, kernel=kernel, UserWarnings=False)
    model.mtx, model.minmax, model.draws, model.betas = g['mtx'], g['minmax'].tolist(), int(g['draws']), g['betas']
    kw = dict(inputs=g['x'], betas=g['betas'], mtx=g['mtx'], minmax=g['minmax'].tolist(), draws=int(g['draws']))
    new = _run(FR, eng, mp, model, kw, CASES, True)
    assert [c[1:3] for c in eng.calls if c[0] == 'deriv_summary'][-3:] == [(0, 16), (16, 16), (32, 5)]
    old = _run(FR, eng, mp, model, kw, CASES, False)
    for extra, got, want in zip(CASES, new, old):
        assert np.shape(got) == np.shape(want) and got.dtype == want.dtype, extra
        assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), extra
    for key, got in zip(GOLDEN_KEYS, new):
        want = g[name + '_' + key]
        scale = np.max(np.abs(want), axis=0, keepdims=True) + 1e-300
        assert np.shape(got) == np.shape(want) and np.max(np.abs(got - want) / scale) < 1e-9, key


@pytest.mark.parametrize('name', ['cubic', 'bern'])
def test_an_input_that_no_term_contains_and_small_chunks(name, fake, phis_of):
    """A fourth input in no term: its slots are 0.0 (and dropped without ReturnFullArray); a one-row chunk budget
    (16 rows per chunk, the least) in both modes."""
    FR, eng, mp = fake
    g = _golden('bss_derivatives')
    phis, kernel = phis_of(name)
    rng = np.random.default_rng(11)
    x = np.hstack([g['x'], rng.random((g['x'].shape[0], 1))])
    mtx = np.hstack([g['mtx'], np.zeros((g['mtx'].shape[0], 1))])
    minmax = g['minmax'].tolist() + [[0.0, 2.0]]
    model = FR.FoKL(phis=phis, kernel=kernel, UserWarnings=False)
    model.mtx, model.minmax, model.draws, model.betas = mtx, minmax, int(g['draws']), g['betas']
    kw = dict(inputs=x, betas=g['betas'], mtx=mtx, minmax=minmax, draws=int(g['draws']))
    cases = [{}, dict(d1=3, d2=3), dict(d1=3, d2=3, ReturnFullArray=True), dict(d1=[1, 0, 0, 1], d2='yes'),
             dict(d1=True, d2=True, IndividualDraws=True, ReturnFullArray=True), dict(d2=[0, 0, 1, 1], IndividualDraws=1)]
    mp.setattr(FR, '_DERIV_CHUNK_BYTES', 8)
    new = _run(FR, eng, mp, model, kw, cases, True)
    assert {c[2] for c in eng.calls if c[0] == 'deriv_summary'} == {16, 5}
    old = _run(FR, eng, mp, model, kw, cases, False)
    for extra, got, want in zip(cases, new, old):
        assert np.shape(got) == np.shape(want), extra
        assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), extra
    assert np.all(new[2][:, 3] == 0.0) and np.all(new[4][:, 3] == 0.0)


def test_device_resident_inputs_are_read_in_place(fake, phis_of):
    FR, eng, mp = fake
    g = _golden('bss_derivatives')
    phis, kernel = phis_of('cubic')
    model = FR.FoKL(phis=phis, kernel=kernel, UserWarnings=False)
    model.mtx, model.minmax, model.draws, model.betas = g['mtx'], g['minmax'].tolist(), int(g['draws']), g['betas']
    model.__dict__['inputs'] = FR._DeviceInputs(eng.upload(g['x'], np.zeros(len(g['x']))))
    mp.setattr(FR, '_DERIV_SUMMARY_MIN_CELLS', 0)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        got = [model.bss_derivatives(), model.bss_derivatives(d1=True, d2=True, IndividualDraws=True)]
        assert isinstance(model.__dict__['inputs'], FR._DeviceInputs)
        mp.setattr(FR, '_DERIV_SUMMARY_MIN_CELLS', 1 << 62)    # the existing path reads them on the host
        want = [model.bss_derivatives(), model.bss_derivatives(d1=True, d2=True, IndividualDraws=True)]
    assert isinstance(model.__dict__['inputs'], np.ndarray)
    for a, b in zip(got, want):
        assert np.array_equal(a.view(np.uint64), b.view(np.uint64))


def test_out_of_range_inputs_still_warn_when_read_in_place(fake, phis_of):
    FR, eng, mp = fake
    g = _golden('bss_derivatives')
    phis, kernel = phis_of('bern')
    model = FR.FoKL(phis=phis, kernel=kernel)
    model.mtx, model.minmax, model.draws, model.betas = g['mtx'], g['minmax'].tolist(), int(g['draws']), g['betas']
    x = g['x'].copy()
    x[3, 1] = 1.25
    model.__dict__['inputs'] = FR._DeviceInputs(eng.upload(x, np.zeros(len(x))))
    mp.setattr(FR, '_DERIV_SUMMARY_MIN_CELLS', 0)
    with pytest.warns(UserWarning, match='should be normalized'):
        model.bss_derivatives()
    assert isinstance(model.__dict__['inputs'], FR._DeviceInputs)


def _rmse_model(FR, n, rng):
    model = FR.FoKL(UserWarnings=False)
    mean = rng.standard_normal(n) * 3.0 + 1.5
    model.draws, model.betas = 4, np.zeros((4, 2))
    model.inputs, model.data = np.zeros((n, 1)), rng.standard_normal((n, 1)) * 2.0 + 1.0
    model.evaluate = lambda *a, **k: (mean, np.zeros((n, 2))) if k.get('ReturnBounds') else mean
    return model, mean


@pytest.mark.parametrize('n', [1, 2, 3, 17, 64, 1000, 4095, 4096, 4097, 4100, 5000, 6000])
def test_coverage3_rmse_of_a_data_column(n):
    from FoKL import FoKLRoutines as FR
    model, mean = _rmse_model(FR, n, np.random.default_rng(n))
    literal = np.sqrt(np.mean(mean - model.data) ** 2)
    _, _, rmse = model.coverage3()
    _, rmse2 = model.coverage3(ReturnBounds=False)
    assert type(rmse) is type(literal) and rmse2 == rmse
    if n <= 4096:
        assert rmse.view(np.uint64) == literal.view(np.uint64)
    else:
        assert abs(rmse - literal) <= 1e-12 * max(np.max(np.abs(mean)), np.max(np.abs(model.data)))
        # a flat data vector keeps its own path: (n,) - (n,) is elementwise
        flat = model.data[:, 0]
        assert model.coverage3(data=flat, inputs=model.inputs)[2] == np.sqrt(np.mean(mean - flat) ** 2)
