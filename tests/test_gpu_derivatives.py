"""fokl_deriv_summary on the device: bss_derivatives with its rows streamed in chunks, and coverage3 at training-set
scale.

* The streamed path equals the existing one (eng_derivative_draws) on the same device, bit for bit up to NaN payloads
  and the sign of a zero: pair widths 0, 1, a few and ~700, draws on both sides of the summary's shared-memory staging
  limit (2048), N at every row-chunk edge, NaN / inf betas, both IndividualDraws modes.
* The golden bss_derivatives and evaluate cases through the streamed path.
* After fit(clean=True) the device-resident inputs are read in place by bss_derivatives() and coverage3().
* cfg4's shape (N = 1e7, 8 inputs, way3, 1000 draws): bss_derivatives(d1, d2 on every input) and the default
  coverage3() complete, sampled rows match the existing path, and the device memory added does not depend on N.
* Malformed arguments return FOKL_EINVAL and leave the output untouched."""
import warnings

import numpy as np
import pytest

from conftest import load_golden

pytestmark = pytest.mark.gpu

EINVAL = -1
CHUNK = 1 << 16        # FoKLRoutines._PREDICT_CHUNK_ROWS
N_EDGES = [1, CHUNK - 1, CHUNK, CHUNK + 1, 3 * CHUNK + 1]
DRAWS = [2, 3, 40, 1000, 2048, 2049, 5000]


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


def _model(FR, phis, mtx, draws, seed, special=False):
    rng = np.random.default_rng(seed)
    M = mtx.shape[1]
    model = FR.FoKL(phis=phis, draws=draws, UserWarnings=False)
    model.mtx, model.minmax = mtx.astype(np.float64), [[0.0, 1.0 + 0.5 * k] for k in range(M)]
    model.betas = rng.standard_normal((draws, mtx.shape[0] + 1)) * np.geomspace(1, 1e-2, mtx.shape[0] + 1)
    if special:
        model.betas[1, 1] = np.nan
        model.betas[0, 2] = np.inf
        model.betas[-1, -1] = -np.inf
        model.betas[2:5] = model.betas[1]
    return model


def _narrow_mtx():
    """4 inputs: input 0 in 9 terms, input 1 in 4, input 2 in exactly one, input 3 in none (width 0)."""
    mtx = np.zeros((11, 4), dtype=np.int64)
    for t in range(9):
        mtx[t, 0] = 1 + t % 5
    mtx[3:7, 1] = [1, 2, 3, 4]
    mtx[9, 1] = 2
    mtx[10, 2] = 3
    return mtx


def _wide_mtx():
    """3 inputs: ~700 two-way terms of inputs 0 and 1, one main effect of input 2."""
    rows = [(a, b, 0) for a in range(1, 27) for b in range(1, 27)] + [(0, 0, 2), (5, 0, 0)]
    return np.array(rows, dtype=np.int64)


def _both(FR, model, x, monkeypatch, **kw):
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        monkeypatch.setattr(FR, '_DERIV_SUMMARY_MIN_CELLS', 0)
        new = model.bss_derivatives(inputs=x, ReturnFullArray=True, **kw)
        monkeypatch.setattr(FR, '_DERIV_SUMMARY_MIN_CELLS', 1 << 62)
        old = model.bss_derivatives(inputs=x, ReturnFullArray=True, **kw)
    assert np.shape(new) == np.shape(old)
    return new, old


@pytest.mark.parametrize('n', N_EDGES)
@pytest.mark.parametrize('draws', DRAWS)
def test_streamed_equals_the_existing_path(FR, phis_cubic, monkeypatch, draws, n):
    model = _model(FR, phis_cubic, _narrow_mtx(), draws, seed=draws + n, special=draws >= 40)
    x = np.random.default_rng(n).random((n, 4))
    new, old = _both(FR, model, x, monkeypatch, d1=True, d2=[1, 0, 1, 1])
    assert same(new, old), (draws, n)
    if n * draws <= 1 << 22:                # every draw: dy is N x 4 x 2 x draws on the host
        new, old = _both(FR, model, x, monkeypatch, d1=True, d2=[1, 0, 1, 1], IndividualDraws=True)
        assert same(new, old), (draws, n)
        assert np.all(np.reshape(new, (n, 4, 2, draws))[:, 3] == 0.0)


@pytest.mark.parametrize('draws,n', [(2, 3 * CHUNK + 1), (40, CHUNK + 1), (2049, 4097), (1000, 1)])
@pytest.mark.parametrize('kernel', ['cubic', 'bern'])
def test_pairs_about_700_wide(FR, phis_cubic, phis_bern, monkeypatch, draws, n, kernel):
    phis = phis_cubic if kernel == 'cubic' else phis_bern
    mtx = _wide_mtx() if kernel == 'cubic' else np.minimum(_wide_mtx(), 10)
    model = _model(FR, phis, mtx, draws, seed=n, special=True)
    if kernel == 'bern':
        model.kernel = 'Bernoulli Polynomials'
    x = np.random.default_rng(draws).random((n, 3))
    new, old = _both(FR, model, x, monkeypatch, d1=True, d2=True)
    assert same(new, old)
    if n * draws <= 1 << 22:
        new, old = _both(FR, model, x, monkeypatch, d1=[0, 1, 1], d2=1, IndividualDraws=True)
        assert same(new, old)


@pytest.mark.parametrize('name', ['cubic', 'bern'])
def test_golden_cases_through_the_streamed_path(name, FR, phis_cubic, phis_bern, monkeypatch):
    gd = load_golden('bss_derivatives')
    g = load_golden('evaluate')
    phis, kernel = (phis_cubic, 'Cubic Splines') if name == 'cubic' else (phis_bern, 'Bernoulli Polynomials')
    dm = FR.FoKL(phis=phis, kernel=kernel, UserWarnings=False)
    dm.mtx, dm.minmax, dm.draws, dm.betas = gd['mtx'], gd['minmax'].tolist(), int(gd['draws']), gd['betas']
    kw = dict(inputs=gd['x'], betas=gd['betas'], mtx=gd['mtx'], minmax=gd['minmax'].tolist(), draws=int(gd['draws']))
    cases = [({}, 'grad'), (dict(d1=[1, 0, 1], d2=[0, 1, 1]), 'd1d2'), (dict(d1=False, d2=1), 'd2_only'),
             (dict(d1=True, d2=True, IndividualDraws=True, ReturnFullArray=True), 'full_draws')]
    out = {}
    for cells in (0, 1 << 62):
        monkeypatch.setattr(FR, '_DERIV_SUMMARY_MIN_CELLS', cells)
        monkeypatch.setattr(FR, '_PREDICT_SUMMARY_MIN_CELLS', cells)
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            out[cells] = [dm.bss_derivatives(**kw, **extra) for extra, _ in cases]
            em = FR.FoKL(phis=phis, kernel=kernel, UserWarnings=False)
            em.mtx, em.minmax, em.draws, em.betas = g['mtx'], g['minmax'].tolist(), 100, g['betas']
            em.inputs, em.data = g['x'], g['data']
            np.random.seed(int(g['seed']))
            out[cells] += [*em.evaluate(g['x'], ReturnBounds=1), *em.coverage3(inputs=g['x'], data=g['data'])]
    for (extra, key), got, old in zip(cases, out[0], out[1 << 62]):
        want = gd[name + '_' + key]
        assert np.max(np.abs(got - want) / (np.max(np.abs(want), axis=0, keepdims=True) + 1e-300)) < 1e-9, key
        assert np.array_equal(got.view(np.uint64), old.view(np.uint64)), key
    scale = np.max(np.abs(g[name + '_mean'])) + 1e-300
    assert np.max(np.abs(out[0][4] - g[name + '_mean'])) < 1e-9 * scale
    assert np.max(np.abs(out[0][6] - g[name + '_cov_mean'])) < 1e-9 * scale
    for a, b in zip(out[0][4:], out[1 << 62][4:]):
        assert same(np.ravel(a), np.ravel(b))


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
        assert isinstance(model.__dict__['inputs'], FR._DeviceInputs) and n * 8 >= 1 << 20
        assert n * model.draws >= FR._DERIV_SUMMARY_MIN_CELLS
        dy = model.bss_derivatives(d1=True, d2=True)
        cm, cb, rmse = model.coverage3()
        assert isinstance(model.__dict__['inputs'], FR._DeviceInputs)
        host = model.inputs
        rdy = model.bss_derivatives(inputs=host, d1=True, d2=True)
        rm, rb, rr = model.coverage3(inputs=host, data=model.data)
    assert same(dy, rdy) and same(cm, rm) and same(cb, rb)
    assert rmse == rr and np.isfinite(rmse)


def test_cfg4_shape_completes_within_a_chunk_memory_bound(FR, phis_cubic, monkeypatch):
    import torch
    n, draws, n_terms = 10_000_000, 1000, 52
    rng = np.random.default_rng(44)
    mtx = np.zeros((n_terms, 8), dtype=np.int64)
    for t in range(n_terms):
        k = 1 + t % 3
        mtx[t, rng.choice(8, k, replace=False)] = rng.integers(1, 6, k)
    model = FR.FoKL(phis=phis_cubic, draws=draws, UserWarnings=False)
    model.mtx, model.minmax = mtx.astype(np.float64), [[0.0, 1.0]] * 8
    model.betas = rng.standard_normal((draws, n_terms + 1)) * np.geomspace(1, 1e-3, n_terms + 1)
    x = rng.random((n, 8))
    model.inputs, model.data = x, rng.standard_normal((n, 1))
    FR._engine()
    torch.cuda.synchronize()
    ldx = (n + 15) // 16 * 16
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        np.random.seed(9)
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        dy = model.bss_derivatives(d1=True, d2=True)
        grew = torch.cuda.max_memory_allocated() - base
        # the uploaded inputs and their (unused) data column, twice (Engine.upload holds a staging copy while it
        # transposes them), the betas blocks and one chunk of dy: 65536 rows x 16 slots; the existing path's derivative
        # columns alone would be ~16 GB here
        bound = 2 * 8 * ldx * 9 + 8 * draws * 8 * n_terms * 3 + 8 * CHUNK * 16 + (64 << 20)
        assert grew < bound, (grew, bound)
        cm, cb, rmse = model.coverage3()
        assert dy.shape == (n, 16) and np.all(np.isfinite(dy)) and np.isfinite(rmse)
        idx = np.sort(rng.choice(n, 2048, replace=False))
        monkeypatch.setattr(FR, '_DERIV_SUMMARY_MIN_CELLS', 1 << 62)
        old = model.bss_derivatives(inputs=x[idx], d1=True, d2=True)
    assert np.array_equal(dy[idx].view(np.uint64), old.view(np.uint64))
    assert abs(rmse - abs(np.mean(cm) - np.mean(model.data))) == 0.0


def test_malformed_arguments_are_rejected_and_leave_the_output_alone(FR, phis_cubic):
    import torch
    eng = FR._engine()
    eng.set_phis(phis_cubic, 'Cubic Splines')
    n, m, draws = 40, 3, 5
    ds = eng.upload(np.random.default_rng(1).random((n, m)), np.zeros(n))
    terms = np.array([[1, 0, 0], [2, 1, 0], [0, 0, 3]], dtype=np.int16)
    deriv = np.array([[1, 0, 0], [1, 0, 0], [0, 0, 2]], dtype=np.uint8)
    div = np.ones((m, 3))
    b = torch.ones(draws * 3, dtype=torch.float64, device=eng.device)
    out = torch.full((n * m * 2 * draws,), 7.0, dtype=torch.float64, device=eng.device)
    good = np.array([[0, 2, 0, 0, 0], [2, 1, 2 * draws, 2, 1]], dtype=np.int64)

    def call(**o):
        a = dict(kernel=eng.kernel_id, x=ds.x.data_ptr(), ldx=ds.ldx, m=m, r0=0, rows=n, terms=terms.ctypes.data,
                 deriv=deriv.ctypes.data, div=div.ctypes.data, c=3, pairs=good, n_pairs=None, betas=b.data_ptr(),
                 draws=draws, mean_only=0, out=out.data_ptr())
        a.update(o)
        pairs = np.ascontiguousarray(a['pairs'], dtype=np.int64)
        n_pairs = len(pairs) if a['n_pairs'] is None else a['n_pairs']
        return eng.lib.fokl_deriv_summary(eng.ctx, a['kernel'], a['x'], a['ldx'], a['m'], a['r0'], a['rows'],
                                          a['terms'], a['deriv'], a['div'], a['c'], pairs.ctypes.data, n_pairs,
                                          a['betas'], a['draws'], a['mean_only'], a['out'])

    def bad_pair(i, v):
        p = good.copy()
        p[1, i] = v
        return p

    bad = [dict(x=None), dict(terms=None), dict(deriv=None), dict(div=None), dict(betas=None), dict(out=None),
           dict(kernel=7), dict(m=0), dict(r0=-1), dict(rows=0), dict(ldx=n - 1), dict(r0=ds.ldx - n + 1),
           dict(c=-1), dict(draws=0), dict(mean_only=2), dict(n_pairs=0), dict(n_pairs=7),
           dict(pairs=bad_pair(0, -1)), dict(pairs=bad_pair(1, -1)), dict(pairs=bad_pair(0, 3)),
           dict(pairs=bad_pair(1, 3)), dict(pairs=bad_pair(2, -1)), dict(pairs=bad_pair(3, -1)),
           dict(pairs=bad_pair(3, m)), dict(pairs=bad_pair(4, 2)), dict(pairs=bad_pair(4, -1)),
           dict(pairs=np.array([good[0], good[0]])), dict(c=2),
           dict(deriv=np.array([[3, 0, 0], [1, 0, 0], [0, 0, 2]], dtype=np.uint8).ctypes.data)]
    for o in bad:
        assert call(**o) == EINVAL, o
        eng.synchronize()
        assert np.all(out.cpu().numpy() == 7.0), o
    assert call() == 0
    eng.synchronize()
    got = out.cpu().numpy().reshape(n, m, 2, draws)
    assert np.all(got[:, 1] == 0.0) and np.all(got[:, 0, 1] == 0.0) and np.all(got[:, 2, 0] == 0.0)
    assert np.all(got[:, 0, 0] != 7.0) and np.all(got[:, 2, 1] != 7.0)
