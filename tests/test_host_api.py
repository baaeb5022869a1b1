"""Host-side mirror of the reference API (no GPU needed): constructor kwargs, clean, term generation, save/load,
and that the hot path fails loudly without a CUDA device."""
import itertools
import os
import pickle

import numpy as np
import pytest

import fokl_oracle as fo
from FoKL import FoKLRoutines, _selection, getKernels


def test_constructor_defaults_and_errors(phis_cubic):
    m = FoKLRoutines.FoKL(phis=phis_cubic)
    assert (m.a, m.atau, m.tolerance, m.burnin, m.draws) == (4, 4, 3, 1000, 1000)
    assert m.kernel == 'Cubic Splines' and m.b is None and m.btau is None and m.relats_in == []
    assert m.gimmie is False and m.way3 is False and m.aic is False and m.setnos is None
    assert (m.threshav, m.threshstda, m.threshstdb) == (0.05, 0.5, 2)
    with pytest.raises(ValueError):
        FoKLRoutines.FoKL(phis=phis_cubic, nonsense=1)
    m2 = FoKLRoutines.FoKL(kernel=1, way3='on', aic='yes', UserWarnings=False)
    assert m2.kernel == 'Bernoulli Polynomials' and m2.way3 is True and m2.aic is True and len(m2.phis) == 20
    assert [len(r) for r in m2.phis] == list(range(2, 22))
    assert set(['kernel', 'phis', 'relats_in', 'a', 'b', 'atau', 'btau', 'tolerance', 'burnin', 'draws', 'gimmie',
                'way3', 'threshav', 'threshstda', 'threshstdb', 'aic', 'update', 'built']) == set(m.hypers)


def test_class_identity_for_pickles(phis_cubic, tmp_path):
    assert FoKLRoutines.FoKL.__module__ == 'FoKL.FoKLRoutines'
    m = FoKLRoutines.FoKL(kernel=1, UserWarnings=False)
    m.betas = np.ones((3, 2))
    path = m.save(str(tmp_path / 'model'))
    assert path.endswith('.fokl')
    again = FoKLRoutines.load(str(tmp_path / 'model'))
    assert isinstance(again, FoKLRoutines.FoKL) and np.array_equal(again.betas, m.betas)
    assert b'FoKL.FoKLRoutines' in pickle.dumps(m)


def test_clean_normalises_like_the_oracle(phis_cubic):
    rng = np.random.default_rng(0)
    x = rng.normal(size=(50, 3)) * [1, 10, 100]
    y = rng.normal(size=50)
    m = FoKLRoutines.FoKL(phis=phis_cubic, UserWarnings=False)
    xi, yi = m.clean(x, y)
    ref, mm = fo.normalize(x)
    assert np.array_equal(xi, ref) and yi.shape == (50, 1)
    assert np.allclose(np.array(m.minmax), np.array(mm))
    assert m.trainlog is None and m.trainset()[0] is m.inputs
    # list-of-columns input is auto-transposed; explicit minmax is honoured
    m3 = FoKLRoutines.FoKL(phis=phis_cubic, UserWarnings=False)
    xi3 = m3.clean([x[:, 0], x[:, 1]], minmax=[[-5, 5], [-50, 50]])
    assert xi3.shape == (50, 2) and np.allclose(xi3[:, 0], (x[:, 0] + 5) / 10)
    with pytest.raises(ValueError):
        m3.clean(x, y, bogus=True)
    with pytest.raises(ValueError):
        m3.clean(x, np.ones((50, 2)))


def test_evaluate_basis_matches_oracle(phis_cubic, phis_bern):
    m = FoKLRoutines.FoKL(phis=phis_cubic, UserWarnings=False)
    c = [phis_cubic[3][k][17] for k in range(4)]
    assert m.evaluate_basis(c, 0.3) == fo.eval_basis(c, 0.3, fo.CUBIC)
    assert m.evaluate_basis(c, 0.3, d=1) == c[1] + 2 * c[2] * 0.3 + 3 * c[3] * 0.3 ** 2
    assert m.evaluate_basis(phis_bern[4], 0.7, kernel=1) == fo.eval_basis(phis_bern[4], 0.7, fo.BERNOULLI)
    with pytest.raises(ValueError):
        m.evaluate_basis(c, 0.3, kernel='nope')


def test_term_generation_matches_reference_semantics():
    for v in ([1, 0, 0, 0], [2, 1, 1, 0, 0], [2, 2, 0, 0], [3, 1, 0, 0, 0, 0], [1, 1, 1, 0, 0, 0], [3, 2, 1, 0], [4]):
        want = np.unique(np.vstack(list(itertools.permutations(np.array(v, dtype=float))))[::-1], axis=0)
        got = _selection.distinct_permutations(v)
        assert np.array_equal(got.astype(float), want)
    assert _selection.distinct_permutations([3, 2, 1, 0, 0, 0, 0, 0]).shape == (336, 8)
    assert _selection.distinct_permutations([1, 1, 1] + [0] * 13).shape == (560, 16)
    for ind, m, way3 in ((4, 5, True), (5, 3, True), (3, 4, False), (6, 2, False), (3, 1, False)):
        sett = 1 if m == 1 else (3 if way3 else 2)
        v = _selection.first_partition(ind, m, sett)
        w = fo.initial_indvec(ind, m, sett)
        while True:
            assert list(w) == v
            a, b = _selection.next_partition(v, m, way3), fo.advance_indvec(w, m, way3)
            assert a == b
            if not a:
                break


def test_numpy_variates_consume_the_stream_like_the_oracle():
    src = _selection.NumpyVariates(4, 4, 100, 30)
    np.random.seed(3)
    got = src.draw(5)
    s1 = np.random.get_state()[1].copy()
    np.random.seed(3)
    z, g1, g2 = fo.draw_variates(5, 30, 4 + 1 + 50 + 2.5, 4 + 2)
    assert np.array_equal(got[:, :5], z) and np.array_equal(got[:, 5], g1) and np.array_equal(got[:, 6], g2)
    assert np.array_equal(s1, np.random.get_state()[1])


def test_fit_fails_loudly_without_a_gpu(phis_cubic):
    import torch
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    m = FoKLRoutines.FoKL(phis=phis_cubic, UserWarnings=False, ConsoleOutput=False)
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        m.fit(np.random.rand(20, 2), np.random.rand(20), clean=True)
    with pytest.raises(RuntimeError):          # fitupdate is a device path now: without a CUDA device it fails loudly
        m.fitupdate(np.random.rand(8, 2), np.random.rand(8))


def test_out_of_scope_entry_points_say_so(phis_cubic):
    m = FoKLRoutines.FoKL(phis=phis_cubic, UserWarnings=False)
    with pytest.raises(ImportError):
        m.to_pyomo(None, None)
    # bss_derivatives: keyword handling mirrors FR:626-740 and fails before any device work
    m.mtx, m.minmax, m.draws = np.array([[1.0, 0.0], [1.0, 2.0]]), [[0, 1], [0, 1]], 2
    with pytest.raises(ValueError, match="does not align"):
        m.bss_derivatives(inputs=np.random.rand(4, 2), betas=np.ones((2, 5)))
    with pytest.raises(ValueError, match="equal length"):
        m.bss_derivatives(inputs=np.random.rand(4, 2), betas=np.ones((2, 3)), d1=[1, 0, 0])
    with pytest.warns(UserWarning, match="no derivatives were requested"):
        assert m.bss_derivatives(inputs=np.random.rand(4, 2), betas=np.ones((2, 3)), d1=False) is None
    m.clear()
    assert hasattr(m, 'phis') and not hasattr(m, 'setnos')


def test_regenerated_spline_table_is_deterministic_and_continuous():
    tab = getKernels.regenerate_spline_table(6)
    assert tab.shape == (6, 499, 4)
    # C0 continuity across pieces: value at t = 1 of piece i equals value at t = 0 of piece i + 1
    end = tab[:, :-1, :].sum(axis=2)
    start = tab[:, 1:, 0]
    assert np.max(np.abs(end - start)) < 1e-12
    gold = np.load(__import__('os').path.join(__import__('conftest').GOLD, 'phis_cubic_48.npy'))
    assert np.allclose(tab, gold[:6], rtol=0, atol=1e-9)


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver times next to the GPU arm) needs no GPU: one JSON line with
    the metric / unit / config of the GPU arm, impl = reference, cpu_baseline and a zero-copy e2e object."""
    import json
    import subprocess
    import sys
    from conftest import ROOT
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1',
                          '--warmup', '0', '--cpu-seconds', '1', '--cpu-rows', '600'], capture_output=True, text=True,
                         timeout=240, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line['impl'] == 'reference' and line['metric'] == 'FoKL.fit candidate-models/sec'
    assert line['unit'] == 'candidate-models/s' and line['higher_is_better'] is True and line['value'] > 0
    assert line['config']['workload'].startswith('cfg4') and line['dtype'] == 'f64'
    assert line['cpu_baseline']['kind'] == 'port' and line['cpu_baseline']['cores'] >= 1
    assert line['e2e'] == {'value': line['value'], 'unit': line['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}


def test_bench_dump_outputs_are_float64_and_bounded(tmp_path, monkeypatch):
    """bench.py --dump-outputs: one float64 .npy per returned array; past the size budget the rows of betas are cut to a
    sample that is the same on every run and keeps draw order."""
    import importlib.util
    import sys
    from conftest import ROOT
    monkeypatch.setattr(sys, 'path', list(sys.path))          # bench.py puts its own entries in front
    spec = importlib.util.spec_from_file_location('bench', os.path.join(ROOT, 'bench.py'))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    betas = np.arange(1000 * 30, dtype=np.float64).reshape(1000, 30)
    arrays = dict(betas=betas, mtx=np.ones((29, 4), dtype=np.int64), evs=np.arange(5.0))
    bench.dump_outputs(str(tmp_path / 'all'), arrays)
    got = {k: np.load(str(tmp_path / 'all' / (k + '.npy'))) for k in arrays}
    assert all(got[k].dtype == np.float64 and np.array_equal(got[k], arrays[k]) for k in arrays)
    monkeypatch.setattr(bench, 'DUMP_BYTES', 100_000)
    cut = []
    for run in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / run), arrays)
        cut.append({k: np.load(str(tmp_path / run / (k + '.npy'))) for k in arrays})
    assert sum(v.nbytes for v in cut[0].values()) <= 100_000 and 0 < cut[0]['betas'].shape[0] < 1000
    assert all(np.array_equal(cut[0][k], cut[1][k]) for k in arrays)
    assert np.array_equal(cut[0]['mtx'], arrays['mtx']) and np.all(np.diff(cut[0]['betas'][:, 0]) > 0)


def test_clean_against_reference_golden(phis_cubic):
    """Host `clean` (format, normalise with minmax / pillow, random train split from the seeded global RNG) against
    outputs of the unmodified reference (tests/golden/clean.npz, oracle/gen_golden.py): bit-identical."""
    import warnings
    from conftest import load_golden
    g = load_golden('clean')
    x, y = g['x'], g['y']
    variants = dict(
        plain=dict(),
        minmax=dict(minmax=[[-5.0, 5.0], [-40.0, 40.0], [-400.0, 400.0]]),
        pillow_pct=dict(pillow=0.1),
        pillow_abs=dict(pillow=[[0.5, 0.25], [1.0, 2.0], [3.0, 4.0]], pillow_type='absolute'),
        train=dict(train=0.6),
    )
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        for name, kw in variants.items():
            model = FoKLRoutines.FoKL(phis=phis_cubic, UserWarnings=False)
            np.random.seed(11)
            model.clean(x, y, _setattr=True, **kw)
            assert np.array_equal(np.asarray(model.inputs), g[name + '_inputs']), name
            assert np.array_equal(np.asarray(model.data), g[name + '_data']), name
            assert np.array_equal(np.asarray(model.minmax, dtype=np.float64), g[name + '_minmax']), name
            want_log = g[name + '_trainlog']
            if want_log.size == 0:
                assert model.trainlog is None, name
            else:
                assert np.array_equal(model.trainlog, want_log), name
            ti, td = model.trainset()
            assert np.array_equal(np.asarray(ti), g[name + '_train_inputs']), name
            assert np.array_equal(np.asarray(td), g[name + '_train_data']), name
        model = FoKLRoutines.FoKL(phis=phis_cubic, UserWarnings=False)
        assert np.array_equal(np.asarray(model.clean([x[:, 0], x[:, 1]])), g['cols_inputs'])
        model = FoKLRoutines.FoKL(phis=phis_cubic, UserWarnings=False)
        xi, yi = model.clean(x[:, 2], y)
        assert np.array_equal(np.asarray(xi), g['oned_inputs']) and np.array_equal(np.asarray(yi), g['oned_data'])


def test_constructor_state_equals_the_reference():
    """Attribute set, defaults, `hypers` / `keep` lists of a fresh model == the unmodified reference's
    (tests/golden/constructor.json, oracle/gen_golden.py)."""
    import json
    import warnings
    from conftest import GOLD
    want = json.load(open(os.path.join(GOLD, 'constructor.json')))

    def dump(m):
        d = {}
        for k, v in vars(m).items():
            if k.startswith('_'):
                continue
            if k == 'phis':
                d[k] = [len(v), len(v[0])]
            elif isinstance(v, (list, tuple)):
                d[k] = list(v)
            elif isinstance(v, np.generic):
                d[k] = v.item()
            else:
                d[k] = v
        return d
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        got = {'default_kernel1': dump(FoKLRoutines.FoKL(kernel=1)),
               'custom': dump(FoKLRoutines.FoKL(kernel='Bernoulli Polynomials', a=9, b=0.01, atau=3, btau=4000, aic=True,
                                                tolerance=5, draws=200, burnin=50, way3=True, gimmie=True, threshav=0.1,
                                                threshstda=0.4, threshstdb=3, UserWarnings=False, ConsoleOutput=False))}
    for case in want:
        assert got[case] == want[case], (case, {k: (got[case].get(k), want[case].get(k)) for k in
                                               set(got[case]) | set(want[case]) if got[case].get(k) != want[case].get(k)})


def test_loads_a_model_saved_by_the_reference():
    """`FoKLRoutines.load` on tests/golden/ref_model.fokl -- trained and pickled by the unmodified reference
    (oracle/gen_golden.py) -- gives a model of this package's FoKL class with the reference's attributes."""
    from conftest import GOLD
    g = np.load(os.path.join(GOLD, 'ref_model_expect.npz'))
    model = FoKLRoutines.load(os.path.join(GOLD, 'ref_model.fokl'))
    assert type(model) is FoKLRoutines.FoKL and model.kernel == 'Bernoulli Polynomials'
    for key in ('betas', 'mtx', 'evs', 'setnos'):
        assert np.array_equal(np.asarray(getattr(model, key)), g[key]), key
    assert np.array_equal(np.asarray(model.inputs), g['inputs']) and np.array_equal(np.asarray(model.data), g['data'])
    assert np.array_equal(np.asarray(model.minmax, dtype=np.float64), g['minmax'])
    assert model.draws == 40 and model.burnin == 40 and len(model.phis) == 20


@pytest.mark.skipif(not os.path.isdir(__import__('ref_harness').REF_SRC),
                    reason='needs the upstream FoKL-GPy sources: set FOKL_REFERENCE_SRC')
def test_reference_loads_a_model_saved_here(tmp_path, phis_bern):
    """The other direction of the save/load layout: a model pickled by this package (attributes set by hand -- no GPU
    here) is loaded by the unmodified reference's `load` as its own FoKL class, attributes intact.  What is checked is
    the reference's own unpickling code, so no stored output can stand in for it: without the upstream sources
    (oracle/ref_harness.py) the test is skipped."""
    import subprocess
    import sys
    from conftest import ROOT
    model = FoKLRoutines.FoKL(kernel=1, draws=7, burnin=3, UserWarnings=False, ConsoleOutput=False)
    model.betas = np.arange(21.0).reshape(7, 3)
    model.mtx = np.array([[1.0, 0.0], [0.0, 2.0]])
    model.evs = np.array([-1.0, -2.0])
    model.inputs, model.data, model.minmax = np.random.rand(5, 2), np.random.rand(5, 1), [[0.0, 1.0], [0.0, 1.0]]
    path = model.save(str(tmp_path / 'mine'))
    code = ("import sys, numpy as np; sys.path.insert(0, %r); import ref_harness; FR = ref_harness.load_reference(); "
            "m = FR.load(%r); assert type(m).__module__ == 'FoKL.FoKLRoutines' and m.__class__ is FR.FoKL; "
            "assert m.betas.shape == (7, 3) and m.draws == 7 and m.kernel == 'Bernoulli Polynomials'; "
            "assert np.array_equal(m.mtx, [[1.0, 0.0], [0.0, 2.0]]) and len(m.phis) == 20; print('ok')"
            % (os.path.join(ROOT, 'oracle'), path))
    out = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and out.stdout.strip().endswith('ok'), out.stderr[-1500:]


def test_bernoulli_table_equals_the_reference_table(bern_table):
    """getKernels.bernoulli() -- the only phis table upstream ships -- against the reference's own loader output
    (tests/golden/bernoulli_table.npy, SURVEY section 8c KAT 4): same structure, same bits."""
    phis = getKernels.bernoulli()
    assert len(phis) == bern_table.shape[0] == 20
    for n, row in enumerate(phis):
        assert len(row) == n + 2
        assert np.array_equal(np.asarray(row, dtype=np.float64), bern_table[n, :n + 2])
