"""`FoKL.fit(raw_row_shard, data_shard, clean=True, train=0.8)` on gloo ranks (CPU stand-in engines): the train split is
the single process's split of the whole dataset.  Each rank is seeded differently; rank 0's numpy state must win, the
per-rank `trainlog` masks must concatenate to the single-process mask (266 of 333 rows kept), every rank must end in the
single process's numpy RNG state, and the fit must meet test_dist_gloo's two-rank criteria against the single-process
fit.  Both `clean` routes run: the host route, and the HBM route on tests/clean_stand_in.py (threshold lowered)."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_ROWS = 333


def _engine_for(route, dist):
    from FoKL import FoKLRoutines as FR
    if route == 'device':
        from clean_stand_in import CleanStandIn
        FR._CLEAN_ON_DEVICE_MIN_CELLS = 0
        return CleanStandIn(dist=dist)
    from mock_engine import MockEngine
    from test_public_api_stand_in import StandInEngine

    class ShardedStandIn(StandInEngine):
        def begin_fit(self, ds):
            MockEngine.__init__(self, ds.x, ds.y, self._phis_arg, self._kernel_arg, dist=dist)
    return ShardedStandIn()


def _fit(route, raw, y, dist=None):
    import spline_table
    from FoKL import FoKLRoutines as FR
    eng = _engine_for(route, dist)
    FR._engine = lambda device=None: eng
    phis = spline_table.to_phis(np.load(os.path.join(ROOT, 'tests', 'golden', 'phis_cubic_48.npy')))
    model = FR.FoKL(phis=phis, way3=True, draws=40, burnin=40, UserWarnings=False, ConsoleOutput=False)
    betas, mtx, evs = model.fit(raw, y, clean=True, train=0.8)
    st = np.random.get_state()
    return dict(betas=betas, mtx=mtx, evs=evs, b=model.b, btau=model.btau, trainlog=model.trainlog,
                rows=np.asarray(model.inputs).shape[0], key=st[1], pos=st[2], gauss=[st[3], st[4]])


def _shards(world):
    """Ragged row shards in rank order: the last shard is the short one for 2 ranks, the middle one for 3."""
    if world == 2:
        return [0, 167, N_ROWS]
    return [0, 120, 190, N_ROWS]


def _worker(rank, world, port, route, out_dir):
    import torch.distributed as dist
    for p in (os.path.join(ROOT, 'fokl-gpy_b200'), os.path.join(ROOT, 'oracle'), os.path.join(ROOT, 'tests'), ROOT):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        from FoKL import FoKLRoutines as FR
        from test_selection_mock import synthetic
        FR.B200_CONFIG['rng'] = 'numpy'
        x, y = synthetic(N_ROWS, 3, 12)
        raw = 5.0 * x - 2.0
        cut = _shards(world)
        lo, hi = cut[rank], cut[rank + 1]
        np.random.seed(70 + 13 * rank)                    # deliberately different host RNG state per rank
        out = _fit(route, raw[lo:hi], y[lo:hi], dist)
        np.savez(os.path.join(out_dir, 'rank%d.npz' % rank), **{k: np.asarray(v) for k, v in out.items()})
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(600)
@pytest.mark.parametrize('route', ['host', 'device'])
@pytest.mark.parametrize('world', [2, 3])
def test_ranks_split_the_single_process_dataset(world, route, tmp_path, monkeypatch):
    import torch.multiprocessing as mp
    from FoKL import FoKLRoutines as FR
    from test_selection_mock import synthetic
    port = 35500 + 7 * world + (route == 'device') + (os.getpid() % 1500)
    mp.spawn(_worker, args=(world, port, route, str(tmp_path)), nprocs=world, join=True)
    r = [np.load(os.path.join(str(tmp_path), 'rank%d.npz' % k)) for k in range(world)]

    monkeypatch.setitem(FR.B200_CONFIG, 'rng', 'numpy')
    monkeypatch.setattr(FR, '_engine', FR._engine)
    monkeypatch.setattr(FR, '_CLEAN_ON_DEVICE_MIN_CELLS', FR._CLEAN_ON_DEVICE_MIN_CELLS)
    x, y = synthetic(N_ROWS, 3, 12)
    np.random.seed(70)
    single = _fit(route, 5.0 * x - 2.0, y)

    assert int(single['rows']) == int(N_ROWS * 0.8) == 266
    assert sum(int(q['rows']) for q in r) == 266
    cut = _shards(world)
    for k in range(world):
        assert r[k]['trainlog'].shape == (cut[k + 1] - cut[k],)
    assert np.array_equal(np.concatenate([q['trainlog'] for q in r]), single['trainlog'])
    for k in range(world):
        assert np.array_equal(r[k]['key'], single['key']) and int(r[k]['pos']) == single['pos'], k
        assert np.array_equal(r[k]['gauss'], np.asarray(single['gauss'], dtype=float)), k
        assert np.isclose(float(r[k]['b']), single['b'], rtol=1e-12)
        assert np.isclose(float(r[k]['btau']), single['btau'], rtol=1e-12)
        assert np.array_equal(r[k]['mtx'], single['mtx'])
        assert np.allclose(r[k]['evs'], single['evs'], rtol=1e-9, atol=0)
        assert r[k]['betas'].shape == single['betas'].shape
    for key in ('betas', 'mtx', 'evs', 'b', 'btau'):
        assert all(np.array_equal(r[0][key], r[k][key]) for k in range(1, world)), key
