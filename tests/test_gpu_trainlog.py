"""fokl_trainlog on the B200 against `generate_trainlog`'s numpy loop (forced by raising _TRAINLOG_ON_DEVICE_MIN_ROWS):
the keep-mask and the whole numpy RNG end state, bit for bit, for n up to 5 * 10^7, several train values, seeds and state
positions; rejected arguments leave every output untouched; and cfg4's shape with train=0.8 (N = 10^7) gives the same
fit, split and RNG state with the split drawn on the host and in HBM."""
import ctypes
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST, DEVICE = 1 << 62, 0


@pytest.fixture
def FR(monkeypatch):
    from FoKL import FoKLRoutines
    monkeypatch.setattr(FoKLRoutines, '_TRAINLOG_ON_DEVICE_MIN_ROWS', FoKLRoutines._TRAINLOG_ON_DEVICE_MIN_ROWS)
    return FoKLRoutines


def _state_at(seed, pos):
    np.random.seed(seed)
    if pos == 0:
        np.random.set_state(('MT19937', np.random.get_state()[1], 0, 0, 0.0))
    elif pos < 624:
        np.random.randint(0, 2 ** 32, size=pos, dtype=np.uint32)
    np.random.standard_normal()          # a cached gaussian the split must leave alone
    return np.random.get_state()


def _split(FR, where, state, train, n):
    FR._TRAINLOG_ON_DEVICE_MIN_ROWS = where
    np.random.set_state(state)
    mask = FR.FoKL().generate_trainlog(train, n)
    return mask, np.random.get_state()


def _same_state(s, t):
    return s[0] == t[0] and np.array_equal(s[1], t[1]) and s[2:] == t[2:]


CASES = [(2, 0.5, 0, 624), (3, 0.9, 1, 0), (1000, 0.8, 2, 1), (4097, 0.999, 3, 623), (20000, 0.05, 4, 624),
         (131073, 1e-9, 5, 1), (10 ** 6, 0.8, 6, 623), ((1 << 20) + 3, 0.5, 7, 0), (3 * 10 ** 6, 0.999, 8, 624),
         (10 ** 7, 0.8, 9, 1), (2 * 10 ** 7, 0.2, 10, 623), (5 * 10 ** 7, 0.05, 11, 0)]


@pytest.mark.parametrize('n,train,seed,pos', CASES)
def test_device_split_equals_the_numpy_loop(FR, n, train, seed, pos):
    st = _state_at(seed, pos)
    want, want_state = _split(FR, HOST, st, train, n)
    got, got_state = _split(FR, DEVICE, st, train, n)
    assert got.dtype == np.bool_ and got.shape == (n,)
    assert np.array_equal(got, want)
    assert _same_state(got_state, want_state)


def test_engine_reports_the_words_numpy_consumed(FR):
    from FoKL.FoKLRoutines import _engine
    n, train = 300000, 0.8
    st = _state_at(12, 624)
    keep, key, pos, words = _engine().trainlog(st[1], st[2], n, int(n * train))
    np.random.set_state(st)
    np.random.randint(0, 2 ** 32, size=words, dtype=np.uint32)
    after = np.random.get_state()
    assert np.array_equal(after[1], key) and after[2] == pos
    assert int(keep.sum().item()) == int(n * train)


def test_rejected_arguments_leave_the_outputs_untouched():
    import torch
    from FoKL.FoKLRoutines import _engine
    eng = _engine()
    key = np.ascontiguousarray(_state_at(1, 5)[1], dtype=np.uint32)
    for n, l_log, pos, null in ((10, 1, 5, None), (10, 11, 5, None), (1 << 31, 2, 5, None), (10, 5, -1, None),
                                (10, 5, 625, None), (10, 5, 5, 'key'), (10, 5, 5, 'keep'), (10, 5, 5, 'key_out')):
        keep = torch.full((16,), 7, dtype=torch.uint8, device=eng.device)
        key_out = np.full(624, 9, dtype=np.uint32)
        p, w = ctypes.c_int(-3), ctypes.c_int64(-3)
        rc = eng.lib.fokl_trainlog(eng.ctx, None if null == 'key' else key.ctypes.data, pos, n, l_log,
                                   None if null == 'keep' else keep.data_ptr(),
                                   None if null == 'key_out' else key_out.ctypes.data, ctypes.byref(p), ctypes.byref(w))
        assert rc == -1, (n, l_log, pos, null)
        assert (keep.cpu().numpy() == 7).all() and (key_out == 9).all() and p.value == -3 and w.value == -3
    with pytest.raises(ValueError):
        eng.rows_compact(eng.upload(np.zeros((10, 2)), np.zeros(10)), torch.ones(10, dtype=torch.uint8,
                                                                                device=eng.device))


def test_cfg4_shape_fit_with_the_split_on_host_and_device(FR, phis_cubic):
    """cfg4's shape (N = 10^7, 8 inputs, 3-way), train=0.8: the same betas, mtx, evs, trainlog and numpy RNG end state
    whether generate_trainlog runs its host loop or fokl_trainlog."""
    sys.path.insert(0, ROOT)
    import bench_data
    x, y = bench_data.make_rows('cfg4', 0, 10 ** 7, n_total=10 ** 7)
    raw = x * np.arange(1.0, 9.0) - 2.0
    del x
    out = {}
    for name, where in (('host', HOST), ('device', DEVICE)):
        FR._TRAINLOG_ON_DEVICE_MIN_ROWS = where
        np.random.seed(21)
        model = FR.FoKL(phis=phis_cubic, way3=True, UserWarnings=False, ConsoleOutput=False)
        betas, mtx, evs = model.fit(raw, y, clean=True, train=0.8)
        out[name] = (betas, mtx, evs, model.trainlog, np.random.get_state())
    h, d = out['host'], out['device']
    for k in range(4):
        assert h[k].dtype == d[k].dtype and np.array_equal(h[k], d[k]), k
    assert _same_state(h[4], d[4])
    assert int(np.count_nonzero(d[3])) == int(10 ** 7 * 0.8)
