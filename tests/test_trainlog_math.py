"""The device train split's rules (csrc/trainlog_math.cuh) built for the host (tests/host_emu/trainlog_emu.cpp), held to
`FoKL.generate_trainlog`'s numpy code without a GPU: the mask, the numpy RNG end state (key, pos) and the MT19937 words
themselves, on n from 2 to 10^6, train from l_log = 2 to 0.999, several seeds, state positions 0, 1, 623 and 624, one-,
two- and three-round splits, U == l_log, and parse tiles from 1 word to the device's."""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import ROOT

_SRC = os.path.join(ROOT, 'tests', 'host_emu', 'trainlog_emu.cpp')
_HDRS = [os.path.join(ROOT, 'fokl-gpy_b200', 'csrc', f) for f in ('trainlog_math.cuh', 'fokl_math.cuh')]
DEVICE_TILE = 4096          # words per parse tile of csrc/trainlog.cu (kParseThreads * kParsePer)
_lib = None


def emu():
    """Build the host emulation into a temporary directory (the tree may be read-only) keyed by its sources."""
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for f in [_SRC] + _HDRS:
            h.update(open(f, 'rb').read())
        so = os.path.join(tempfile.gettempdir(), 'fokl_trainlog_emu_%s_%d.so' % (h.hexdigest()[:16], os.getuid()))
        if not os.path.exists(so):
            tmp = so + '.%d.tmp' % os.getpid()
            subprocess.check_call(['g++', '-O2', '-std=c++17', '-shared', '-fPIC', '-o', tmp, _SRC])
            os.replace(tmp, so)
        L = ctypes.CDLL(so)
        vp, i64, i32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int
        L.emu_mt_words.argtypes = [vp, i32, i64, vp, vp, vp]
        L.emu_mt_words.restype = None
        L.emu_trainlog.argtypes = [vp, i32, i64, i64, i32, vp, vp, vp, vp, vp]
        L.emu_trainlog.restype = i32
        _lib = L
    return _lib


def trainlog(state, n, l_log, tile=DEVICE_TILE):
    """(rc, keep bool[n], key_out, pos_out, words, rounds) from a legacy numpy state tuple."""
    key = np.ascontiguousarray(state[1], dtype=np.uint32)
    keep = np.zeros(n, dtype=np.uint8)
    key_out = np.zeros(624, dtype=np.uint32)
    pos_out, words, rounds = ctypes.c_int(-1), ctypes.c_int64(-1), ctypes.c_int(0)
    rc = emu().emu_trainlog(key.ctypes.data, int(state[2]), n, l_log, tile, keep.ctypes.data, key_out.ctypes.data,
                            ctypes.byref(pos_out), ctypes.byref(words), ctypes.byref(rounds))
    return rc, keep.view(bool), key_out, pos_out.value, words.value, rounds.value


def host_split(train, n):
    from FoKL import FoKLRoutines as FR
    return FR.FoKL.generate_trainlog(None, train, n)


def _state_at(seed, pos):
    """The legacy state of `seed` moved to `pos` words into its block (624: the block is used up, 0: not yet begun)."""
    np.random.seed(seed)
    if pos == 0:
        np.random.set_state(('MT19937', np.random.get_state()[1], 0, 0, 0.0))
    elif pos < 624:
        np.random.randint(0, 2 ** 32, size=pos, dtype=np.uint32)
    st = np.random.get_state()
    assert st[2] == pos
    return st


def _check(seed, pos, n, train, tile=DEVICE_TILE):
    st = _state_at(seed, pos)
    want = host_split(train, n)
    want_state = np.random.get_state()
    l_log = max(int(n * train), 2)
    rc, keep, key, p, words, rounds = trainlog(st, n, l_log, tile)
    assert rc == 0
    assert np.array_equal(keep, want), (seed, pos, n, train)
    assert np.array_equal(key, want_state[1]) and p == want_state[2], (seed, pos, n, train)
    return words, rounds


@pytest.mark.parametrize('pos', [0, 1, 623, 624])
def test_mt_words_match_randint(pos):
    st = _state_at(5, pos)
    count = 3 * 624 + 17
    want = np.random.randint(0, 2 ** 32, size=count, dtype=np.uint32)
    want_state = np.random.get_state()
    out = np.zeros(count, dtype=np.uint32)
    key_out, pos_out = np.zeros(624, dtype=np.uint32), ctypes.c_int(-1)
    key = np.ascontiguousarray(st[1], dtype=np.uint32)
    emu().emu_mt_words(key.ctypes.data, pos, count, out.ctypes.data, key_out.ctypes.data, ctypes.byref(pos_out))
    assert np.array_equal(out, want)
    assert np.array_equal(key_out, want_state[1]) and pos_out.value == want_state[2]


N_GRID = [2, 3, 5, 17, 100, 624, 1000, 4097, 20000, 131073, 10 ** 6]
TRAINS = [1e-9, 0.05, 0.5, 0.8, 0.999]


@pytest.mark.parametrize('n', N_GRID)
@pytest.mark.parametrize('train', TRAINS)
def test_split_matches_generate_trainlog(n, train):
    for seed, pos in ((0, 624), (1, 0), (2, 1), (3, 623)):
        if n >= 10 ** 6 and seed > 1:
            break
        _check(seed, pos, n, train)


@pytest.mark.parametrize('tile', [1, 2, 7, 64, 1000])
def test_split_is_independent_of_the_parse_tile(tile):
    """Small tiles put the bound range across mask boundaries and the kDepends words everywhere."""
    for n, train in ((50, 0.8), (3000, 0.5), (40000, 0.999), (257, 0.05)):
        _check(7, 11, n, train, tile)


def test_round_counts_and_edges():
    """One-, two- and three-round splits, l_log = 2, and U == l_log (the shuffle's every step is inside the kept set)."""
    seen = set()
    for seed in range(40):
        for n, train in ((2, 0.0), (2, 1.0 - 1e-9), (3, 0.9), (1000, 0.8), (1000, 0.999), (10, 0.999), (500, 0.5)):
            words, rounds = _check(seed, 624, n, train)
            seen.add(rounds)
            assert words >= 2 * max(int(n * train), 2) - 1
    assert {1, 2, 3} <= seen, seen
    # U == l_log: n = l_log = 2 ends with both rows kept, and so does every train that keeps all rows
    st = _state_at(3, 624)
    rc, keep, _, _, _, _ = trainlog(st, 2, 2)
    assert rc == 0 and keep.all()


def test_rejected_arguments_leave_the_outputs_untouched():
    st = _state_at(1, 5)
    for n, l_log, pos in ((10, 1, 5), (10, 11, 5), (1 << 31, 2, 5), (10, 5, -1), (10, 5, 625)):
        key = np.ascontiguousarray(st[1], dtype=np.uint32)
        keep = np.full(max(min(n, 16), 1), 7, dtype=np.uint8)
        key_out = np.full(624, 9, dtype=np.uint32)
        p, w = ctypes.c_int(-3), ctypes.c_int64(-3)
        rc = emu().emu_trainlog(key.ctypes.data, pos, n, l_log, DEVICE_TILE, keep.ctypes.data, key_out.ctypes.data,
                                ctypes.byref(p), ctypes.byref(w), None)
        assert rc == -1
        assert (keep == 7).all() and (key_out == 9).all() and p.value == -3 and w.value == -3


@pytest.mark.parametrize('n,train,pos', [(2, 0.5, 624), (5000, 0.8, 0), (70001, 0.05, 623)])
def test_generate_trainlog_device_route_on_a_host_stand_in(monkeypatch, n, train, pos):
    """generate_trainlog's device route (Engine.trainlog and the ctypes argument list of fokl_trainlog, served by the
    host build) leaves the host loop's mask and the whole numpy state, cached gaussian included."""
    import types

    import torch
    from FoKL import FoKLRoutines as FR
    from FoKL._engine import Engine

    class HostEngine:
        trainlog = Engine.trainlog
        _ck = Engine._ck

    eng = HostEngine()
    eng.torch, eng.device, eng.ctx = torch, torch.device('cpu'), None
    calls = []

    def fokl_trainlog(ctx, key, pos_, n_, l_log, keep, key_out, pos_out, words):
        calls.append((n_, l_log))
        return emu().emu_trainlog(key, pos_, n_, l_log, DEVICE_TILE, keep, key_out, pos_out, words, None)
    eng.lib = types.SimpleNamespace(fokl_trainlog=fokl_trainlog, fokl_last_error=lambda ctx: b'bad argument')
    monkeypatch.setattr(FR, '_engine', lambda device=None: eng)
    monkeypatch.setattr(FR, '_have_cuda', lambda: True)
    st = _state_at(4, pos)
    np.random.standard_normal()
    st = np.random.get_state()
    out = {}
    for where in (1 << 62, 0):
        monkeypatch.setattr(FR, '_TRAINLOG_ON_DEVICE_MIN_ROWS', where)
        np.random.set_state(st)
        out[where] = (FR.FoKL().generate_trainlog(train, n), np.random.get_state())
    (h, hs), (d, ds) = out[1 << 62], out[0]
    assert calls == [(n, max(int(n * train), 2))]
    assert d.dtype == np.bool_ and np.array_equal(h, d)
    assert hs[0] == ds[0] and np.array_equal(hs[1], ds[1]) and hs[2:] == ds[2:] and hs[3] == 1
