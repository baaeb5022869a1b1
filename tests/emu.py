"""ctypes wrapper around tests/host_emu/fokl_emu.cpp (host emulation of the CUDA kernels' math)."""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, 'host_emu', 'fokl_emu.cpp')
_SO = os.path.join(_HERE, 'host_emu', 'libfokl_emu.so')
_CSRC = os.path.join(os.path.dirname(_HERE), 'fokl-gpy_b200', 'csrc')

_vp, _i64, _i32, _u64, _f64 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_uint64, ctypes.c_double


class EmuHypers(ctypes.Structure):
    _fields_ = [(k, _f64) for k in ('a', 'b', 'atau', 'btau', 'sigsqd0', 'tausqd0', 'yty', 'sum_y')] + \
               [('n', _i64), ('draws', ctypes.c_int32), ('from0', ctypes.c_int32), ('from1', ctypes.c_int32),
                ('reserved', ctypes.c_int32)]


def _newest_dep():
    deps = [_SRC] + [os.path.join(_CSRC, f) for f in ('fokl_math.cuh', 'cand_math.cuh', 'gram_plan.h', 'update_math.cuh')]
    return max(os.path.getmtime(d) for d in deps)


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_SO) or os.path.getmtime(_SO) < _newest_dep():
        subprocess.check_call(['g++', '-O2', '-ffp-contract=off', '-std=c++17', '-shared', '-fPIC', '-o', _SO, _SRC])
    L = ctypes.CDLL(_SO)
    L.emu_basis_cubic.argtypes = [_vp, _i64, _vp, _i32, _vp, _i32, _vp]
    L.emu_basis_cubic.restype = _i32
    L.emu_phind.argtypes = [_vp, _i64, _i32, _vp, _vp]
    L.emu_phind.restype = _i32
    L.emu_basis_bernoulli.argtypes = [_vp, _i64, _vp, _i32, _vp, _i32, _vp]
    L.emu_basis_bernoulli.restype = None
    L.emu_deriv_cubic.argtypes = [_vp, _i64, _vp, _i32, _vp, _i32, _i32, _f64, _vp]
    L.emu_deriv_cubic.restype = _i32
    L.emu_deriv_bernoulli.argtypes = [_vp, _i64, _vp, _i32, _vp, _i32, _i32, _f64, _vp]
    L.emu_deriv_bernoulli.restype = None
    L.emu_candidate.argtypes = [_vp, _i64, _vp, _vp, _i32, ctypes.POINTER(EmuHypers), _i32, _u64, _u64, _vp, _vp,
                                _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]
    L.emu_candidate.restype = _i32
    L.emu_kill_scores.argtypes = [_vp, _i64, _vp, _vp, _i32, _vp, _i32, ctypes.POINTER(EmuHypers), _vp]
    L.emu_kill_scores.restype = _i32
    L.emu_kill_loop.argtypes = [_vp, _i64, _vp, _vp, _i32, _vp, _vp, _vp, _i32, ctypes.POINTER(EmuHypers), _vp, _i32, _i32, _vp, _vp]
    L.emu_kill_loop.restype = _i32
    L.emu_philox_normals.argtypes = [_u64, _u64, _i32, _i32, _vp]
    L.emu_philox_normals.restype = None
    L.emu_philox_gammas.argtypes = [_u64, _u64, _i32, _f64, _vp]
    L.emu_philox_gammas.restype = None
    L.emu_gram_plan.argtypes = [_vp, _i64] + [_i32] * 11 + [_vp, _vp, _vp]
    L.emu_gram_plan.restype = _i32
    L.emu_update_chain.argtypes = [_vp] * 13 + [_u64, _u64] + [_vp] * 5
    L.emu_update_chain.restype = _i32
    _lib = L
    return L


def basis_cubic(x, orders, tab):
    x = np.ascontiguousarray(x, dtype=np.float64)
    orders = np.ascontiguousarray(orders, dtype=np.int32)
    tab = np.ascontiguousarray(tab, dtype=np.float64)
    out = np.zeros((len(x), len(orders)))
    bad = lib().emu_basis_cubic(x.ctypes.data, len(x), orders.ctypes.data, len(orders), tab.ctypes.data, tab.shape[1],
                                out.ctypes.data)
    return out, bad


def basis_bernoulli(x, orders, tab):
    x = np.ascontiguousarray(x, dtype=np.float64)
    orders = np.ascontiguousarray(orders, dtype=np.int32)
    tab = np.ascontiguousarray(tab, dtype=np.float64)
    out = np.zeros((len(x), len(orders)))
    lib().emu_basis_bernoulli(x.ctypes.data, len(x), orders.ctypes.data, len(orders), tab.ctypes.data, tab.shape[1],
                              out.ctypes.data)
    return out


def deriv_factors(x, orders, tab, e, div, cubic=True):
    """bss_derivatives factor values: e-th derivative of the basis functions `orders` at x, divided by div (e > 0)."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    orders = np.ascontiguousarray(orders, dtype=np.int32)
    tab = np.ascontiguousarray(tab, dtype=np.float64)
    out = np.zeros((len(x), len(orders)))
    fn = lib().emu_deriv_cubic if cubic else lib().emu_deriv_bernoulli
    fn(x.ctypes.data, len(x), orders.ctypes.data, len(orders), tab.ctypes.data, tab.shape[1], int(e), float(div),
       out.ctypes.data)
    return out


def phind(x, n_piece=499):
    x = np.ascontiguousarray(x, dtype=np.float64)
    ph = np.zeros(len(x), dtype=np.int32)
    xs = np.zeros(len(x))
    bad = lib().emu_phind(x.ctypes.data, len(x), n_piece, ph.ctypes.data, xs.ctypes.data)
    return ph, xs, bad


def candidate(G, Xty, idx, hyp, rng_mode=0, seed=0, stream=0, variates=None, sign_fix=None):
    """hyp: dict with a, b, atau, btau, sigsqd0, tausqd0, yty, sum_y, n, draws."""
    G = np.ascontiguousarray(G, dtype=np.float64)
    Xty = np.ascontiguousarray(np.asarray(Xty).reshape(-1), dtype=np.float64)
    idx = np.ascontiguousarray(idx, dtype=np.int32)
    p = len(idx)
    D = int(hyp['draws'])
    h = EmuHypers(hyp['a'], hyp['b'], hyp['atau'], hyp['btau'], hyp['sigsqd0'], hyp['tausqd0'], hyp['yty'],
                  hyp['sum_y'], int(hyp['n']), D, int(np.ceil(D / 2)), int(np.ceil(D / 2 + 1)), 0)
    ev = np.zeros(1)
    betahat = np.zeros(p)
    lamb = np.zeros(p)
    Q = np.zeros((p, p))          # row r = eigenvector r (column-major p x p)
    betas = np.zeros((D, p))
    sigs = np.zeros(D)
    taus = np.zeros(D)
    info = np.zeros(1, dtype=np.int32)
    v = None if variates is None else np.ascontiguousarray(variates, dtype=np.float64)
    s = None if sign_fix is None else np.ascontiguousarray(sign_fix, dtype=np.float64)
    lib().emu_candidate(G.ctypes.data, G.shape[1], Xty.ctypes.data, idx.ctypes.data, p, ctypes.byref(h), rng_mode,
                        seed, stream, None if v is None else v.ctypes.data, None if s is None else s.ctypes.data,
                        ev.ctypes.data, betahat.ctypes.data, lamb.ctypes.data, Q.ctypes.data, betas.ctypes.data,
                        sigs.ctypes.data, taus.ctypes.data, info.ctypes.data)
    return dict(ev=ev[0], betahat=betahat, lamb=lamb, Q=Q.T.copy(), betas=betas, sigs=sigs, taus=taus,
                info=int(info[0]))


def kill_scores(G, Xty, idx, props, hyp):
    G = np.ascontiguousarray(G, dtype=np.float64)
    Xty = np.ascontiguousarray(np.asarray(Xty).reshape(-1), dtype=np.float64)
    idx = np.ascontiguousarray(idx, dtype=np.int32)
    props = np.ascontiguousarray(props, dtype=np.int32)
    D = int(hyp['draws'])
    h = EmuHypers(hyp['a'], hyp['b'], hyp['atau'], hyp['btau'], hyp['sigsqd0'], hyp['tausqd0'], hyp['yty'],
                  hyp['sum_y'], int(hyp['n']), D, int(np.ceil(D / 2)), int(np.ceil(D / 2 + 1)), 0)
    ev = np.zeros(len(props) + 1)
    bad = lib().emu_kill_scores(G.ctypes.data, G.shape[1], Xty.ctypes.data, idx.ctypes.data, len(idx),
                                props.ctypes.data, len(props), ctypes.byref(h), ev.ctypes.data)
    return ev, bad


def kill_loop(G, Xty, idx, cand_pos, bv0, bv1, hyp, threshav=0.05, threshstda=0.5, threshstdb=2.0, icpt=1.0,
              evmin=0.0, aic_adj=0.0, start=0, packed=True):
    """Returns dict(n_acc, tested, bad, acc (candidate indices), calls (tested count at each acceptance), ev).
    packed: symmetric tableau stored as its lower triangle (the shared-memory form) or in full (the global-memory form)."""
    G = np.ascontiguousarray(G, dtype=np.float64)
    Xty = np.ascontiguousarray(np.asarray(Xty).reshape(-1), dtype=np.float64)
    idx = np.ascontiguousarray(idx, dtype=np.int32)
    cand_pos = np.ascontiguousarray(cand_pos, dtype=np.int32)
    bv0 = np.ascontiguousarray(bv0, dtype=np.float64)
    bv1 = np.ascontiguousarray(bv1, dtype=np.float64)
    vm = len(cand_pos)
    D = int(hyp['draws'])
    h = EmuHypers(hyp['a'], hyp['b'], hyp['atau'], hyp['btau'], hyp['sigsqd0'], hyp['tausqd0'], hyp['yty'],
                  hyp['sum_y'], int(hyp['n']), D, int(np.ceil(D / 2)), int(np.ceil(D / 2 + 1)), 0)
    params = np.array([threshav, threshstda, threshstdb, icpt, evmin, aic_adj], dtype=np.float64)
    out_i = np.zeros(3 + 2 * max(vm, 1), dtype=np.int32)
    out_ev = np.zeros(max(vm, 1))
    bad = lib().emu_kill_loop(G.ctypes.data, G.shape[1], Xty.ctypes.data, idx.ctypes.data, len(idx), cand_pos.ctypes.data,
                              bv0.ctypes.data, bv1.ctypes.data, vm, ctypes.byref(h), params.ctypes.data, start,
                              int(bool(packed)), out_i.ctypes.data, out_ev.ctypes.data)
    k = int(out_i[0])
    return dict(n_acc=k, tested=int(out_i[1]), bad=int(bad), acc=out_i[3:3 + k].copy(),
                calls=out_i[3 + vm:3 + vm + k].copy(), ev=out_ev[:k].copy())


_GRAM_STATS = ('n_tiles', 'max_slots', 'blocks', 'max_positions_per_tile', 'max_ksplit', 'sp_spread', 'flex_late', 'pad',
               'loose', 'flex0', 'flex1', 'flex2', 'min_ksplit', 'box8', 'box32', 'box128', 'max_runs')


def gram_plan(A, p_old, c, cap=352, warps=16, kchunks=1, mode=1, gap=0, cross_only=False, allow_loose=True, pad_mode=-1,
              force_r=0):
    """Walk the K2 work plan on the host (slabs of kchunks 16-row chunks): returns (rc, block (p + 1) x c with NaN where
    nothing was written, cover counts, stats dict).  A: [n][p_old + gap + c + 1] in the physical column order of
    fokl_gram_update_ex (old | gap | new | y), or None for the plan checks and statistics alone.  stats: tiles, slots
    and blocks, the k-split range, the pad layout chosen, loose items, busy warps in each consumer form (flex0/1/2),
    tensor-map boxes of each kind and the longest run table of the bulk-copy kernel."""
    p1 = p_old + c + 1
    if A is None:
        n, ptr = 0, None
    else:
        A = np.ascontiguousarray(A, dtype=np.float64)
        n = A.shape[0]
        assert A.shape[1] == p1 + gap
        ptr = A.ctypes.data
    out = np.full((p1, c), np.nan)
    cover = np.zeros((p1, c), dtype=np.int32)
    stats = np.zeros(len(_GRAM_STATS), dtype=np.int32)
    rc = lib().emu_gram_plan(ptr, n, p_old, c, cap, warps, kchunks, mode, gap, int(bool(cross_only)),
                             int(bool(allow_loose)), pad_mode, force_r, out.ctypes.data, cover.ctypes.data,
                             stats.ctypes.data)
    return rc, out, cover, {k: int(v) for k, v in zip(_GRAM_STATS, stats)}


def update_chain(mode, po, pn, draws, astar, atau_star, b, btau, sigsqd0, yty, squerr, n, arrays, variates=None, seed=0,
                 stream=0):
    """csrc/update_math.cuh update_chain on one host thread.  arrays: dict with the keys of fokl_update_chain
    (lam_o, c_o, t_o, m_o, lam_n, c_n, M, Mt, K, W; missing = not used by the mode)."""
    mdl = np.array([mode, po, pn, draws], dtype=np.int32)
    par = np.array([astar, atau_star, b, btau, sigsqd0, yty, squerr, n], dtype=np.float64)
    keep = []

    def ptr(k):
        v = arrays.get(k)
        if v is None:
            return None
        v = np.ascontiguousarray(v, dtype=np.float64)
        keep.append(v)
        return v.ctypes.data
    var = None if variates is None else np.ascontiguousarray(variates, dtype=np.float64)
    gam_o = np.zeros((draws, max(po, 1)))
    gam_n = np.zeros((draws, max(pn, 1)))
    sigs, taus, lik = np.zeros(draws), np.zeros(draws), np.zeros(draws)
    bad = lib().emu_update_chain(mdl.ctypes.data, par.ctypes.data, ptr('lam_o'), ptr('c_o'), ptr('t_o'), ptr('m_o'),
                                 ptr('lam_n'), ptr('c_n'), ptr('M'), ptr('Mt'), ptr('K'), ptr('W'),
                                 None if var is None else var.ctypes.data, seed, stream, gam_o.ctypes.data,
                                 gam_n.ctypes.data, sigs.ctypes.data, taus.ctypes.data, lik.ctypes.data)
    return dict(gam_o=gam_o[:, :po], gam_n=gam_n[:, :pn], sigs=sigs, taus=taus, lik=lik, bad=bad)
