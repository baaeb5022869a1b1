"""K2 (fokl_gram_update / fokl_gram_update_ex, csrc/gram.cu + csrc/gram_plan.h) against exact and long-double
references on every pipeline, plan form and row-split edge.

Three pipelines form the block: the bulk-copy / mbarrier ring (gram_kernel_mb<15>), the cp.async ring (gram_kernel<16>,
no loose items) and the tensor-map ring (gram_kernel_tma<15 | 12>, only for the joint [y | X] layout with ld % 16 == 0).
Every case reads fokl_gram_last_config and replays the host plan (tests/host_emu) with the same slot cap, warps, slab
depth and placement, and asserts that the form its test id names is the one that ran: pipeline and warps (mb15, cp16,
tma15, tma12), the consumer forms present (f0 / f1 / f2: all regular blocks, one loose block first, all loose; m: the
cp.async kernel's masked form), a k-split > 1 (ks), the pad layout (pad1), the widest tensor-map box (b8 / b32 / b128),
a multi-tile plan (tiles), the slab depth (kbN) and the row splits (nsN, last1 = a last split of one row, mid = a last
split that ends inside a slab).

Data.  EXACT: integers in [-2^13, 2^13] times 2^s per column (s in [-200, 200]), with the intercept column of ones and
an all-zero column: every partial sum of every dot product is an exact float64 (n <= 2^26), so every pipeline, knob,
split and budget must return the bits of any float64 GEMM of the same data -- a dropped, doubled or misplaced row,
chunk, slot, fragment or split cannot hide.  FULL MANTISSA: zero-mean Gaussian and positive U(0,1)^2 columns (partial
sums grow linearly) times 2^s, s in [-30, 30], four rows 2^24 larger, against a long-double dot product; per entry both the deterministic bound
gamma_L sum|a b| and the probabilistic one 8 sqrt(L) u sum|a b| (u = 2^-53, L = ceil(rows_per_split / ksplit) + nsplit
ksplit): a scheme that is exact on small integers but drops mantissa bits fails these.

Layout poison in every case: rows [n, ld) of every column and of y are NaN, so are the gap columns, the columns past
p_old + c + gap of a wider buffer and the output block before the call; skipped below-diagonal fragments must read
exactly 0, and fokl_gram_scatter into a NaN-filled G with ldg > P must write exactly the block's rows and columns."""
import ctypes
import math
import os

import numpy as np
import pytest

import emu

pytestmark = pytest.mark.gpu

EINVAL = -1
U = 2.0 ** -53
KNOBS = ('FOKL_GRAM_KERNEL', 'FOKL_GRAM_WARPS', 'FOKL_GRAM_KB', 'FOKL_GRAM_STAGES', 'FOKL_GRAM_KSPLIT', 'FOKL_GRAM_PLACE')
PIPE_NAMES = {0: 'cp', 1: 'mb', 2: 'tma'}
N_A = 4097                     # rows of the shape matrix: 16 full 256-row slabs + one row


# ---- fixture: a private context (SM budgets and knobs never leak into the session engine) -----------------------------
@pytest.fixture(scope='module')
def gctx():
    import torch
    from FoKL import _lib
    lib = _lib.load()
    torch.cuda.set_device(0)
    torch.zeros(1, device='cuda:0')
    ctx = ctypes.c_void_p()
    assert lib.fokl_ctx_create(ctypes.byref(ctx), 0, None) == 0
    yield lib, ctx
    torch.cuda.synchronize()
    lib.fokl_ctx_destroy(ctx)


@pytest.fixture(autouse=True)
def _no_inherited_knobs(monkeypatch):
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)


def _report(tag, ratio):
    """Largest err / (sqrt(L) u sum|ab|) of a full-mantissa case, appended to $FOKL_GRAM_REF_REPORT when set."""
    path = os.environ.get('FOKL_GRAM_REF_REPORT')
    if path:
        with open(path, 'a') as f:
            f.write('%s %.4g\n' % (tag, ratio))


# ---- data ---------------------------------------------------------------------------------------------------------------
def exact_data(rng, p, n):
    """(p + 1, n): logical columns old | new | y, each integers in [-2^13, 2^13] times 2^s; column 0 = ones, column 2
    (when p > 2) all zero."""
    A = rng.integers(-2 ** 13, 2 ** 13 + 1, size=(p + 1, n)).astype(np.float64)
    A *= np.ldexp(1.0, rng.integers(-200, 201, size=p + 1))[:, None]
    A[0] = 1.0
    if p > 2:
        A[2] = 0.0
    return A


def full_data(rng, p, n, family):
    """Full-mantissa columns.  Four rows are 2^24 times larger than the rest, so that a handful of products dominate
    every sum: operand bits a kernel drops there cannot average out over the rows."""
    A = rng.standard_normal((p + 1, n)) if family == 'gauss' else rng.random((p + 1, n)) ** 2
    A[:, np.unique([0, n // 3, n // 2, n - 1])] *= 2.0 ** 24
    A *= np.ldexp(1.0, rng.integers(-30, 31, size=p + 1))[:, None]
    A[0] = 1.0
    return A


def exact_ref(A, p_old, c, rows=None):
    """Exact block (p + 1) x c (logical rows) of exact data: any float64 GEMM."""
    p = p_old + c
    n = A.shape[1]
    if (p + 1) * c * n < 10 ** 8:
        return A @ A[p_old:p].T
    import torch
    Ad = torch.from_numpy(A).cuda()
    return (Ad @ Ad[p_old:p].T).cpu().numpy()


def skipped_mask(p_old, c, cross_only=False):
    """Entries the kernel must leave 0: 8 x 8 fragments of the new x new part entirely below the diagonal (every new row
    for a cross-only block)."""
    p = p_old + c
    a, j = np.meshgrid(np.arange(p + 1) - p_old, np.arange(c), indexing='ij')
    new = (a >= 0) & (a < c)
    return new if cross_only else new & (a // 8 > j // 8)


# ---- device layout + call -------------------------------------------------------------------------------------------------
def layout(A, p_old, c, joint, gap=0, extra=0, ld_pad=0):
    """[y | X] buffer (row 0 = y when joint), X's columns old | gap | new | extra; NaN everywhere but the data."""
    import torch
    n = A.shape[1]
    p = p_old + c
    ld = -(-n // 16) * 16 + ld_pad
    full = torch.full((1 + p + gap + extra, ld), float('nan'), dtype=torch.float64, device='cuda:0')
    Ad = torch.from_numpy(A).cuda()
    full[1:1 + p_old, :n] = Ad[:p_old]
    full[1 + p_old + gap:1 + p + gap, :n] = Ad[p_old:p]
    if joint:
        full[0, :n] = Ad[p]
        y = full[0]
    else:
        y = torch.full((ld,), float('nan'), dtype=torch.float64, device='cuda:0')
        y[:n] = Ad[p]
    return full, y, ld


def last_config(lib, ctx):
    cfg = np.zeros(9, dtype=np.int64)
    assert lib.fokl_gram_last_config(ctx, cfg.ctypes.data) == 0
    return dict(pipe=int(cfg[0]), warps=int(cfg[1]), kb=int(cfg[2]), stages=int(cfg[3]), n_tiles=int(cfg[4]),
                nsplit=int(cfg[5]), rows_per_split=int(cfg[6]), max_slots=int(cfg[7]), cap=int(cfg[8]))


def call(gctx, X_ptr, y_ptr, ld, n, p_old, c, gap=0, cross_only=False, budget=0, twice=True):
    """fokl_gram_update_ex into an NaN-filled block; runs twice and requires the same bits (determinism)."""
    import torch
    lib, ctx = gctx
    p = p_old + c
    assert lib.fokl_ctx_set_sm_budget(ctx, budget) == 0
    outs = []
    for _ in range(2 if twice else 1):
        block = torch.full(((p + 1) * c,), float('nan'), dtype=torch.float64, device='cuda:0')
        rc = lib.fokl_gram_update_ex(ctx, X_ptr, ld, n, p_old, c, p_old + gap, 1 if cross_only else 0, y_ptr,
                                     block.data_ptr())
        assert rc == 0, lib.fokl_last_error(ctx)
        assert lib.fokl_ctx_synchronize(ctx) == 0, lib.fokl_last_error(ctx)
        outs.append(block)
    lib.fokl_ctx_set_sm_budget(ctx, 0)
    got = outs[0].cpu().numpy().reshape(p + 1, c)
    if twice:
        assert np.array_equal(got.view(np.int64), outs[1].cpu().numpy().reshape(p + 1, c).view(np.int64))
    return got, outs[0], last_config(lib, ctx)


def run(gctx, A, p_old, c, joint=False, gap=0, extra=3, ld_pad=0, cross_only=False, budget=0):
    full, y, ld = layout(A, p_old, c, joint, gap, extra, ld_pad)
    got, dev, cfg = call(gctx, full[1].data_ptr(), y.data_ptr(), ld, A.shape[1], p_old, c, gap, cross_only, budget)
    del full, y
    return got, dev, cfg


# ---- path check -----------------------------------------------------------------------------------------------------------
def plan_of(cfg, p_old, c, gap=0, cross_only=False):
    """The host plan the library ran (same cap, warps, kb / 16 and placement)."""
    place = int(os.environ.get('FOKL_GRAM_PLACE', '2'))
    force_r = int(os.environ.get('FOKL_GRAM_KSPLIT', '0'))
    rc, _, _, st = emu.gram_plan(None, p_old, c, cap=cfg['cap'], warps=cfg['warps'],
                                 kchunks=cfg['kb'] // 16 if cfg['pipe'] else 1, mode=place, gap=gap,
                                 cross_only=cross_only, allow_loose=cfg['pipe'] != 0, force_r=force_r)
    assert rc == 0, rc
    assert st['n_tiles'] == cfg['n_tiles'] and st['max_slots'] == cfg['max_slots'], (st, cfg)
    return st


def check_path(cfg, claim, p_old, c, n, gap=0, cross_only=False):
    st = plan_of(cfg, p_old, c, gap, cross_only)
    last = n - (cfg['nsplit'] - 1) * cfg['rows_per_split']
    assert 1 <= last <= cfg['rows_per_split'] and cfg['rows_per_split'] % cfg['kb'] == 0
    forms = {f for f in (0, 1, 2) if st['flex%d' % f] > 0}
    for tok in claim.split('-'):
        if tok[:2] in ('mb', 'cp') or tok.startswith('tma'):
            name = tok.rstrip('0123456789')
            assert (PIPE_NAMES[cfg['pipe']], cfg['warps']) == (name, int(tok[len(name):])), (claim, cfg)
        elif tok == 'm':
            assert st['flex1'] + st['flex2'] > 0, st
        elif tok[0] == 'f':
            assert forms == {int(d) for d in tok[1:]}, (claim, st)
        elif tok == 'ks':
            assert st['max_ksplit'] > 1, st
        elif tok.startswith('pad'):
            assert st['pad'] == int(tok[3:]), st
        elif tok[0] == 'b' and tok[1:].isdigit():
            assert max(k for k in (8, 32, 128) if st['box%d' % k] > 0) == int(tok[1:]), st
        elif tok == 'tiles':
            assert cfg['n_tiles'] > 1, cfg
        elif tok.startswith('kb'):
            assert cfg['kb'] == int(tok[2:]), (claim, cfg)
        elif tok.startswith('ns'):
            assert cfg['nsplit'] == int(tok[2:]), (claim, cfg)
        elif tok == 'last1':
            assert last == 1, (cfg, n)
        elif tok == 'mid':
            assert last % cfg['kb'] != 0, (cfg, n)
        else:
            raise AssertionError('unknown form token ' + tok)
    # the bulk-copy kernel's run table holds max_slots / 2 runs
    assert st['max_runs'] <= cfg['max_slots'] // 2
    return st


# ---- value checks ---------------------------------------------------------------------------------------------------------
def check_exact(got, A, p_old, c, cross_only=False, ref=None):
    ref = exact_ref(A, p_old, c) if ref is None else ref
    want = np.where(skipped_mask(p_old, c, cross_only), 0.0, ref)
    bad = ~(got == want)
    assert not bad.any(), 'wrong entries (row, col): %s' % (np.argwhere(bad)[:10].tolist(),)
    return ref


def error_L(cfg, st):
    return max(math.ceil(cfg['rows_per_split'] / ks) + cfg['nsplit'] * ks for ks in {st['min_ksplit'], st['max_ksplit']})


def check_full(got, A, p_old, c, cfg, st, tag, entries=None, cross_only=False):
    """Long-double reference per entry (all of them, or `entries` = (rows, cols)); A[q] is logical column q (an array or
    a dict of the columns the entries need).  Returns the largest err / (sqrt(L) u sum|ab|)."""
    L = error_L(cfg, st)
    gamma = L * U / (1 - L * U)
    skip = skipped_mask(p_old, c, cross_only)
    rows, cols = np.nonzero(~skip) if entries is None else entries
    worst = 0.0
    for r in np.unique(rows):
        js = np.asarray(cols)[np.asarray(rows) == r]
        a, al = A[r], A[r].astype(np.longdouble)
        for j0 in range(0, len(js), 16):
            jj = js[j0:j0 + 16]
            B = np.stack([A[p_old + j] for j in jj])
            ref = (al[None, :] * B.astype(np.longdouble)).sum(axis=1)      # pairwise along the contiguous axis
            absum = np.abs(a[None, :] * B).sum(axis=1)
            err = np.abs(got[r, jj].astype(np.longdouble) - ref).astype(np.float64)
            assert np.all(err <= gamma * absum), (tag, int(r), jj.tolist())
            ratio = err / (np.sqrt(L) * U * absum + 1e-300)
            assert np.all(ratio <= 8.0), (tag, int(r), float(ratio.max()))
            worst = max(worst, float(ratio.max()))
    assert np.all(got[skip] == 0.0)
    _report(tag + ' L=%d' % L, worst)
    return worst


def check_scatter(gctx, block_dev, got, p_old, c):
    """fokl_gram_scatter into NaN-filled G (ldg = P + 5) and Xty: exactly the block's rows / columns, exactly symmetric."""
    import torch
    lib, ctx = gctx
    p = p_old + c
    ldg = p + 5
    G = torch.full((ldg, ldg), float('nan'), dtype=torch.float64, device='cuda:0')
    Xty = torch.full((ldg,), float('nan'), dtype=torch.float64, device='cuda:0')
    assert lib.fokl_gram_scatter(ctx, block_dev.data_ptr(), p_old, c, G.data_ptr(), ldg, Xty.data_ptr()) == 0
    torch.cuda.synchronize()
    Gh, Xh = G.cpu().numpy(), Xty.cpu().numpy()
    want = np.full((ldg, ldg), np.nan)
    for j in range(c):
        col = got[:p, j].copy()
        col[p_old + j + 1:p] = got[p_old + j, j + 1:]       # below-diagonal new rows: the mirrored upper entries
        want[:p, p_old + j] = col
        want[p_old + j, :p] = col
    wx = np.full(ldg, np.nan)
    wx[p_old:p] = got[p]
    assert np.array_equal(Gh, want, equal_nan=True)
    assert np.array_equal(Gh, Gh.T, equal_nan=True)
    assert np.array_equal(Xh, wx, equal_nan=True)


def set_knobs(monkeypatch, **kw):
    names = dict(kernel='FOKL_GRAM_KERNEL', warps='FOKL_GRAM_WARPS', kb='FOKL_GRAM_KB', stages='FOKL_GRAM_STAGES',
                 ksplit='FOKL_GRAM_KSPLIT', place='FOKL_GRAM_PLACE')
    for k, v in kw.items():
        if v is not None:
            monkeypatch.setenv(names[k], str(v))


# variant -> (joint layout, ld % 16, knobs)
VARIANTS = {
    'sep': (False, 0, {}),
    'jointld2': (True, 2, {}),                         # [y | X] but ld % 16 == 2: not TMA-eligible
    'tma': (True, 0, dict(kernel='tma')),
    'tma12': (True, 0, dict(kernel='tma', warps=12)),
    'cpasync': (False, 0, dict(kernel='cpasync')),
    'mb': (False, 0, dict(kernel='mb')),
}

# (a) shapes x pipelines at the default knobs, n = 4097.  Claims: separate y (default dispatch), joint + tma, joint + tma
# + 12 warps, cp.async; the joint layout with ld % 16 == 2 dispatches as separate y.
SHAPES_A = [
    ((0, 1), ('mb15-f1-ks-ns17', 'tma15-f1-ks-b8-ns17', 'tma12-f1-ks-b8-ns17', 'cp16-m-ns17')),
    ((1, 1), ('mb15-f1-ks-ns17', 'tma15-f1-ks-b8-ns17', 'tma12-f1-ks-b8-ns17', 'cp16-m-ns17')),
    ((1, 7), ('mb15-f1-ks-ns17', 'tma15-f1-ks-b8-ns17', 'tma12-f1-ks-b8-ns17', 'cp16-m-ns17')),
    ((1, 8), ('mb15-f1-ks-ns17', 'tma15-f1-ks-b8-ns17', 'tma12-f1-ks-b8-ns17', 'cp16-m-ns17')),
    ((1, 9), ('mb15-f1-ks-ns17', 'tma15-f1-ks-b8-ns33', 'tma12-f1-ks-b8-ns33', 'cp16-m-ns33')),
    ((7, 16), ('mb15-f1-ks-ns17', 'tma15-f1-ks-b8-ns33', 'tma12-f1-ks-b8-ns33', 'cp16-m-ns33')),
    ((8, 17), ('mb15-f01-ks-pad1-ns17', 'tma15-f01-ks-pad1-b8-ns33', 'tma12-f01-ks-pad1-b8-ns33', 'cp16-m-pad1-ns65')),
    ((9, 24), ('mb15-f01-ks-pad1-ns17', 'tma15-f01-ks-pad1-b8-ns33', 'tma12-f01-ks-pad1-b8-ns33', 'cp16-m-pad1-ns65')),
    ((16, 33), ('mb15-f01-ns33', 'tma15-f01-b32-ns65', 'tma12-f01-b32-ns65', 'cp16-m-ns65')),
    ((50, 8), ('mb15-f1-ks-ns33', 'tma15-f1-ks-b32-ns65', 'tma12-f1-ks-b32-ns65', 'cp16-m-ns65')),
    ((14, 56), ('mb15-f01-pad1-ns33', 'tma15-f01-pad1-b32-ns65', 'tma12-f01-pad1-b32-ns65', 'cp16-m-pad1-ns65')),
    ((1, 146), ('cp16-m-ns129', 'tma15-f012-b128-ns129', 'tma12-f012-b128-tiles-ns65', 'cp16-m-ns129')),
    ((28, 168), ('cp16-m-pad1-tiles-ns65', 'tma15-f01-pad1-b128-tiles-ns65', 'tma12-f01-pad1-b128-tiles-ns65',
                 'cp16-m-pad1-tiles-ns65')),
    ((58, 168), ('cp16-m-pad1-tiles-ns65', 'tma15-f01-pad1-b128-tiles-ns65', 'tma12-f01-pad1-b128-tiles-ns43',
                 'cp16-m-pad1-tiles-ns65')),
    ((130, 40), ('cp16-m-ns129', 'tma15-f01-b128-ns129', 'tma12-f01-b128-ns129', 'cp16-m-ns129')),
    ((20, 300), ('cp16-m-tiles-ns37', 'tma15-f01-b128-tiles-ns37', 'tma12-f01-b128-tiles-ns29', 'cp16-m-tiles-ns37')),
    ((400, 17), ('cp16-m-tiles-ns65', 'tma15-f01-b128-tiles-ns65', 'tma12-f012-b128-tiles-ns65', 'cp16-m-tiles-ns65')),
]
CASES_A = []
for (_p_old, _c), (_sep, _tma, _tma12, _cp) in SHAPES_A:
    for _v, _cl in (('sep', _sep), ('jointld2', _sep), ('tma', _tma), ('tma12', _tma12), ('cpasync', _cp)):
        CASES_A.append(pytest.param(_p_old, _c, _v, _cl, id='%d+%d-%s-%s' % (_p_old, _c, _v, _cl)))


@pytest.mark.parametrize('p_old,c,variant,claim', CASES_A)
def test_shape_matrix_exact(gctx, monkeypatch, p_old, c, variant, claim):
    """(a) every shape x pipeline at the default knobs, exact data: the bits of a float64 GEMM, NaN poison never read,
    skipped fragments 0, scatter exact and symmetric, two runs identical."""
    joint, ld_pad, knobs = VARIANTS[variant]
    set_knobs(monkeypatch, **knobs)
    A = exact_data(np.random.default_rng(1000 * p_old + c), p_old + c, N_A)
    got, dev, cfg = run(gctx, A, p_old, c, joint=joint, ld_pad=ld_pad)
    check_path(cfg, claim, p_old, c, N_A)
    check_exact(got, A, p_old, c)
    check_scatter(gctx, dev, got, p_old, c)


# shapes of the earlier numpy comparison: separate y (default dispatch) and [y | X] with the tensor-map kernel forced
LEGACY = [((1, 1, 1), 'cp16-kb16-ns1', 'tma15-kb16-ns1'), ((10, 1, 2), 'cp16-kb16-ns1', 'tma15-kb16-ns1'),
          ((33, 3, 5), 'cp16-kb16-ns3', 'tma15-kb16-ns3'), ((1000, 9, 8), 'mb15-kb128-ns8', 'tma15-kb128-ns8'),
          ((4097, 63, 1), 'mb15-kb128-ns33', 'tma15-kb64-ns65'), ((4097, 64, 64), 'cp16-kb32-ns129', 'tma15-kb32-ns129'),
          ((2500, 65, 67), 'cp16-kb32-ns79', 'tma15-kb32-ns79'), ((100000, 130, 40), 'cp16-kb32-ns143', 'tma15-kb32-ns143'),
          ((300001, 20, 168), 'cp16-kb32-ns74', 'tma15-kb32-ns74')]


@pytest.mark.parametrize('joint', [False, True])
@pytest.mark.parametrize('shape,claim_sep,claim_tma', LEGACY)
def test_gram_block_matches_reference(gctx, monkeypatch, shape, claim_sep, claim_tma, joint):
    """Exact data: the bits of a float64 GEMM; Gaussian data: the long-double bounds (all entries, or a sample where
    n (p + 1) c > 5e8); both scattered exactly and symmetrically."""
    n, p_old, c = shape
    if joint:
        set_knobs(monkeypatch, kernel='tma')
    rng = np.random.default_rng(n + p_old)
    A = exact_data(rng, p_old + c, n)
    got, dev, cfg = run(gctx, A, p_old, c, joint=joint)
    check_path(cfg, claim_tma if joint else claim_sep, p_old, c, n)
    check_exact(got, A, p_old, c)
    check_scatter(gctx, dev, got, p_old, c)
    # fokl_gram_update is fokl_gram_update_ex with the new block right behind the old one
    import torch
    lib, ctx = gctx
    full, y, ld = layout(A, p_old, c, joint)
    blk = torch.full(((p_old + c + 1) * c,), float('nan'), dtype=torch.float64, device='cuda:0')
    assert lib.fokl_gram_update(ctx, full[1].data_ptr(), ld, n, p_old, c, y.data_ptr(), blk.data_ptr()) == 0
    torch.cuda.synchronize()
    assert np.array_equal(blk.cpu().numpy().reshape(got.shape).view(np.int64), got.view(np.int64))
    del full, y
    B = full_data(rng, p_old + c, n, 'gauss')
    got, dev, cfg = run(gctx, B, p_old, c, joint=joint)
    st = plan_of(cfg, p_old, c)
    entries = _sample_entries(np.random.default_rng(3), p_old, c, 256) if n * (p_old + c + 1) * c > 5e8 else None
    check_full(got, B, p_old, c, cfg, st, 'legacy n=%d %d+%d %s' % (n, p_old, c, 'tma' if joint else 'sep'), entries)
    check_scatter(gctx, dev, got, p_old, c)


# (b) knob sweeps: every slab depth x every ring depth the dispatcher's shared-memory check accepts, every forced
# k-split and placement, on four shapes; exact data, so every setting must give the same bits.
SWEEP_SHAPES = [(1, 9), (8, 17), (50, 8), (1, 146)]


def _smem_accepts(pipe, slots, kb, stages):
    import torch
    cap = torch.cuda.get_device_properties(0).shared_memory_per_block_optin - 1024
    if pipe == 'tma':
        need = stages * (kb // 16) * slots * 128 + 2 * 8 * 8 + 1024
    else:
        need = stages * slots * (kb + 4) * 8 + slots * 8 + 2 * 4 * 8 + 16
    return need <= cap


@pytest.mark.parametrize('kb', [16, 32, 64, 128, 256])
@pytest.mark.parametrize('pipe', ['mb', 'cpasync', 'tma'])
@pytest.mark.parametrize('p_old,c', SWEEP_SHAPES)
def test_knob_sweep_slab_and_ring(gctx, monkeypatch, p_old, c, pipe, kb):
    """(b) FOKL_GRAM_KB x FOKL_GRAM_STAGES: accepted settings give the exact bits, the others FOKL_EINVAL with the block
    untouched."""
    import torch
    lib, ctx = gctx
    A = exact_data(np.random.default_rng(1000 * p_old + c), p_old + c, N_A)
    ref = exact_ref(A, p_old, c)
    joint = pipe == 'tma'
    full, y, ld = layout(A, p_old, c, joint, extra=3)
    st_range = range(2, 9) if pipe == 'tma' else range(3 if pipe == 'cpasync' else 2, 5)
    ran = 0
    for stages in st_range:
        set_knobs(monkeypatch, kernel=pipe, kb=kb, stages=stages)
        warps = 16 if pipe == 'cpasync' else 15
        slots = emu.gram_plan(None, p_old, c, cap=352, warps=warps, kchunks=1, mode=2,
                              allow_loose=pipe != 'cpasync')[3]['max_slots']
        if not _smem_accepts(pipe, slots, kb, stages):
            block = torch.full(((p_old + c + 1) * c,), float('nan'), dtype=torch.float64, device='cuda:0')
            rc = lib.fokl_gram_update_ex(ctx, full[1].data_ptr(), ld, N_A, p_old, c, p_old, 0, y.data_ptr(),
                                         block.data_ptr())
            assert rc == EINVAL
            assert torch.isnan(block).all()
            continue
        got, _, cfg = call(gctx, full[1].data_ptr(), y.data_ptr(), ld, N_A, p_old, c)
        claim = '%s%d-kb%d' % ({'mb': 'mb', 'cpasync': 'cp', 'tma': 'tma'}[pipe], warps, kb)
        check_path(cfg, claim, p_old, c, N_A)
        assert cfg['stages'] == stages
        check_exact(got, A, p_old, c, ref=ref)
        ran += 1
    if kb <= 32:
        assert ran > 0


@pytest.mark.parametrize('pipe', ['mb', 'tma'])
@pytest.mark.parametrize('p_old,c', SWEEP_SHAPES)
def test_knob_sweep_ksplit_and_placement(gctx, monkeypatch, p_old, c, pipe):
    """(b) FOKL_GRAM_KSPLIT in {1, 2, 4, 8, 16} and FOKL_GRAM_PLACE in {0, 1, 2}: the exact bits in every plan form."""
    A = exact_data(np.random.default_rng(1000 * p_old + c), p_old + c, N_A)
    ref = exact_ref(A, p_old, c)
    full, y, ld = layout(A, p_old, c, pipe == 'tma', extra=3)
    seen_split = set()
    for place in (0, 1, 2):
        for ks in (1, 2, 4, 8, 16):
            set_knobs(monkeypatch, kernel=pipe, ksplit=ks, place=place)
            got, _, cfg = call(gctx, full[1].data_ptr(), y.data_ptr(), ld, N_A, p_old, c)
            st = check_path(cfg, '%s15' % pipe, p_old, c, N_A)
            assert st['max_ksplit'] <= ks
            seen_split.add(st['max_ksplit'])
            check_exact(got, A, p_old, c, ref=ref)
    if c < 100:
        assert max(seen_split) >= 4, seen_split


# (c) row edges: n around every 16-row chunk and slab threshold (4 kb - 1, 4 kb), odd n for the cp.async 8-byte tail
ROW_NS = [1, 2, 15, 16, 17, 33, 127, 128, 255, 256, 257, 511, 512, 1023, 1024, 1025]


def _row_claim(p_old, c, variant, n):
    """The form the dispatcher picks (read off csrc/gram.cu): the deepest slab with n >= 4 kb that fits."""
    wide = c > 100
    if variant == 'mb':
        kb = 16 if wide or n < 256 else (64 if n < 512 else 128 if n < 1024 else 256)
        return 'mb15-kb%d' % kb
    small = 16 if n < 128 else 32
    if variant == 'cpasync':
        return 'cp16-kb%d' % (small if wide or n < 256 else 64)
    if variant == 'tma':
        return 'tma15-kb%d' % (small if wide or n < 256 else 64 if n < 512 else 128)
    if wide or n < 256:
        return ('tma15' if variant == 'joint' else 'cp16') + '-kb%d' % small
    return 'mb15-kb%d' % (64 if n < 512 else 128 if n < 1024 else 256)


CASES_C = [pytest.param(p_old, c, v, n, id='%d+%d-%s-n%d-%s' % (p_old, c, v, n, _row_claim(p_old, c, v, n)))
           for (p_old, c) in [(8, 17), (1, 146)] for v in ('sep', 'joint', 'mb', 'cpasync', 'tma') for n in ROW_NS]


@pytest.mark.parametrize('p_old,c,variant,n', CASES_C)
def test_row_edges(gctx, monkeypatch, p_old, c, variant, n):
    joint = variant in ('joint', 'tma')
    if variant in ('mb', 'cpasync', 'tma'):
        set_knobs(monkeypatch, kernel=variant)
    A = exact_data(np.random.default_rng(n), p_old + c, n)
    got, dev, cfg = run(gctx, A, p_old, c, joint=joint)
    check_path(cfg, _row_claim(p_old, c, variant, n), p_old, c, n)
    check_exact(got, A, p_old, c)


# (c) row splits under an SM budget (one tile, forced 64-row slabs): nsplit = budget, with a last split of one row
# and one that ends inside a slab
CASES_S = []
for _b in (1, 2, 9, 10, 11, 12, 13, 14, 15, 16, 17):
    for _edge, _n in (('last1', max(1, (_b - 1) * 128 + 1)), ('mid', (_b - 1) * 128 + 100)):
        for _pipe in ('mb', 'cpasync', 'tma'):
            _cl = '%s-kb64-ns%d-%s' % ({'mb': 'mb15', 'cpasync': 'cp16', 'tma': 'tma15'}[_pipe], _b, _edge)
            CASES_S.append(pytest.param(_b, _n, _pipe, id='budget%d-n%d-%s' % (_b, _n, _cl)))


@pytest.mark.parametrize('p_old,c', [(50, 8), (8, 17)])
@pytest.mark.parametrize('budget,n,pipe', CASES_S)
def test_row_splits_under_sm_budget(gctx, monkeypatch, p_old, c, budget, n, pipe):
    """nsplit = 1, nsplit mod 8 = 1 ... 7 and 0 (gram_reduce_kernel's 8-way body and its tail), a single-row last split and
    a last split ending mid-slab: exact bits, and every budget gives the same bits."""
    set_knobs(monkeypatch, kernel=pipe, kb=64, stages=4)       # (the ring depth picked for a short n may not fit kb = 64)
    A = exact_data(np.random.default_rng(n + budget), p_old + c, n)
    got, _, cfg = run(gctx, A, p_old, c, joint=pipe == 'tma', budget=budget)
    claim = '%s-kb64-ns%d-%s' % ({'mb': 'mb15', 'cpasync': 'cp16', 'tma': 'tma15'}[pipe], budget,
                                 'last1' if (n - 1) % 128 == 0 else 'mid')
    check_path(cfg, claim, p_old, c, n)
    check_exact(got, A, p_old, c)


# (d) gap and cross-only (fokl_gram_update_ex) in every pipeline
GAP_SHAPES = [(10, 1, 2, 3), (2500, 65, 67, 9), (100000, 30, 40, 168), (300001, 20, 168, 56)]
GAP_CLAIMS = {(10, 1, 2, 3): ('cp16', 'tma15', 'cp16'), (2500, 65, 67, 9): ('cp16', 'tma15', 'cp16'),
              (100000, 30, 40, 168): ('mb15', 'tma15', 'cp16'), (300001, 20, 168, 56): ('cp16', 'tma15', 'cp16')}
CASES_D = []
for _s in GAP_SHAPES:
    for _v, _cl in zip(('sep', 'tma', 'cpasync', 'mb'), GAP_CLAIMS[_s] + ('mb15',)):
        CASES_D.append(pytest.param(_s, _v, _cl, id='n%d-%d+%d-gap%d-%s-%s' % (_s + (_v, _cl))))


@pytest.mark.parametrize('shape,variant,claim', CASES_D)
def test_gap_and_cross_only(gctx, monkeypatch, shape, variant, claim):
    """New block `gap` NaN columns above the old ones: exact bits, and with full-mantissa data the same bits as the
    contiguous layout (the same plan); FOKL_GRAM_CROSS_ONLY: the (old | y) rows exact, every new row left 0."""
    n, p_old, c, gap = shape
    joint, _, knobs = VARIANTS[variant]
    set_knobs(monkeypatch, **knobs)
    rng = np.random.default_rng(n + gap)
    A = exact_data(rng, p_old + c, n)
    ref = None
    for g in (gap, 0):
        for cross in (False, True):
            got, _, cfg = run(gctx, A, p_old, c, joint=joint, gap=g, cross_only=cross)
            check_path(cfg, claim, p_old, c, n, gap=g, cross_only=cross)
            ref = check_exact(got, A, p_old, c, cross_only=cross, ref=ref)
    B = full_data(rng, p_old + c, n, 'gauss')
    g0 = run(gctx, B, p_old, c, joint=joint, gap=0)[0]
    gg = run(gctx, B, p_old, c, joint=joint, gap=gap)[0]
    assert np.array_equal(g0.view(np.int64), gg.view(np.int64))


@pytest.mark.parametrize('p_stable,k,c,gap,claim', [(58, 30, 168, 40, 'cp16-m-ns143'), (9, 1, 8, 3, 'mb15-kb256-ns131')])
def test_engine_cross_only_call(gctx, p_stable, k, c, gap, claim):
    """The engine's cross block (FoKL/_engine.py _append_split): X based at column p_stable of the [y | X] buffer, y the
    buffer's row 0 -- not in front of X, so never the tensor-map kernel; the old columns are the k survivors, the new
    block sits `gap` columns above them."""
    import torch
    n = 100001
    rng = np.random.default_rng(p_stable + k)
    A = exact_data(rng, k + c, n)                      # logical: k old | c new | y
    ld = -(-n // 16) * 16
    full = torch.full((1 + p_stable + k + gap + c, ld), float('nan'), dtype=torch.float64, device='cuda:0')
    Ad = torch.from_numpy(A).cuda()
    full[0, :n] = Ad[k + c]
    full[1:1 + p_stable, :n] = 7.0                    # stable columns: not part of this call
    full[1 + p_stable:1 + p_stable + k, :n] = Ad[:k]
    full[1 + p_stable + k + gap:, :n] = Ad[k:k + c]
    got, _, cfg = call(gctx, full[1 + p_stable].data_ptr(), full[0].data_ptr(), ld, n, k, c, gap, cross_only=True)
    check_path(cfg, claim, k, c, n, gap=gap, cross_only=True)
    check_exact(got, A, k, c, cross_only=True)


# (e) full-mantissa data on a subset that reaches every pipeline, FLEX form, k-split > 1 and nsplit > 8
CASES_E = [
    ((1, 9), 'sep', 'mb15-f1-ks'), ((1, 9), 'cpasync', 'cp16-m'), ((50, 8), 'tma', 'tma15-f1-ks-b32'),
    ((8, 17), 'sep', 'mb15-f01-ks-pad1'), ((1, 146), 'tma', 'tma15-f012-b128'), ((400, 17), 'tma12', 'tma12-f012-tiles'),
    ((58, 168), 'sep', 'cp16-m-pad1-tiles'), ((16, 33), 'mb', 'mb15-f01'), ((20, 300), 'tma', 'tma15-f01-b128-tiles'),
]


@pytest.mark.parametrize('family', ['gauss', 'basis'])
@pytest.mark.parametrize('shape,variant,claim', [pytest.param(*x, id='%d+%d-%s-%s' % (x[0] + x[1:])) for x in CASES_E])
def test_full_mantissa(gctx, monkeypatch, shape, variant, claim, family):
    p_old, c = shape
    n = 20001
    joint, ld_pad, knobs = VARIANTS[variant]
    set_knobs(monkeypatch, **knobs)
    A = full_data(np.random.default_rng(p_old * 7 + c), p_old + c, n, family)
    got, _, cfg = run(gctx, A, p_old, c, joint=joint, ld_pad=ld_pad)
    st = check_path(cfg, claim, p_old, c, n)
    assert cfg['nsplit'] > 8
    entries = None
    if n * (p_old + c + 1) * c > 5e8:
        entries = _sample_entries(np.random.default_rng(1), p_old, c, 256)
    check_full(got, A, p_old, c, cfg, st, 'e %d+%d %s %s' % (p_old, c, variant, family), entries)


def _sample_entries(rng, p_old, c, k):
    """Every entry of the block's first and last 8 x 8 fragment, the y row's first and last 8, plus k random entries
    (never a skipped one)."""
    p = p_old + c
    rows, cols = [], []
    for r0, c0 in ((0, 0), (max(0, p - 7), max(0, c - 8))):
        for r in range(r0, min(r0 + 8, p + 1)):
            for j in range(c0, min(c0 + 8, c)):
                rows.append(r); cols.append(j)
    skip = skipped_mask(p_old, c)
    ok = np.argwhere(~skip)
    pick = ok[rng.choice(len(ok), size=min(k, len(ok)), replace=False)]
    rows += list(pick[:, 0]); cols += list(pick[:, 1])
    rows += [p] * min(c, 8); cols += list(range(min(c, 8)))
    e = np.unique(np.array([rows, cols]).T, axis=0)
    e = e[~skip[e[:, 0], e[:, 1]]]
    return e[:, 0], e[:, 1]


# (f) production sizes in the engine's own [y | X] buffer with the default dispatch
def _device_exact(full, rows, n, seed):
    import torch
    g = torch.Generator(device='cuda:0')
    g.manual_seed(seed)
    for r in rows:
        v = torch.randint(-2 ** 13, 2 ** 13 + 1, (n,), generator=g, device='cuda:0', dtype=torch.int32).double()
        s = int(torch.randint(-200, 201, (1,), generator=g, device='cuda:0').item())
        full[r, :n] = v * 2.0 ** s
        del v


@pytest.mark.parametrize('p_old,c,n,claim', [
    pytest.param(58, 168, 10 ** 7, 'tma15-f01-pad1-b128-tiles-ns74', id='cfg4-58+168-N1e7-tma15-f01-pad1-b128-tiles-ns74'),
    pytest.param(400, 1680, 10 ** 6, 'tma15-f01-b128-tiles-ns1', id='cfg5-400+1680-N1e6-tma15-f01-b128-tiles-ns1'),
])
def test_production_sizes_exact(gctx, p_old, c, n, claim):
    """The engine's widest substage shapes, bit for bit against a device GEMM (~18 GB of design matrix each)."""
    import torch
    p = p_old + c
    ld = -(-n // 16) * 16
    full = torch.full((1 + p, ld), float('nan'), dtype=torch.float64, device='cuda:0')
    _device_exact(full, range(1 + p), n, p)
    full[1, :n] = 1.0
    full[3, :n] = 0.0
    try:
        got, _, cfg = call(gctx, full[1].data_ptr(), full[0].data_ptr(), ld, n, p_old, c)
        check_path(cfg, claim, p_old, c, n)
        D = full[:, :n]
        R = (D @ D[1 + p_old:1 + p].T).cpu().numpy()    # buffer order: y first
        ref = np.concatenate([R[1:], R[:1]])
        want = np.where(skipped_mask(p_old, c), 0.0, ref)
        bad = ~(got == want)
        assert not bad.any(), np.argwhere(bad)[:10].tolist()
    finally:
        del full
        torch.cuda.empty_cache()


def test_production_cfg4_full_mantissa_sampled(gctx):
    """cfg4's widest substage (58 + 168, N = 1e7) with Gaussian data: long-double reference on sampled entries."""
    import torch
    p_old, c, n = 58, 168, 10 ** 7
    p = p_old + c
    ld = n
    full = torch.empty((1 + p, ld), dtype=torch.float64, device='cuda:0')
    g = torch.Generator(device='cuda:0')
    g.manual_seed(5)
    for r in range(1 + p):
        full[r] = torch.randn(n, generator=g, device='cuda:0', dtype=torch.float64) * 2.0 ** ((r * 7) % 61 - 30)
    full[:, [0, n // 3, n // 2, n - 1]] *= 2.0 ** 24     # dominant rows, as in full_data
    full[1] = 1.0
    try:
        got, _, cfg = call(gctx, full[1].data_ptr(), full[0].data_ptr(), ld, n, p_old, c)
        st = check_path(cfg, 'tma15-f01-pad1-b128-tiles-ns74', p_old, c, n)
        rng = np.random.default_rng(2)
        rows = np.unique(np.concatenate([[0, p_old - 1, p_old, p - 1, p], rng.choice(p, 3, replace=False)]))
        cols = np.unique(np.concatenate([[0, c - 1], rng.choice(c, 4, replace=False)]))
        rr, cc = np.meshgrid(rows, cols, indexing='ij')
        rr, cc = rr.ravel(), cc.ravel()
        keep = ~skipped_mask(p_old, c)[rr, cc]
        rr, cc = rr[keep], cc[keep]
        need = sorted(set(rr.tolist()) | set((p_old + cc).tolist()))
        # logical column q of the block = buffer row q + 1 (y = row 0)
        A = {q: full[0 if q == p else q + 1].cpu().numpy() for q in need}
        check_full(got, A, p_old, c, cfg, st, 'f cfg4 gauss', entries=(rr, cc))
    finally:
        del full
        torch.cuda.empty_cache()


# (h) error paths: FOKL_EINVAL, block untouched
def test_error_paths_leave_the_block_untouched(gctx, monkeypatch):
    import torch
    lib, ctx = gctx
    p_old, c, n = 8, 17, 1000
    A = exact_data(np.random.default_rng(0), p_old + c, n)
    full, y, ld = layout(A, p_old, c, True)
    X = full[1].data_ptr()
    Y = y.data_ptr()
    block = torch.full(((p_old + c + 1) * c,), float('nan'), dtype=torch.float64, device='cuda:0')
    B = block.data_ptr()
    cases = {
        'odd ld': (X, Y, ld + 1, n, p_old, c, p_old, 0),
        'X misaligned': (X + 8, Y, ld, n, p_old, c, p_old, 0),
        'y misaligned': (X, Y + 8, ld, n, p_old, c, p_old, 0),
        'ld < n': (X, Y, n - 2, n, p_old, c, p_old, 0),
        'c = 0': (X, Y, ld, n, p_old, 0, p_old, 0),
        'n = 0': (X, Y, ld, 0, p_old, c, p_old, 0),
        'new_col0 < p_old': (X, Y, ld, n, p_old, c, p_old - 1, 0),
        'cross-only without old columns': (X, Y, ld, n, 0, c, 0, 1),
        'more than 65000 columns': (X, Y, ld, n, 64990, 10, 64990, 0),
    }
    for name, (x, yy, l, nn, po, cc, col0, flags) in cases.items():
        rc = lib.fokl_gram_update_ex(ctx, x, l, nn, po, cc, col0, flags, yy, B)
        assert rc == EINVAL, name
    # a forced slab that does not fit shared memory: 160 staged columns x 256-row slabs on the bulk-copy ring
    A2 = exact_data(np.random.default_rng(1), 147, 2048)
    full2, y2, ld2 = layout(A2, 1, 146, False)
    set_knobs(monkeypatch, kernel='mb', kb=256)
    assert lib.fokl_gram_update_ex(ctx, full2[1].data_ptr(), ld2, 2048, 1, 146, 1, 0, y2.data_ptr(), B) == EINVAL
    torch.cuda.synchronize()
    assert torch.isnan(block).all()
