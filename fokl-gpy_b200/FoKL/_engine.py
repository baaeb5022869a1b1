"""Device engine: owns the HBM-resident state of one `fit` and drives libfokl_b200.so through ctypes.

PyTorch is used only as the carrier of device memory, the CUDA stream and (multi-GPU) the NCCL process
group; every numerical stage is a hand-written sm_100a kernel behind the C ABI (include/fokl_b200.h).

HBM layout (all float64):
    x     [M][ldx]     normalised inputs, column-major (one input per row of the tensor), ldx = ceil16(N)
    y     [ldx]        data
    X     [Pcap][ld]   design matrix, column-major: X[j] is column j (N doubles), column 0 = ones; allocated as
                       rows 1.. of a [1 + Pcap][ld] buffer whose row 0 is a copy of y, so that K2 sees [y | X] as one
                       2-D tensor (TMA tensor maps, csrc/gram.cu)
    G     [Gcap][Gcap] master Gram X'X of the columns currently in X (symmetric), Xty [Gcap]
Multi-GPU: every rank holds N/world rows of x, y, X; Gram blocks are summed with one NCCL allreduce per
substage, after which every rank owns the full G (SURVEY section 8e, axis 1).
"""
import contextlib
import ctypes
import math
import os
import warnings

import numpy as np

from . import _lib

CUBIC = 'Cubic Splines'
BERNOULLI = 'Bernoulli Polynomials'


def _round_up(v, m):
    return ((int(v) + m - 1) // m) * m


def pack_phis(phis, kernel):
    """Reference `phis` structure -> dense float64 table (cubic [n][n_piece][4]; Bernoulli [n][width])."""
    n = len(phis)
    if kernel == CUBIC:
        n_piece = len(phis[0][0])
        tab = np.empty((n, n_piece, 4), dtype=np.float64)
        for s in range(n):
            for k in range(4):
                tab[s, :, k] = phis[s][k]
        return tab
    width = max(len(r) for r in phis)
    tab = np.zeros((n, max(width, 2)), dtype=np.float64)
    for s in range(n):
        tab[s, :len(phis[s])] = phis[s]
    return tab


class DeviceDataset:
    """Normalised inputs and data resident in HBM (this rank's row shard)."""

    def __init__(self, x, y, n, m, ldx):
        self.x, self.y, self.n, self.m, self.ldx = x, y, n, m, ldx


class CandidateResult:
    __slots__ = ('ev', 'info', 'stats', 'betas', 'sigs', 'taus', 'betahat', 'lamb', 'Q', 'p', 'vec_off', 'mat_off',
                 'draws', 'refined', 'stats_host')

    def betas_of(self, c):
        o = self.draws * self.vec_off[c]
        return self.betas[o:o + self.draws * self.p[c]].view(self.draws, self.p[c])

    def stats_of(self, c):
        o = 3 * self.vec_off[c]
        return self.stats[o:o + 3 * self.p[c]].view(3, self.p[c])


class PendingCandidates:
    """A batch of candidate models enqueued by Engine.evaluate_launch; finish() reads the BICs back."""

    def __init__(self, engine, res, ev, info, col_sets, side, keep_alive):
        self.engine, self.res, self.ev, self.info = engine, res, ev, info
        self.col_sets, self.side, self.keep_alive = col_sets, side, keep_alive

    def _unpack(self, h):
        res, n = self.res, len(self.col_sets)
        n_i = (n + 1) // 2
        res.ev = h[:n].copy()
        res.info = h[n:n + n_i].view(np.int32)[:n].copy()
        res.stats_host = h[n + n_i:] if res.stats is not None else None

    def finish(self, refine_tol=None):
        """Synchronise and return the CandidateResult.  refine_tol > 0: near-interpolating / degenerate fits are
        recomputed from an N-length residual pass over the *current* X (FR:1551), so the models must still be there."""
        eng, res = self.engine, self.res
        res.stats_host = None
        if self.side:
            # read back on the side stream itself: the main stream may hold later work (the next kill loop) that these
            # copies must not queue behind; afterwards the main stream may touch the batch's tensors
            with eng.torch.cuda.stream(eng.side_stream):
                self._unpack(self.pack.cpu().numpy())
            main_stream = eng.torch.cuda.current_stream(eng.device)
            main_stream.wait_stream(eng.side_stream)
            for tns in (self.pack, res.betas, res.sigs, res.taus, res.betahat, res.lamb, res.Q):
                if tns is not None:
                    tns.record_stream(main_stream)      # allocated on the side stream's pool, read on the main stream
        else:
            self._unpack(self.pack.cpu().numpy())
        res.refined = np.zeros(len(res.ev), dtype=bool)
        if refine_tol is not None and refine_tol > 0:
            bad = eng.refine_mask(res.ev, res.p, refine_tol)
            res.refined = bad
            for c in np.nonzero(bad)[0]:
                res.ev[c] = eng.residual_bic(self.col_sets[c],
                                             res.betahat[res.vec_off[c]:res.vec_off[c] + res.p[c]])
        self.keep_alive = None
        return res


class Engine:
    kill_from_eig = True      # kill_loop_launch(eig=...) is available (the selection loop asks before using it)

    def __init__(self, device=None, group=None):
        import torch
        self.torch = torch
        if not torch.cuda.is_available():
            raise RuntimeError("FoKL (B200 build) needs a CUDA device: there is no CPU fallback for fit().")
        self.lib = _lib.load()
        if device is None:
            device = torch.device('cuda', torch.cuda.current_device())
        self.device = torch.device(device)
        self.dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.group = group
        self.dist = None
        self.world = 1
        self.rank = 0
        if group is not None or (torch.distributed.is_available() and torch.distributed.is_initialized()
                                 and group is not False):
            self.dist = torch.distributed
            self.world = self.dist.get_world_size(group if group not in (None, False) else None)
            self.rank = self.dist.get_rank(group if group not in (None, False) else None)
            if self.world == 1:
                self.dist = None
        if group is False:
            self.group = None
        ctx = ctypes.c_void_p()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        rc = self.lib.fokl_ctx_create(ctypes.byref(ctx), self.dev_index, ctypes.c_void_p(stream))
        if rc != 0:
            raise RuntimeError("fokl_ctx_create failed with code %d" % rc)
        self.ctx = ctx
        self._phis_key = None
        self.kernel_id = None
        self.n_orders = 0
        self.ds = None
        self.X = self.Xfull = None
        self.P = 0
        self.G = self.Xty = self.G2 = self.Xty2 = self.G3 = self.Xty3 = None
        self.block = None
        self.n_global = 0
        self.sum_y = self.yty = 0.0
        self.gibbs_launch_batches = 0
        self.work = dict(eig_solves=0, chains_run=0, kill_loops=0, kill_proposals_scored=0, secular_steps=0)     # work counters (bench.py)
        self.profile = None      # set to {} to collect CUDA-event timings per stage (bench.py)
        self.ctx_side = None
        self.side_stream = None
        # build-ahead of the next substage's columns (prefetch_terms): its own context / stream, and the physical layout
        # of X while a block sits above a gap: logical column j lives at j (j < P_base) or j + gap (j >= P_base)
        self.ctx_pf = None
        self.pf_stream = None
        self.pf = None
        self.gap = 0
        self.P_base = 0

    # ------------------------------------------------------------------------------------------------
    def release(self):
        """Free the design-matrix buffer kept between fits."""
        self.X = self.Xfull = None
        self.Pcap = 0

    def close(self):
        self.X = self.Xfull = None
        if getattr(self, '_bounce_pool', None) is not None:
            self._bounce_pool.shutdown(wait=False)
            self._bounce_pool = self._bounce = None
        if getattr(self, 'ctx_side', None) is not None and self.ctx_side:
            self.lib.fokl_ctx_destroy(self.ctx_side)
            self.ctx_side = None
        if getattr(self, 'ctx_pf', None) is not None and self.ctx_pf:
            self.lib.fokl_ctx_destroy(self.ctx_pf)
            self.ctx_pf = None
        if getattr(self, 'ctx', None) is not None and self.ctx:
            self.lib.fokl_ctx_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            msg = self.lib.fokl_last_error(self.ctx)
            msg = msg.decode() if msg else ''
            if rc == _lib.ERANGE:
                raise ValueError(msg)
            raise RuntimeError("libfokl_b200 error %d: %s" % (rc, msg))

    def synchronize(self):
        self._ck(self.lib.fokl_ctx_synchronize(self.ctx))
        if self.ctx_pf is not None:
            rc = self.lib.fokl_ctx_synchronize(self.ctx_pf)      # also reports a range error of a build-ahead basis launch
            if rc != 0:
                msg = self.lib.fokl_last_error(self.ctx_pf)
                msg = msg.decode() if msg else ''
                if rc == _lib.ERANGE:
                    raise ValueError(msg)
                raise RuntimeError("libfokl_b200 error %d: %s" % (rc, msg))

    def launch_count(self):
        n = int(self.lib.fokl_launch_count(self.ctx))
        if getattr(self, 'ctx_side', None) is not None and self.ctx_side:
            n += int(self.lib.fokl_launch_count(self.ctx_side))
        return n

    def _allreduce(self, t):
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM, group=self.group)

    def ctl_allreduce(self, arr):
        """Sum a small host array over the ranks and return it (host).  Control traffic of the selection loop (two
        scalars per verified model): it travels on its OWN communicator and on the side stream, so it neither queues
        behind the Gram block's allreduce -- which waits for the K2 kernel the main stream is running -- nor orders
        the main stream after it."""
        torch = self.torch
        if self.dist is None:
            return arr
        if getattr(self, '_ctl_group', None) is None:
            ranks = None if self.group is None else self.dist.get_process_group_ranks(self.group)
            self._ctl_group = self.dist.new_group(ranks=ranks)
        self._side()
        with torch.cuda.stream(self.side_stream):
            t = torch.from_numpy(np.ascontiguousarray(arr)).to(self.device)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM, group=self._ctl_group)
            out = t.cpu().numpy()
        return out

    # ---- optional per-stage timing with CUDA events on the launching stream ------------------------
    def _tic(self):
        if self.profile is None:
            return None
        e = self.torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def _toc(self, start, name, **extra):
        if start is None:
            return
        e = self.torch.cuda.Event(enable_timing=True)
        e.record()
        self.profile.setdefault('_events', []).append((name, start, e, extra))

    def profile_summary(self):
        """Resolve recorded events: {stage: dict(ms=total, launches=count, **summed extras)}."""
        out = {}
        if not self.profile:
            return out
        self.torch.cuda.synchronize(self.device)
        for name, a, b, extra in self.profile.get('_events', []):
            d = out.setdefault(name, dict(ms=0.0, calls=0))
            d['ms'] += a.elapsed_time(b)
            d['calls'] += 1
            for k, v in extra.items():
                d[k] = d.get(k, 0) + v
        return out

    # ------------------------------------------------------------------------------------------------
    def set_phis(self, phis, kernel):
        key = (id(phis), kernel, len(phis))
        if key == self._phis_key:
            return
        tab = np.ascontiguousarray(pack_phis(phis, kernel))
        if getattr(self, '_phis_tab', None) is not None and self._phis_kernel == kernel and \
                self._phis_tab.shape == tab.shape and np.array_equal(self._phis_tab, tab):
            self._phis_key = key         # same table as the one already on the device (e.g. a second sp500() call)
            self._phis_ref = phis
            return
        if kernel == CUBIC:
            self._ck(self.lib.fokl_set_phis_cubic(self.ctx, tab.ctypes.data, tab.shape[0], tab.shape[1]))
            self.kernel_id = _lib.KERNEL_CUBIC
        elif kernel == BERNOULLI:
            self._ck(self.lib.fokl_set_phis_bernoulli(self.ctx, tab.ctypes.data, tab.shape[0], tab.shape[1]))
            self.kernel_id = _lib.KERNEL_BERNOULLI
        else:
            raise ValueError("The kernel %r is not currently supported." % (kernel,))
        self._pf_tab_key = None          # the build-ahead context uploads its own copy on next use
        self.n_orders = tab.shape[0]
        self._phis_tab, self._phis_kernel = tab, kernel
        self._phis_key = key
        self._phis_ref = phis   # keep alive so id() stays unique

    # ------------------------------------------------------------------------------------------------
    def upload(self, inputs, data):
        """Host numpy (N x M inputs, N or N x 1 data) -> DeviceDataset.  H2D copies + one transpose.  float32 inputs
        are widened (exactly) and column-major ones (a transposed view, a pandas frame's block) transposed on the
        device, so neither costs a host pass."""
        torch = self.torch
        inputs = np.asarray(inputs)
        if inputs.ndim == 1:
            inputs = inputs[:, None]
        if inputs.dtype not in (np.float32, np.float64):
            inputs = np.asarray(inputs, dtype=np.float64)
        column_major = not inputs.flags.c_contiguous and inputs.flags.f_contiguous
        if not column_major:
            inputs = np.ascontiguousarray(inputs)
        data = np.ascontiguousarray(np.asarray(data, dtype=np.float64).reshape(-1))
        n, m = inputs.shape
        if data.shape[0] != n:
            raise ValueError("inputs and data must have the same number of rows")
        ldx = _round_up(max(n, 1), 16)
        x = torch.zeros((m, ldx), dtype=torch.float64, device=self.device)
        y = torch.zeros((ldx,), dtype=torch.float64, device=self.device)
        if column_major:
            x[:, :n].copy_(self._h2d(inputs.T))
        else:
            x[:, :n].copy_(self._h2d(inputs).t())
        y[:n].copy_(self._h2d(data))
        self.h2d_bytes = inputs.nbytes + data.nbytes
        return DeviceDataset(x, y, n, m, ldx)

    def _h2d(self, a):
        """Contiguous float32 / float64 numpy array -> device tensor of the same shape and dtype.  Pinned host pages go
        out as one async DMA.  Ordinary (pageable) arrays -- what a user of `FoKL.fit(inputs, data)` passes -- would be
        staged by the driver through its own small bounce buffer at ~11 GB/s; from 64 MB up they are instead copied by a
        few host threads into two pinned buffers that alternate, each DMA overlapping the host copy of the next chunk."""
        torch = self.torch
        with warnings.catch_warnings():
            warnings.simplefilter('ignore', UserWarning)     # a read-only array (a pandas block) is only read here
            t = torch.from_numpy(a)
        if a.nbytes < (64 << 20) or t.is_pinned():
            return t.to(self.device, non_blocking=True)
        from concurrent.futures import ThreadPoolExecutor
        flat = a.reshape(-1)
        out = torch.empty(flat.shape[0], dtype=t.dtype, device=self.device)
        chunk = (32 << 20) // a.itemsize
        if getattr(self, '_bounce', None) is None:
            self._bounce = [torch.empty((32 << 20) // 8, dtype=torch.float64).pin_memory() for _ in range(2)]
            self._bounce_pool = ThreadPoolExecutor(max_workers=max(2, min(8, (os.cpu_count() or 4) // 2)))
            self._bounce_events = [None, None]
        pool, nthr = self._bounce_pool, self._bounce_pool._max_workers
        events = self._bounce_events          # (kept across calls: the next array reuses the buffers of this one)
        for k, lo in enumerate(range(0, flat.shape[0], chunk)):
            hi = min(lo + chunk, flat.shape[0])
            b = k & 1
            if events[b] is not None:
                events[b].synchronize()                 # the DMA that last read this buffer is done
            bounce = self._bounce[b].view(t.dtype)
            dst = bounce.numpy()
            step = -(-(hi - lo) // nthr)
            list(pool.map(lambda r: np.copyto(dst[r:min(r + step, hi - lo)], flat[lo + r:min(lo + r + step, hi)]),
                          range(0, hi - lo, step)))
            out[lo:hi].copy_(bounce[:hi - lo], non_blocking=True)
            events[b] = torch.cuda.Event()
            events[b].record(torch.cuda.current_stream(self.device))
        return out.view(*a.shape)

    def upload_clean(self, inputs, data, resolve_minmax):
        """Host numpy RAW inputs (N x M float64) and data -> DeviceDataset with the inputs min-max normalised in HBM.
        resolve_minmax(column_minmax) -> [[min, max], ...] is the host policy (user bounds, pillow, warnings);
        column_minmax() computes the data's per-column bounds on the device (reduced over all ranks)."""
        torch = self.torch
        ds = self.upload(inputs, data)
        n, m = ds.n, ds.m

        def column_minmax():
            mmx = torch.empty(2 * m, dtype=torch.float64, device=self.device)
            self._ck(self.lib.fokl_column_minmax(self.ctx, ds.x.data_ptr(), n, ds.ldx, m, mmx.data_ptr()))
            if self.dist is not None:
                lo, hi = mmx[0::2].contiguous(), mmx[1::2].contiguous()
                self.dist.all_reduce(lo, op=self.dist.ReduceOp.MIN, group=self.group)
                self.dist.all_reduce(hi, op=self.dist.ReduceOp.MAX, group=self.group)
                mmx = torch.stack([lo, hi], dim=1).reshape(-1)
            h = mmx.cpu().numpy()
            return [[h[2 * k], h[2 * k + 1]] for k in range(m)]

        bounds = resolve_minmax(column_minmax)
        flat = np.ascontiguousarray(np.asarray(bounds, dtype=np.float64).reshape(-1))
        if flat.shape[0] != 2 * m:
            raise ValueError("Input 'minmax' must correspond to input variables (i.e., columns of 'inputs').")
        self._ck(self.lib.fokl_normalize(self.ctx, ds.x.data_ptr(), n, ds.ldx, m, flat.ctypes.data))
        return ds

    def rows_compact(self, ds, keep, n_keep=None):
        """DeviceDataset of the rows of `ds` where the host bool vector `keep` (N) is True, in ascending row order --
        `inputs[keep, :]`, `data[keep]` -- formed in HBM by fokl_rows_compact; only the N mask bytes cross the bus.
        `keep` may instead be a device uint8 / bool tensor of N entries (fokl_trainlog's mask), with its count of
        nonzero entries in n_keep; then nothing crosses the bus."""
        torch = self.torch
        if isinstance(keep, torch.Tensor):
            if keep.shape != (ds.n,) or keep.dtype not in (torch.uint8, torch.bool) or keep.device != ds.x.device \
                    or not keep.is_contiguous() or n_keep is None:
                raise ValueError("a device keep mask must be a contiguous uint8 / bool tensor with one entry per row, "
                                 "beside the dataset, and come with its count")
            n_keep, mask = int(n_keep), keep
        else:
            keep = np.ascontiguousarray(keep, dtype=np.bool_)
            if keep.shape != (ds.n,):
                raise ValueError("keep must be a boolean vector with one entry per row")
            n_keep = int(np.count_nonzero(keep))
            mask = torch.from_numpy(keep.view(np.uint8)).to(self.device)
        ldx = _round_up(max(n_keep, 1), 16)
        x = torch.empty((ds.m, ldx), dtype=torch.float64, device=self.device)
        y = torch.empty((ldx,), dtype=torch.float64, device=self.device)
        n_out = ctypes.c_int64(-1)
        self._ck(self.lib.fokl_rows_compact(self.ctx, ds.x.data_ptr(), ds.y.data_ptr(), ds.n, ds.ldx, ds.m,
                                            mask.data_ptr(), x.data_ptr(), y.data_ptr(), ldx, ctypes.byref(n_out)))
        if n_out.value != n_keep:
            raise RuntimeError("fokl_rows_compact kept %d rows, expected %d" % (n_out.value, n_keep))
        return DeviceDataset(x, y, n_keep, ds.m, ldx)

    def trainlog(self, key, pos, n, l_log):
        """`generate_trainlog`'s split of n rows (l_log = max(int(n * train), 2)) drawn in HBM by fokl_trainlog from the
        legacy MT19937 state (key[624], pos): (device uint8 keep-mask of n entries, key and pos after the last word the
        host loop consumes, words consumed)."""
        key = np.ascontiguousarray(key, dtype=np.uint32)
        if key.shape != (624,):
            raise ValueError("key must hold the 624 words of an MT19937 state")
        keep = self.torch.empty(int(n), dtype=self.torch.uint8, device=self.device)
        key_out = np.empty(624, dtype=np.uint32)
        pos_out, words = ctypes.c_int(-1), ctypes.c_int64(-1)
        self._ck(self.lib.fokl_trainlog(self.ctx, key.ctypes.data, int(pos), int(n), int(l_log), keep.data_ptr(),
                                        key_out.ctypes.data, ctypes.byref(pos_out), ctypes.byref(words)))
        return keep, key_out, pos_out.value, words.value

    def begin_fit(self, ds):
        """Bind a dataset; allocate X (ones column) and the Gram state; compute the data moments."""
        torch = self.torch
        self.ds = ds
        n = ds.n
        if self.X is None or self.X.shape[1] != ds.ldx:
            # first fit with this row count: start small, grow geometrically.  Later fits of the same shape reuse the
            # design-matrix buffer at the capacity the previous fit reached (no allocator churn, no growth copies);
            # Engine.release() / close() gives it back.
            self.ld = ds.ldx
            self.Pcap = 0
            self.X = None
            self._ensure_columns(64 if n * 64 * 8 < (4 << 30) else 16)
        self.drop_prefetch()
        self.gap = self.P_base = 0
        self._ck(self.lib.fokl_fill_ones(self.ctx, self.X.data_ptr(), n))
        self.Xfull[0].copy_(ds.y)
        self.P = 0
        mom = torch.zeros(3, dtype=torch.float64, device=self.device)
        self._ck(self.lib.fokl_y_moments(self.ctx, ds.y.data_ptr(), n, mom.data_ptr()))
        self._allreduce(mom)
        momh = mom.cpu().numpy()
        self.n_global = int(round(momh[0]))
        self.sum_y = float(momh[1])
        self.yty = float(momh[2])
        self.Gcap = 0
        self._ensure_gram(64)
        # Gram entries of the ones column are the moments just reduced (G00 = n, Xty0 = sum y): no N-length pass
        self.G[0, 0] = float(self.n_global)
        self.Xty[0] = self.sum_y
        self.P = 1
        return self

    def _ensure_columns(self, need):
        """Grow the column-major design matrix to at least `need` columns (geometric growth, contents kept).  The
        free-memory query (cudaMemGetInfo costs tens of milliseconds on a busy device) is only made after an
        allocation has actually failed."""
        torch = self.torch
        if self.X is not None and need <= self.Pcap:
            return
        new_cap = max(need, int(self.Pcap * 1.5) + 8)
        col_bytes = self.ld * 8
        Xn = None
        try:
            Xn = torch.empty((new_cap + 1, self.ld), dtype=torch.float64, device=self.device)
        except torch.OutOfMemoryError:
            torch.cuda.empty_cache()
            free, _ = torch.cuda.mem_get_info(self.device)
            new_cap = min(new_cap, max(need, int(free * 0.9) // col_bytes - 1))
            try:
                Xn = torch.empty((new_cap + 1, self.ld), dtype=torch.float64, device=self.device)
            except torch.OutOfMemoryError:
                Xn = None
        if Xn is None:
            raise MemoryError("design matrix of %d columns x %d rows does not fit in device memory" % (need, self.ds.n))
        if self.X is not None and self.P > 0:
            end = self.P + self.gap + 1                          # y row + the columns built so far (incl. a block above a gap)
            Xn[:end].copy_(self.Xfull[:end])
        self.Xfull = Xn
        self.X = Xn[1:]
        self.Pcap = new_cap

    def _ensure_gram(self, need):
        torch = self.torch
        if need <= self.Gcap:
            return
        cap = max(need, self.Gcap * 2, 64)
        G = torch.zeros((cap, cap), dtype=torch.float64, device=self.device)
        Xty = torch.zeros((cap,), dtype=torch.float64, device=self.device)
        if self.G is not None and self.P > 0:
            G[:self.P, :self.P].copy_(self.G[:self.P, :self.P])
            Xty[:self.P].copy_(self.Xty[:self.P])
        self.G, self.Xty = G, Xty
        self.G2, self.G3 = torch.zeros_like(G), torch.zeros_like(G)
        self.Xty2, self.Xty3 = torch.zeros_like(Xty), torch.zeros_like(Xty)
        self.Gcap = cap

    def _append_built(self, c):
        """Columns [P, P + c) of X have just been written: update G and Xty (K2 + allreduce + scatter)."""
        torch = self.torch
        p_old = self.P
        self._ensure_gram(p_old + c)
        need = (p_old + c + 1) * c
        if self.block is None or self.block.numel() < need:
            self.block = torch.empty((int(need * 1.5) + 64,), dtype=torch.float64, device=self.device)
        t = self._tic()
        self._ck(self.lib.fokl_gram_update(self.ctx, self.X.data_ptr(), self.ld, self.ds.n, p_old, c,
                                           self.Xfull.data_ptr(), self.block.data_ptr()))
        # algorithmic flops (SURVEY 8d): cross block + upper triangle of the symmetric new block + X_new' y
        self._toc(t, 'gram', flops=2.0 * self.ds.n * (p_old * c + c * (c + 1) / 2 + c), bytes=8.0 * self.ds.n * (p_old + c + 1),
                  cols=p_old + c + 1)
        if self.dist is not None:
            t = self._tic()
            self._allreduce(self.block[:need])
            self._toc(t, 'allreduce', bytes=8.0 * need)
        self._ck(self.lib.fokl_gram_scatter(self.ctx, self.block.data_ptr(), p_old, c, self.G.data_ptr(), self.Gcap,
                                            self.Xty.data_ptr()))
        self.P = p_old + c

    # ---- build-ahead of a substage's columns ------------------------------------------------------------------------
    # The candidate stage of substage s (one cluster eigensolver, one 2000-draw chain, the kill loop) leaves the device
    # almost idle, and the columns of substage s + 1 do not depend on its outcome: only the NEW columns of s can be
    # deleted (FR:1660), so the first p_stable = p_old(s) columns are final.  prefetch_terms() therefore runs K1 and the
    # (old[0, p_stable) | new | y) x new part of K2 for s + 1 on a second context / stream while s is being decided;
    # append_terms(.., p_stable) later adds the small cross block new x (survivors of s) and scatters everything.  The
    # new block is written ABOVE the columns s may still delete (a gap in X, closed by the next compaction).  Every
    # append that names p_stable is computed by this same two-part scheme whether or not it was started ahead of time,
    # so the Gram bits -- and with them the whole fit -- do not depend on the timing.
    def _pf_ctx(self):
        torch = self.torch
        if self.ctx_pf is None:
            self.pf_stream = torch.cuda.Stream(device=self.device)
            ctx = ctypes.c_void_p()
            rc = self.lib.fokl_ctx_create(ctypes.byref(ctx), self.dev_index, ctypes.c_void_p(self.pf_stream.cuda_stream))
            if rc != 0:
                raise RuntimeError("fokl_ctx_create (build-ahead context) failed with code %d" % rc)
            self.ctx_pf = ctx
            sms = torch.cuda.get_device_properties(self.device).multi_processor_count
            # its Gram kernel leaves these SMs to the candidate stage it runs next to (one 16-CTA cluster + single CTAs)
            self.lib.fokl_ctx_set_sm_budget(ctx, max(sms - 20, sms // 2))
            self.lib.fokl_ctx_set_high_priority(self.ctx, 1)
            self._pf_tab_key = None
        key = (id(self._phis_tab), self._phis_kernel)
        if self._pf_tab_key != key:
            tab = self._phis_tab
            fn = self.lib.fokl_set_phis_cubic if self._phis_kernel == CUBIC else self.lib.fokl_set_phis_bernoulli
            rc = fn(self.ctx_pf, tab.ctypes.data, tab.shape[0], tab.shape[1])
            if rc != 0:
                raise RuntimeError("build-ahead context: basis table upload failed with code %d" % rc)
            self._pf_tab_key = key
        return self.ctx_pf

    def _ck_pf(self, rc):
        if rc != 0:
            msg = self.lib.fokl_last_error(self.ctx_pf)
            raise RuntimeError("libfokl_b200 error %d (build-ahead context): %s" % (rc, msg.decode() if msg else ''))

    def drop_prefetch(self):
        """Forget a build-ahead block (roll-back, end of the fit): wait for its kernels first -- what follows may
        overwrite the columns they read or write."""
        if self.pf is not None:
            self.pf_stream.synchronize()
            self.pf = None

    def phys_cols(self, cols):
        cols = np.asarray(cols, dtype=np.int32)
        if self.gap == 0:
            return np.ascontiguousarray(cols)
        return np.ascontiguousarray(np.where(cols >= self.P_base, cols + self.gap, cols).astype(np.int32))

    def prefetch_terms(self, terms, p_stable, after=None, wait_eig=False):
        """Start K1 + the first part of K2 for `terms` on the build-ahead stream.  p_stable: the leading columns of the
        model that no pending decision can delete.  after: an event on the main stream the build must wait for (default:
        everything enqueued so far).  wait_eig: also wait for the eigensolver launches of the candidate batches enqueued
        last on the main and the side context -- their clusters need whole groups of free SMs, which the Gram kernel's
        long-lived thread blocks would deny them."""
        torch = self.torch
        terms = np.ascontiguousarray(terms, dtype=np.int16)
        c, m = terms.shape
        if m != self.ds.m:
            raise ValueError("term width does not match the number of inputs")
        if c == 0 or p_stable < 1 or p_stable > (self.P_base if self.gap else self.P):
            return None
        self.drop_prefetch()
        ctx = self._pf_ctx()
        # position: below the current block if the gap has room above the columns that may survive, else above it
        lo = self.P
        if self.gap > 0 and lo + c <= self.P_base + self.gap:
            b0 = lo
        else:
            b0 = self.P + self.gap
        cap0 = self.Pcap
        try:
            self._ensure_columns(b0 + c)
        except MemoryError:
            return None
        n = self.ds.n
        block_a = torch.empty(((p_stable + c + 1) * c,), dtype=torch.float64, device=self.device)
        if after is None or self.Pcap != cap0:       # a re-allocation copied X on the main stream just now
            after = self.mark()
        self.pf_stream.wait_event(after)
        if wait_eig:
            self._ck_pf(self.lib.fokl_ctx_wait_eig(ctx, self.ctx))
            if self.ctx_side is not None:
                self._ck_pf(self.lib.fokl_ctx_wait_eig(ctx, self.ctx_side))
        with torch.cuda.stream(self.pf_stream):
            t = self._tic()
            self._ck_pf(self.lib.fokl_basis_build(ctx, self.kernel_id, self.ds.x.data_ptr(), n, self.ds.ldx, m,
                                                 terms.ctypes.data, c, self.X[b0].data_ptr(), self.ld))
            self._toc(t, 'basis', bytes=8.0 * n * (m + c), cells=float(n) * c)
            t = self._tic()
            self._ck_pf(self.lib.fokl_gram_update_ex(ctx, self.X.data_ptr(), self.ld, n, p_stable, c, b0, 0,
                                                    self.Xfull.data_ptr(), block_a.data_ptr()))
            self._toc(t, 'gram', flops=2.0 * n * (p_stable * c + c * (c + 1) / 2 + c), bytes=8.0 * n * (p_stable + c + 1),
                      cols=p_stable + c + 1)
            done = torch.cuda.Event()
            done.record(self.pf_stream)
        self.pf = dict(terms=terms, p_stable=int(p_stable), b0=int(b0), c=int(c), block=block_a, done=done)
        return self.pf

    def _close_gap(self):
        """Move the block above the gap down so that the model is one contiguous run of columns again."""
        if self.gap == 0:
            return
        keep = self.phys_cols(np.arange(self.P, dtype=np.int32))
        t = self._tic()
        self._ck(self.lib.fokl_columns_compact(self.ctx, self.X.data_ptr(), self.ld, self.ds.n, keep.ctypes.data, self.P))
        self._toc(t, 'compact')
        self.gap = 0
        self.P_base = self.P

    def _append_split(self, terms, p_stable):
        """append_terms through the two-part scheme (see above): commit the matching build-ahead block, or build it now."""
        torch = self.torch
        c = terms.shape[0]
        pf = self.pf
        if pf is None or pf['p_stable'] != p_stable or pf['c'] != c or not np.array_equal(pf['terms'], terms):
            self.drop_prefetch()
            self._close_gap()
            pf = self.prefetch_terms(terms, p_stable)
            if pf is None:
                raise MemoryError("design matrix does not fit in device memory")
        self.pf = None
        main = torch.cuda.current_stream(self.device)
        main.wait_event(pf['done'])
        self._close_gap()                      # the previous substage kept all its columns: no compaction closed the gap
        p_old, n, b0 = self.P, self.ds.n, pf['b0']
        k = p_old - p_stable
        self._ensure_gram(p_old + c)
        need = (p_old + c + 1) * c
        if self.block is None or self.block.numel() < need:
            self.block = torch.empty((int(need * 1.5) + 64,), dtype=torch.float64, device=self.device)
        blk = self.block[:need].view(p_old + c + 1, c)
        a = pf['block'].view(p_stable + c + 1, c)
        blk[:p_stable].copy_(a[:p_stable])
        blk[p_old:].copy_(a[p_stable:])
        if k > 0:
            # cross block: new columns x the columns that survived the previous substage (X base shifted to p_stable)
            bb = torch.empty(((k + c + 1) * c,), dtype=torch.float64, device=self.device)
            t = self._tic()
            self._ck(self.lib.fokl_gram_update_ex(self.ctx, self.X[p_stable].data_ptr(), self.ld, n, k, c, b0 - p_stable,
                                                  _lib.GRAM_CROSS_ONLY, self.Xfull.data_ptr(), bb.data_ptr()))
            self._toc(t, 'gram', flops=2.0 * n * k * c, bytes=8.0 * n * (k + c), cols=k + c)
            blk[p_stable:p_old].copy_(bb.view(k + c + 1, c)[:k])
        a.record_stream(main)
        if self.dist is not None:
            t = self._tic()
            self._allreduce(self.block[:need])
            self._toc(t, 'allreduce', bytes=8.0 * need)
        self._ck(self.lib.fokl_gram_scatter(self.ctx, self.block.data_ptr(), p_old, c, self.G.data_ptr(), self.Gcap,
                                            self.Xty.data_ptr()))
        self.P_base, self.gap = p_old, b0 - p_old
        self.P = p_old + c

    def append_terms(self, terms, p_stable=None):
        """K1 + K2 for `terms` (C x M integer orders): appends C columns to X, extends G / Xty.  p_stable (optional):
        number of leading columns that were already final when the previous substage began -- selects the two-part
        scheme that prefetch_terms() can start ahead of time."""
        terms = np.ascontiguousarray(terms, dtype=np.int16)
        c, m = terms.shape
        if m != self.ds.m:
            raise ValueError("term width does not match the number of inputs")
        if c == 0:
            return
        if p_stable is not None and 1 <= p_stable <= self.P:
            self._append_split(terms, int(p_stable))
            return
        self.drop_prefetch()
        self._close_gap()
        self._ensure_columns(self.P + c)
        t = self._tic()
        self._ck(self.lib.fokl_basis_build(self.ctx, self.kernel_id, self.ds.x.data_ptr(), self.ds.n, self.ds.ldx, m,
                                           terms.ctypes.data, c, self.X[self.P].data_ptr(), self.ld))
        self._toc(t, 'basis', bytes=8.0 * self.ds.n * (m + c), cells=float(self.ds.n) * c)
        self._append_built(c)

    def compact(self, keep):
        """Keep only columns `keep` (ascending, includes 0) of X / G / Xty: the X <- xers step (FR:1695)."""
        keep = np.ascontiguousarray(keep, dtype=np.int32)
        p_new = len(keep)
        if p_new == self.P:
            return
        src = self.phys_cols(keep)              # where the kept columns live (a block may sit above a gap)
        t = self._tic()
        self._ck(self.lib.fokl_columns_compact(self.ctx, self.X.data_ptr(), self.ld, self.ds.n, src.ctypes.data, p_new))
        self._toc(t, 'compact')
        self.gap = 0
        self.P_base = p_new
        self._ck(self.lib.fokl_gram_compact(self.ctx, self.G.data_ptr(), self.Gcap, self.Xty.data_ptr(),
                                            keep.ctypes.data, p_new, self.G2.data_ptr(), self.Gcap, self.Xty2.data_ptr()))
        # three buffers in rotation: the Gram a compaction starts from stays intact across the NEXT compaction as well,
        # so the chains that verify substage s - 1 on the side stream (they index the Gram as it was before the
        # compaction of s - 1) may still be running when the compaction of s is enqueued
        self.G, self.G2, self.G3 = self.G2, self.G3, self.G
        self.Xty, self.Xty2, self.Xty3 = self.Xty2, self.Xty3, self.Xty
        self.P = p_new

    # ------------------------------------------------------------------------------------------------
    def make_hypers(self, a, b, atau, btau, sigsqd0, tausqd0, draws):
        h = _lib.Hypers()
        h.a, h.b, h.atau, h.btau = float(a), float(b), float(atau), float(btau)
        h.sigsqd0, h.tausqd0 = float(sigsqd0), float(tausqd0)
        h.yty, h.sum_y = self.yty, self.sum_y
        h.n = self.n_global
        h.draws = int(draws)
        h.stat_from0 = int(math.ceil(draws / 2))
        h.stat_from1 = int(math.ceil(draws / 2 + 1))
        h.reserved = 0
        return h

    def evaluate(self, col_sets, hyp, rng_mode=_lib.RNG_NONE, run_chain=None, seed=0, stream_ids=None,
                 variates=None, sign_fix=None, want_betas=False, want_eig=False, refine_tol=1e-7):
        """K3/K4 on a batch of candidate models (lists of column indices into the current X / G).

        Returns a CandidateResult; `ev` is a host numpy array (this call synchronises)."""
        return self.evaluate_launch(col_sets, hyp, rng_mode=rng_mode, run_chain=run_chain, seed=seed,
                                    stream_ids=stream_ids, variates=variates, sign_fix=sign_fix, want_betas=want_betas,
                                    want_eig=want_eig).finish(refine_tol)

    def _side(self):
        """Second context on a private (non-blocking) stream: a batch launched there runs next to the work of the main
        context (used for the chains that verify a substage while the next substage's full model is evaluated)."""
        if getattr(self, 'ctx_side', None) is None:
            self.side_stream = self.torch.cuda.Stream(device=self.device)
            ctx = ctypes.c_void_p()
            rc = self.lib.fokl_ctx_create(ctypes.byref(ctx), self.dev_index, ctypes.c_void_p(self.side_stream.cuda_stream))
            if rc != 0:
                raise RuntimeError("fokl_ctx_create (side context) failed with code %d" % rc)
            self.ctx_side = ctx
            # its batches run next to the main context's full-model evaluation (one cluster of up to 16 CTAs)
            sms = self.torch.cuda.get_device_properties(self.device).multi_processor_count
            self.lib.fokl_ctx_set_sm_budget(ctx, max(sms - int(os.environ.get('FOKL_B200_SIDE_RESERVE', '16')), 16))
            # ... and the main context's candidate stage (the full model: one cluster, latency-bound, on the critical path)
            # goes to a high-priority stream so that its CTAs are placed ahead of the batch's: cfg4 full models
            # 34.0 -> 30.6 ms per fit next to the side batches (gpurun_out/r4l, profiles/r02_bench_lines.txt)
            if os.environ.get('FOKL_B200_MAIN_HP', '1') not in ('0', ''):
                self.lib.fokl_ctx_set_high_priority(self.ctx, 1)
        return self.ctx_side

    def gram_state(self):
        """(G, Xty, ldg) of the current model as tensor references: stays valid (for reading) across the next
        append_terms calls and TWO compactions, which write to other buffers or to rows / columns beyond the current P."""
        return (self.G, self.Xty, self.Gcap)

    def truncate(self, p):
        """Forget the columns from p on (roll-back of a speculative append_terms)."""
        self.drop_prefetch()
        p = int(p)
        if self.gap > 0 and p > self.P_base:
            self._close_gap()
        elif self.gap > 0:
            self.gap = 0
        self.P = p
        self.P_base = min(self.P_base, p)

    def mark(self):
        """An event on the main stream: evaluate_launch(side=True, after=mark) then orders the side batch after the work
        enqueued up to here only, not after what the main stream is given later."""
        e = self.torch.cuda.Event()
        e.record(self.torch.cuda.current_stream(self.device))
        return e

    def evaluate_launch(self, col_sets, hyp, rng_mode=_lib.RNG_NONE, run_chain=None, seed=0, stream_ids=None,
                        variates=None, sign_fix=None, want_betas=False, want_eig=False, gram=None, side=False,
                        after=None):
        """Enqueue K3/K4 for a batch of candidate models and return a PendingCandidates; nothing is read back until
        its finish().  gram: (G, Xty, ldg) to index instead of the current Gram (gram_state() of an earlier model);
        side: enqueue on the side context's stream, concurrently with the main stream's work."""
        torch = self.torch
        G, Xty, ldg = gram if gram is not None else (self.G, self.Xty, self.Gcap)
        main_stream = torch.cuda.current_stream(self.device)
        if side:
            self._side()
            # Order the side stream after the main stream's work up to `after` (or up to now), then make every
            # allocation / zero-fill / upload of this batch on the side stream itself: a fill enqueued on the main stream
            # behind later main-stream work could otherwise land after the batch's kernels have written their results.
            if after is not None:
                self.side_stream.wait_event(after)
            else:
                self.side_stream.wait_stream(main_stream)
        with (torch.cuda.stream(self.side_stream) if side else contextlib.nullcontext()):
            n_cand = len(col_sets)
            p = np.array([len(s) for s in col_sets], dtype=np.int64)
            offs = np.zeros(n_cand + 1, dtype=np.int32)
            offs[1:] = np.cumsum(p)
            flat = np.ascontiguousarray(np.concatenate([np.asarray(s, dtype=np.int32) for s in col_sets]))
            vec_off = np.concatenate([[0], np.cumsum(p)[:-1]]).astype(np.int64)
            mat_off = np.concatenate([[0], np.cumsum(p * p)[:-1]]).astype(np.int64)
            total_p = int(p.sum())
            D = int(hyp.draws)
            f64 = dict(dtype=torch.float64, device=self.device)
            chain_any = rng_mode != _lib.RNG_NONE and (run_chain is None or bool(np.any(run_chain)))
            # ev | info | stats share one buffer: one read-back in finish() instead of three
            n_i = (n_cand + 1) // 2
            pack = torch.zeros(n_cand + n_i + (3 * total_p if chain_any else 0), **f64)
            ev = pack[:n_cand]
            info = pack[n_cand:n_cand + n_i].view(torch.int32)[:n_cand]
            betahat = torch.empty(total_p, **f64)
            stats = pack[n_cand + n_i:] if chain_any else None
            betas = torch.empty(D * total_p, **f64) if (chain_any and want_betas) else None
            sigs = torch.empty(D * n_cand, **f64) if (chain_any and want_betas) else None
            taus = torch.empty(D * n_cand, **f64) if (chain_any and want_betas) else None
            lamb = torch.empty(total_p, **f64) if want_eig else None
            Q = torch.empty(int((p * p).sum()), **f64) if want_eig else None
            rc_arr = None
            if run_chain is not None:
                rc_arr = np.ascontiguousarray(run_chain, dtype=np.uint8)
            sid = None
            if stream_ids is not None:
                sid = np.ascontiguousarray(stream_ids, dtype=np.uint64)
            var_t = None
            if rng_mode == _lib.RNG_INJECTED:
                var_t = variates if torch.is_tensor(variates) else torch.from_numpy(
                    np.ascontiguousarray(variates, dtype=np.float64)).to(self.device)
            sf_t = None
            if sign_fix is not None:
                sf_t = sign_fix if torch.is_tensor(sign_fix) else torch.from_numpy(
                    np.ascontiguousarray(sign_fix, dtype=np.float64)).to(self.device)

        def ptr(t):
            return None if t is None else t.data_ptr()

        ctx = self.ctx
        t = None
        if side:
            ctx = self._side()
            with torch.cuda.stream(self.side_stream):
                t = self._tic()
        else:
            t = self._tic()
        rc = self.lib.fokl_candidates_eval(
            ctx, G.data_ptr(), ldg, Xty.data_ptr(), flat.ctypes.data, offs.ctypes.data, n_cand,
            ctypes.byref(hyp), None if rc_arr is None else rc_arr.ctypes.data, rng_mode, ctypes.c_uint64(int(seed)),
            None if sid is None else sid.ctypes.data, ptr(var_t), ptr(sf_t), ptr(ev), ptr(betahat), ptr(lamb), ptr(Q),
            ptr(betas), ptr(sigs), ptr(taus), ptr(stats), ptr(info))
        if rc != 0:
            msg = self.lib.fokl_last_error(ctx)
            raise RuntimeError("libfokl_b200 error %d: %s" % (rc, msg.decode() if msg else ''))
        if side:
            with torch.cuda.stream(self.side_stream):
                self._toc(t, 'side_batch', cands=n_cand, pmax=int(p.max()), psum=int(p.sum()))
        else:
            self._toc(t, 'candidates_chain' if chain_any else 'candidates_bic', cands=n_cand, pmax=int(p.max()))
        self.gibbs_launch_batches += 1
        self.work['eig_solves'] += n_cand
        if chain_any:
            self.work['chains_run'] += int(n_cand if rc_arr is None else np.count_nonzero(rc_arr))
        res = CandidateResult()
        res.p, res.vec_off, res.mat_off, res.draws = p, vec_off, mat_off, D
        res.stats, res.betas, res.sigs, res.taus = stats, betas, sigs, taus
        res.betahat, res.lamb, res.Q = betahat, lamb, Q
        pend = PendingCandidates(self, res, ev, info, col_sets, side, (G, Xty, var_t, sf_t))
        pend.pack = pack
        return pend

    # ---- chains of nested models (csrc/nested.cu) ---------------------------------------------------------------------
    def nested_chains_launch(self, col_sets, hyp, seed, stream_ids, gram=None, side=False, after=None, head=None):
        """Intercept statistics of the chains of NESTED models: col_sets[i + 1] is col_sets[i] minus one or more columns
        (col_sets[i][0] = the intercept column).  One eigensolver run (the first model), then one secular-equation step +
        one GEMM per removed column, then all chains in one launch.  Returns a handle; finish() -> dict(mean0 = per model
        the mean of the intercept's draws over rows stat_from0 .., ok = False if a step met equal eigenvalues or a chain
        saw bstar < 0 -- evaluate the models with evaluate_launch then).
        head (optional): (columns, lamb, Q) of a super-model of col_sets[0] that is already decomposed on the same Gram
        (the substage's full model): the run starts from it instead of a cold solve of col_sets[0]."""
        torch = self.torch
        G, Xty, ldg = gram if gram is not None else (self.G, self.Xty, self.Gcap)
        pend = None
        if head is not None:
            head_cols, lam0, Q0 = head
            head_cols = np.ascontiguousarray(head_cols, dtype=np.int32)
            if side:
                self._side()
                if after is not None:
                    self.side_stream.wait_event(after)
                else:
                    self.side_stream.wait_stream(torch.cuda.current_stream(self.device))
        else:
            head_cols = np.ascontiguousarray(col_sets[0], dtype=np.int32)
            pend = self.evaluate_launch([head_cols], hyp, rng_mode=_lib.RNG_NONE, want_eig=True, gram=(G, Xty, ldg),
                                        side=side, after=after)
            lam0, Q0 = pend.res.lamb, pend.res.Q
        head = head_cols
        p0 = len(head)
        ctx = self._side() if side else self.ctx
        n_models = len(col_sets)
        widths = np.array([len(c) for c in col_sets], dtype=np.int32)
        offs = np.zeros(n_models, dtype=np.int64)
        offs[1:] = np.cumsum(widths.astype(np.int64))[:-1]
        total = int(widths.sum())
        pos_of = {int(c): e for e, c in enumerate(head)}
        with (torch.cuda.stream(self.side_stream) if side else contextlib.nullcontext()):
            f64 = dict(dtype=torch.float64, device=self.device)
            lam_all, ct_all, q0_all = torch.empty(total, **f64), torch.empty(total, **f64), torch.empty(total, **f64)
            status = torch.zeros(1, dtype=torch.int32, device=self.device)
            xty = Xty.index_select(0, torch.as_tensor(head.astype(np.int64), device=self.device)).clone()
            lam = lam0[:p0]
            Qs = Q0[:p0 * p0].view(p0, p0)            # rows = eigenvectors, columns = the head model's columns
            work = torch.empty(4 * p0 + 8, **f64)
            t = self._tic()
            # the deletions of the whole run are known: only the intercept's column of Q, the columns of the variables
            # still to be removed (their rows give u) and the vector Q'X'y have to be carried from model to model
            dels, prev = [], set(int(c) for c in head)
            for i, cols in enumerate(col_sets):
                if i > 0 or pend is None:
                    cur = set(int(c) for c in cols)
                    if not cur <= prev:
                        raise ValueError("nested_chains_launch: model %d is not a subset of its predecessor" % i)
                    dels.append([pos_of[c] for c in sorted(prev - cur)])
                    prev = cur
                else:
                    dels.append([])
            order = [m for d in dels for m in d]
            need = torch.as_tensor(np.asarray([pos_of[int(head[0])]] + order, dtype=np.int64), device=self.device)
            R = Qs.index_select(1, need).contiguous()            # p x (1 + remaining deletions)
            ct = torch.mv(Qs, xty)
            steps = used = 0
            col_of = {m: 1 + j for j, m in enumerate(order)}     # column of R holding variable m
            for i in range(n_models):
                for m in dels[i]:
                    p = lam.numel()
                    u = R[:, col_of[m]].contiguous()
                    mu = torch.empty(p - 1, **f64)
                    zt = torch.empty((p - 1, p), **f64)
                    rc = self.lib.fokl_secular_step(ctx, lam.data_ptr(), u.data_ptr(), p, mu.data_ptr(), zt.data_ptr(), p,
                                                    work.data_ptr(), status.data_ptr())
                    if rc != 0:
                        msg = self.lib.fokl_last_error(ctx)
                        raise RuntimeError("libfokl_b200 error %d: %s" % (rc, msg.decode() if msg else ''))
                    # Q_new = Z' Q on the carried columns (plain FP64 GEMM, cuBLAS) and Q_new' X'y = Z' (Q'X'y - (X'y)_m u):
                    # the new eigenvectors have no component on the removed variable
                    ct = torch.mv(zt, ct - xty[m] * u)
                    R = torch.matmul(zt, R)
                    lam = mu
                    steps += 1
                    used += 1
                    if used >= 64 and used * 4 >= R.shape[1]:
                        # drop the columns of the variables already removed: the GEMM shrinks with the work left
                        keep = [0] + [col_of[mm] for mm in order[steps:]]
                        R = R.index_select(1, torch.as_tensor(np.asarray(keep, dtype=np.int64), device=self.device))
                        col_of = {mm: 1 + j for j, mm in enumerate(order[steps:])}
                        used = 0
                o, w = int(offs[i]), int(widths[i])
                lam_all[o:o + w].copy_(lam)
                ct_all[o:o + w].copy_(ct)
                q0_all[o:o + w].copy_(R[:, 0])
            p_dev = torch.from_numpy(widths).to(self.device)
            off_dev = torch.from_numpy(offs).to(self.device)
            sid_dev = torch.from_numpy(np.ascontiguousarray(stream_ids, dtype=np.uint64).view(np.int64)).to(self.device)
            mean0 = torch.empty(n_models, **f64)
            info = torch.zeros(n_models, dtype=torch.int32, device=self.device)
            rc = self.lib.fokl_chain_icpt(ctx, n_models, p_dev.data_ptr(), off_dev.data_ptr(), sid_dev.data_ptr(),
                                          lam_all.data_ptr(), ct_all.data_ptr(), q0_all.data_ptr(), ctypes.byref(hyp),
                                          ctypes.c_uint64(int(seed)), mean0.data_ptr(), info.data_ptr())
            if rc != 0:
                msg = self.lib.fokl_last_error(ctx)
                raise RuntimeError("libfokl_b200 error %d: %s" % (rc, msg.decode() if msg else ''))
            self._toc(t, 'nested_chains', cands=n_models, steps=steps, pmax=int(p0))
        self.work['eig_solves'] += 0            # (the head's solve was counted by evaluate_launch)
        self.work['chains_run'] += n_models
        self.work['secular_steps'] = self.work.get('secular_steps', 0) + steps
        eng = self
        keep = (lam_all, ct_all, q0_all, p_dev, off_dev, sid_dev, xty, work, pend)

        class _Pending:
            def finish(_self):
                with (torch.cuda.stream(eng.side_stream) if side else contextlib.nullcontext()):
                    st = int(status.cpu().item())
                    m0 = mean0.cpu().numpy()
                    inf = info.cpu().numpy()
                if side:
                    main_stream = torch.cuda.current_stream(eng.device)
                    main_stream.wait_stream(eng.side_stream)
                    for tns in keep[:8] + (mean0, info, status):
                        tns.record_stream(main_stream)
                ok = st == 0 and not inf.any() and bool(np.all(np.isfinite(m0)))
                return dict(mean0=m0, ok=ok, status=st)
        return _Pending()

    def refine_mask(self, ev, p, refine_tol=1e-7):
        """Candidates whose Gram-only BIC is not trustworthy (non-finite, or a residual variance below refine_tol of
        var(y): catastrophic cancellation) and must be recomputed from an N-length residual pass."""
        n = float(self.n_global)
        var_y = self.yty / n - (self.sum_y / n) ** 2
        with np.errstate(all='ignore'):
            siglik = np.exp((ev - p * np.log(n) - (n - 1.0)) / n)
        return ~np.isfinite(ev) | ~(siglik > refine_tol * var_y)

    def kill_scores(self, cols, positions, hyp):
        """BIC of the model `cols` minus each column at `positions` (indices into cols), plus the model's own BIC,
        from one Cholesky factorisation on the device.  Returns (ev numpy [k + 1], ok)."""
        torch = self.torch
        cols = np.ascontiguousarray(cols, dtype=np.int32)
        positions = np.ascontiguousarray(positions, dtype=np.int32)
        k = len(positions)
        ev = torch.empty(k + 1, dtype=torch.float64, device=self.device)
        info = torch.zeros(1, dtype=torch.int32, device=self.device)
        t = self._tic()
        self._ck(self.lib.fokl_kill_scores(self.ctx, self.G.data_ptr(), self.Gcap, self.Xty.data_ptr(), cols.ctypes.data,
                                           len(cols), positions.ctypes.data if k else None, k, ctypes.byref(hyp),
                                           ev.data_ptr(), info.data_ptr()))
        self._toc(t, 'kill_scores', cands=k, pmax=len(cols))
        evh = ev.cpu().numpy()
        ok = int(info.item()) == 0 and bool(np.all(np.isfinite(evh)))
        return evh, ok

    def kill_loop(self, cols, cand_pos, bv0, bv1, hyp, threshav, threshstda, threshstdb, icpt, evmin, aic_adj, start):
        """The kill loop of one substage (FR:1666-1690) in one launch (fokl_kill_loop).  Returns dict(n_acc, tested,
        bad, acc, calls, ev) as host values (this call synchronises)."""
        return self.kill_loop_launch(cols, cand_pos, bv0, bv1, hyp, threshav, threshstda, threshstdb, icpt, evmin,
                                     aic_adj, start).finish()

    def kill_loop_launch(self, cols, cand_pos, bv0, bv1, hyp, threshav, threshstda, threshstdb, icpt, evmin, aic_adj,
                         start, eig=None):
        """Enqueue fokl_kill_loop; the returned handle's finish() reads the result back (host work can go in between).
        eig (optional): (lamb, Q) device tensors of the eigendecomposition of G[cols][cols] as evaluate_launch(...,
        want_eig=True) returns them for exactly this column list -- the loop's tableau is then formed from it by the
        whole device instead of by len(cols) sequential pivots."""
        torch = self.torch
        cols = np.ascontiguousarray(cols, dtype=np.int32)
        cand_pos = np.ascontiguousarray(cand_pos, dtype=np.int32)
        bv0 = np.ascontiguousarray(bv0, dtype=np.float64)
        bv1 = np.ascontiguousarray(bv1, dtype=np.float64)
        vm = len(cand_pos)
        kp = _lib.KillParams(float(threshav), float(threshstda), float(threshstdb), float(icpt), float(evmin),
                             float(aic_adj), int(start), 0, None if eig is None else eig[0].data_ptr(),
                             None if eig is None else eig[1].data_ptr())
        # one output buffer: [3 + 2 vm] int32 viewed in the first doubles, then vm doubles
        n_i = 3 + 2 * vm
        n_i_d = (n_i + 1) // 2
        out = torch.zeros(n_i_d + max(vm, 1), dtype=torch.float64, device=self.device)
        t = self._tic()
        self._ck(self.lib.fokl_kill_loop(self.ctx, self.G.data_ptr(), self.Gcap, self.Xty.data_ptr(), cols.ctypes.data,
                                         len(cols), cand_pos.ctypes.data, bv0.ctypes.data, bv1.ctypes.data, vm,
                                         ctypes.byref(hyp), ctypes.byref(kp), out.data_ptr(),
                                         out.data_ptr() + 8 * n_i_d))
        self._toc(t, 'kill_loop', cands=vm, pmax=len(cols))

        class _Pending:
            def finish(_self):
                h = out.cpu().numpy()
                oi = h[:n_i_d].view(np.int32)
                k = int(oi[0])
                self.work['kill_loops'] += 1
                self.work['kill_proposals_scored'] += int(oi[1])
                return dict(n_acc=k, tested=int(oi[1]), bad=int(oi[2]), acc=oi[3:3 + k].copy(),
                            calls=oi[3 + vm:3 + vm + k].copy(), ev=h[n_i_d:n_i_d + k].copy())
        return _Pending()

    # ---- update fits (FoKL/_update.py, csrc/update.cu) ---------------------------------------------------------------
    def sym_eigh(self, A):
        """(lam ascending, Q with eigenvectors as columns) of a symmetric positive definite p x p device matrix, by the
        library's own eigensolver (fokl_candidates_eval without a chain, the matrix passed in place of the Gram)."""
        torch = self.torch
        A = A.contiguous()
        p = int(A.shape[0])
        hyp = self.make_hypers(1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1)
        dummy = torch.zeros(p, dtype=torch.float64, device=self.device)
        res = self.evaluate_launch([list(range(p))], hyp, want_eig=True, gram=(A, dummy, p)).finish(None)
        return res.lamb[:p].clone(), res.Q[:p * p].view(p, p).t().contiguous()

    def residual_sse(self, p, betahat_dev):
        """|y - X[:, :p] betahat|^2 over all rows of all ranks (FR:2083), by an N-length pass."""
        torch = self.torch
        cols = self.phys_cols(list(range(int(p))))
        out = torch.zeros(2, dtype=torch.float64, device=self.device)
        bh = betahat_dev.contiguous()
        self._ck(self.lib.fokl_residual_moments(self.ctx, self.X.data_ptr(), self.ld, self.ds.n, len(cols),
                                                cols.ctypes.data, bh.data_ptr(), self.ds.y.data_ptr(), out.data_ptr()))
        self._allreduce(out)
        return float(out[1].item())

    def update_chain(self, spec, arrays, rng_mode, seed=0, stream_id=0, variates=None):
        from ._update import engine_update_chain
        return engine_update_chain(self, spec, arrays, rng_mode, seed=seed, stream_id=stream_id, variates=variates)

    def residual_bic(self, cols, betahat_dev):
        """BIC of FR:1551-1554 from an explicit N-length residual pass over X (used when the Gram-only
        formula has lost too many digits to cancellation)."""
        torch = self.torch
        cols = self.phys_cols(cols)
        out = torch.zeros(2, dtype=torch.float64, device=self.device)
        self._ck(self.lib.fokl_residual_moments(self.ctx, self.X.data_ptr(), self.ld, self.ds.n, len(cols),
                                                cols.ctypes.data, betahat_dev.data_ptr(), self.ds.y.data_ptr(),
                                                out.data_ptr()))
        self._allreduce(out)
        sr, srr = out.cpu().numpy()
        n = float(self.n_global)
        siglik = srr / n - (sr / n) ** 2
        with np.errstate(all='ignore'):
            lik = -(n / 2) * np.log(siglik) - (n - 1) / 2
        return len(cols) * np.log(n) - 2 * lik
