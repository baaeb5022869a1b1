"""A host stand-in engine for the device form of `clean` (FoKL._clean_on_device, FoKL._evaluate_clean).  TEST
INFRASTRUCTURE: the product's own Engine.upload / upload_clean / rows_compact run unchanged on CPU tensors, and `lib`
holds Python functions with the C ABI's argument lists (include/fokl_b200.h) for fokl_column_minmax, fokl_normalize
and fokl_rows_compact (each computing what the header defines, with the kernels' IEEE operations), next to
tests/fake_device.py's basis / product stand-ins and test_predict_summary's fokl_predict_summary.  The fit itself runs
on the selection-loop stand-in (tests/mock_engine.py) over the dataset the device path left in the tensors."""
import types

import numpy as np
import torch

from fake_device import FakeDeviceEngine, _view
from FoKL._engine import Engine
from mock_engine import MockEngine
from test_public_api_stand_in import StandInEngine
from test_predict_summary import _product, summary


class CleanStandIn(StandInEngine):
    upload = Engine.upload
    _h2d = Engine._h2d
    upload_clean = Engine.upload_clean
    rows_compact = Engine.rows_compact
    _ck = Engine._ck

    def __init__(self, dist=None):
        super().__init__()
        self.torch, self.device, self.ctx = torch, torch.device('cpu'), None
        self.dist, self.group, self.world, self.rank = None, None, 1, 0
        if dist is not None and dist.get_world_size() > 1:
            self.dist, self.world, self.rank = dist, dist.get_world_size(), dist.get_rank()
        self._dist_arg = dist
        self.log = []
        fake = FakeDeviceEngine()
        self._fake = fake
        self.lib = types.SimpleNamespace(
            fokl_column_minmax=self._column_minmax, fokl_normalize=self._normalize, fokl_rows_compact=self._rows_compact,
            fokl_fill_ones=fake._fill_ones, fokl_basis_build=fake._basis_build, fokl_predict_draws=self._predict_draws,
            fokl_predict_summary=self._predict_summary, fokl_last_error=lambda ctx: b'bad argument')

    def set_phis(self, phis, kernel):
        StandInEngine.set_phis(self, phis, kernel)
        self._fake.set_phis(phis, kernel)
        self.kernel_id = self._fake.kernel_id

    def begin_fit(self, ds):
        MockEngine.__init__(self, ds.x[:, :ds.n].t().numpy().copy(), ds.y[:ds.n].numpy().copy(), self._phis_arg,
                            self._kernel_arg, dist=self._dist_arg)

    # ---- C ABI on host addresses -----------------------------------------------------------------------------------
    def _column_minmax(self, ctx, x, n, ldx, m, out):
        self.log.append(('column_minmax', n, m))
        if not x or not out or n < 1 or m < 1 or ldx < n:
            return -1
        xv = _view(x, (m, ldx), np.float64)[:, :n]
        o = _view(out, (2 * m,), np.float64)
        o[0::2], o[1::2] = xv.min(axis=1), xv.max(axis=1)
        return 0

    def _normalize(self, ctx, x, n, ldx, m, minmax):
        self.log.append(('normalize', n, m))
        if not x or not minmax or n < 1 or m < 1 or ldx < n:
            return -1
        xv = _view(x, (m, ldx), np.float64)
        mm = _view(minmax, (2 * m,), np.float64)
        for k in range(m):
            xv[k, :n] = (xv[k, :n] - mm[2 * k]) / (mm[2 * k + 1] - mm[2 * k])
        return 0

    def _rows_compact(self, ctx, x, y, n, ldx, m, keep, x_out, y_out, ldx_out, n_out):
        self.log.append(('rows_compact', n, m))
        if not (x and y and keep and x_out and y_out and n_out) or n < 1 or m < 1 or ldx < n:
            return -1
        k = _view(keep, (n,), np.uint8) != 0
        kept = int(k.sum())
        if ldx_out < kept:
            return -1
        xo = _view(x_out, (m, ldx_out), np.float64)
        yo = _view(y_out, (ldx_out,), np.float64)
        xo[:, :kept] = _view(x, (m, ldx), np.float64)[:, :n][:, k]
        yo[:kept] = _view(y, (n,), np.float64)[k]
        xo[:, kept:] = 0.0
        yo[kept:] = 0.0
        n_out._obj.value = kept
        return 0

    def _predict_draws(self, ctx, X, ld, n, p, betas, draws, out):
        self.log.append(('predict_draws', n))
        _view(out, (n, draws), np.float64)[:] = _product(_view(X, (p, ld), np.float64)[:, :n],
                                                         _view(betas, (draws, p), np.float64))
        return 0

    def _predict_summary(self, ctx, X, ld, n, p, betas, draws, rank_lo, rank_hi, mean, lo, hi):
        self.log.append(('predict_summary', n))
        v = _product(_view(X, (p, ld), np.float64)[:, :n], _view(betas, (draws, p), np.float64))
        m, l, h = summary(v, rank_lo, rank_hi)
        _view(mean, (n,), np.float64)[:] = m
        if rank_lo >= 0:
            _view(lo, (n,), np.float64)[:] = l
            _view(hi, (n,), np.float64)[:] = h
        return 0
