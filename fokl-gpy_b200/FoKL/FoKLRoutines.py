"""FoKLRoutines -- drop-in `FoKL` class whose `fit` runs on hand-written sm_100a CUDA kernels.

API mirror of the reference's src/FoKL/FoKLRoutines.py ("FR"): same class / module names (pickles record
`FoKL.FoKLRoutines.FoKL`, FR:1840-1842), same constructor hyper-parameters and defaults (FR:205-216), same
`fit` / `clean` / `evaluate` / `coverage3` / `save` / `load` / `clear` signatures, return types and
side effects (attributes, `[ind, ev]` console line FR:1700).  The numerics of the training hot path live
in libfokl_b200.so (see ._engine, include/fokl_b200.h); there is no CPU fallback -- without a CUDA
device or the built library `fit` raises.

Differences that are deliberate and documented (DESIGN.md):
  * the Gibbs draws come from a Philox counter RNG on the device, seeded from the global numpy RNG
    (so `np.random.seed` still makes `fit` reproducible).  `B200_CONFIG['rng'] = 'numpy'` (or env
    FOKL_B200_RNG=numpy) injects the legacy numpy variates in the reference's exact order instead;
  * `relats_in` with exclusions raises, as it does upstream (FR:1631 is broken);
  * `update=True` (fitupdate, FR:1850-2583) runs on the device too (FoKL/_update.py, csrc/update.cu);
  * `to_pyomo` is not built and raises (DESIGN.md section 7);
    `bss_derivatives`, `evaluate` and `coverage3` run on the device like `fit`;
  * `bss_derivatives(kernel=<int>)` resolves the index and an unknown kernel name raises ValueError -- upstream both die
    of an UnboundLocalError (FR:728-777).  Every other host-side call is held to the live reference outcome by outcome
    (values, exception types, warning texts) by tests/test_reference_differential.py.
"""
import copy
import math
import os
import pickle
import sys
import time
import warnings

import numpy as np

from . import getKernels

# process-wide knobs of the B200 build (not hyper-parameters; never pickled)
B200_CONFIG = {
    'rng': os.environ.get('FOKL_B200_RNG', 'philox'),       # 'philox' | 'numpy'
    'eager_chains': os.environ.get('FOKL_B200_EAGER', '0') not in ('0', '', 'false', 'False'),
    'device': None,                                         # torch device / index; None = current device
    # evaluate the chains that verify a substage together with the next substage's full model (same fit, bit for bit)
    'pipeline': os.environ.get('FOKL_B200_PIPELINE', '1') not in ('0', '', 'false', 'False'),
    # build the next substage's columns and the stable part of its Gram block while the current substage's candidate
    # stage runs (same Gram bits, same fit)
    # (opt-in: measured 165 ms vs 151 ms per cfg4 fit, DESIGN.md section 3b -- the second pass over the new columns and
    # the SMs left to the candidate stage cost more than the overlap returns)
    'prefetch': os.environ.get('FOKL_B200_PREFETCH', '0') not in ('0', '', 'false', 'False'),
    # chains of the nested accepted models of a substage by secular-equation updates instead of one eigensolver run per
    # model (csrc/nested.cu); same decisions, the intercept means agree to ~1e-13
    'nested_chains': os.environ.get('FOKL_B200_NESTED', '1') not in ('0', '', 'false', 'False'),
    'nested_min_p': int(os.environ.get('FOKL_B200_NESTED_MIN_P', '256')),     # narrower batches: one solver per model
    # a substage's kill loop starts from the full model's eigendecomposition (tableau = -A^-1 formed by the whole
    # device) instead of sweeping its p pivots one after the other; same decisions, BICs agree to ~1e-12
    'kill_from_eig': os.environ.get('FOKL_B200_KILL_FROM_EIG', '1') not in ('0', '', 'false', 'False'),
}

_ENGINES = {}
LAST_FIT_INFO = {}

# evaluate / coverage3 / bss_derivatives reduce the N x draws product on the device (fokl_predict_summary: mean and two
# order statistics per row, the same bits as numpy on the full product) once it has at least this many cells; smaller
# products are copied to the host and reduced by numpy (fokl_predict_draws)
_PREDICT_SUMMARY_MIN_CELLS = 1 << 24
# rows of the design matrix built per K1 launch on the summary path (a multiple of 16 for K1's 16-byte stores): bounds
# the device memory of a prediction independently of N
_PREDICT_CHUNK_ROWS = 1 << 16
# bss_derivatives streams its rows through fokl_deriv_summary (eng_derivative_summary) once N * draws reaches this many
# cells and draws > 1 -- evaluate's rule.  It is a name of its own so that the mean-only path through
# fokl_predict_summary (eng_derivative_draws) stays selectable on its own.
_DERIV_SUMMARY_MIN_CELLS = 1 << 24
# device bytes of one row chunk of dy on that path (N x M x 2 x draws with IndividualDraws=True): fewer rows per chunk
# than _PREDICT_CHUNK_ROWS when a chunk would be larger
_DERIV_CHUNK_BYTES = 256 << 20
# `clean` (fit(clean=True), evaluate(inputs, clean=True)) formats, normalises and splits the dataset in HBM once the raw
# inputs have at least this many cells; smaller datasets take the host path, where the pass over them costs little
_CLEAN_ON_DEVICE_MIN_CELLS = 1 << 20
# generate_trainlog draws its split in HBM (fokl_trainlog: the host loop's mask and numpy RNG end state, bit for bit)
# from this many rows, wherever the dataset is cleaned; below it the host loop costs little
_TRAINLOG_ON_DEVICE_MIN_ROWS = 1 << 20


def _engine(device=None):
    """One Engine (CUDA context handle + scratch) per (process, device)."""
    from ._engine import Engine
    import torch
    if device is None:
        device = B200_CONFIG['device']
    if device is None:
        if not torch.cuda.is_available():
            raise RuntimeError("FoKL (B200 build) needs a CUDA device: there is no CPU fallback for fit().")
        device = torch.cuda.current_device()
    dev = torch.device('cuda', device) if isinstance(device, int) else torch.device(device)
    key = (dev.index, torch.cuda.current_stream(dev).cuda_stream)
    if key not in _ENGINES:
        _ENGINES[key] = Engine(dev)
    return _ENGINES[key]


def load(filename, directory=None):
    """Load a FoKL class from a file written by `save` (FR:24-46)."""
    if filename[-5::] != ".fokl":
        filename = filename + ".fokl"
    filepath = os.path.join(directory, filename) if directory is not None else filename
    with open(filepath, "rb") as file:
        return pickle.load(file)


def _str_to_bool(s):
    """'on'/'off'-style strings and other truthy values to bool (FR:49-68)."""
    if isinstance(s, str):
        if s in ['yes', 'y', 'on', 'all', 'true', 'both']:
            return True
        if s in ['no', 'n', 'off', 'none', 'n/a', 'false']:
            return False
        warnings.warn(f"Could not understand string '{s}' as a boolean.", category=UserWarning)
        return s
    if s is None or not s:
        return False
    try:
        return bool(s != 0)
    except Exception:
        warnings.warn("Could not convert non-string to a boolean.", category=UserWarning)
        return s


def _process_kwargs(default, user):
    """Merge user kwargs over defaults, raising on unknown keys (FR:71-90)."""
    if isinstance(default, dict):
        if not isinstance(user, dict):
            raise ValueError("Input 'user' must be a dictionary formed by kwargs.")
        for kw in user.keys():
            if kw not in default:
                raise ValueError(f"Unexpected keyword argument: '{kw}'")
            default[kw] = user[kw]
        return default
    if isinstance(default, list):
        for kw in user.keys():
            if kw not in default:
                raise ValueError(f"Unexpected keyword argument: '{kw}'")
        return user
    raise ValueError("Input 'default' must be a dictionary or list.")


def _set_attributes(self, attrs):
    """Set the items of the dictionary `attrs` as attributes of `self` (FR:93-100)."""
    if isinstance(attrs, dict):
        for key, value in attrs.items():
            setattr(self, key, value)
    else:
        warnings.warn("Input must be a Python dictionary.")


def _merge_dicts(d1, d2):
    d = d1.copy()
    d.update(d2)
    return d


def _column_minmax_host(inputs):
    """Per-column [min, max] of a host array; under torch.distributed the bounds are reduced over all ranks (every
    rank holds a row shard of the same dataset and must normalise it identically)."""
    mm = inputs.shape[1]
    bounds = [[np.min(inputs[:, m]), np.max(inputs[:, m])] for m in range(mm)]
    try:
        import torch
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            dev = torch.device('cuda', torch.cuda.current_device()) if dist.get_backend() == 'nccl' else torch.device('cpu')
            lo = torch.tensor([b[0] for b in bounds], dtype=torch.float64, device=dev)
            hi = torch.tensor([b[1] for b in bounds], dtype=torch.float64, device=dev)
            dist.all_reduce(lo, op=dist.ReduceOp.MIN)
            dist.all_reduce(hi, op=dist.ReduceOp.MAX)
            bounds = [[a, b] for a, b in zip(lo.cpu().numpy(), hi.cpu().numpy())]
    except ImportError:
        pass
    return bounds


def _have_cuda():
    try:
        import torch
        return torch.cuda.is_available()
    except ImportError:
        return False


def _device_trainlog(train, n):
    """`generate_trainlog(train, n)`'s mask as a device uint8 tensor, drawn by fokl_trainlog from the legacy numpy RNG,
    whose state it then advances exactly as the host loop would (has_gauss / cached_gaussian are left as they were).
    None when the split is not drawn on the device: train >= 1, n below _TRAINLOG_ON_DEVICE_MIN_ROWS or at least 2^31,
    or no CUDA device."""
    if not (train < 1 and _TRAINLOG_ON_DEVICE_MIN_ROWS <= n < (1 << 31) and _have_cuda()):
        return None
    state = np.random.get_state()
    keep, key, pos, _ = _engine().trainlog(state[1], state[2], n, max(int(n * train), 2))
    np.random.set_state((state[0], key, pos, state[3], state[4]))
    return keep


def _dist_world():
    """torch.distributed when it is initialised with more than one rank, else None."""
    try:
        import torch.distributed as dist
    except ImportError:
        return None
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        return dist
    return None


class _DeviceInputs:
    """Normalised inputs that so far exist only in HBM (fit(clean=True) normalised them on the device).  `FoKL.inputs`
    copies them to a host numpy array on first access, so the attribute behaves exactly like the reference's."""

    def __init__(self, ds):
        self.ds = ds

    def to_numpy(self):
        ds = self.ds
        return np.ascontiguousarray(ds.x[:, :ds.n].t().contiguous().cpu().numpy())


_CLEAN_DEFAULTS = {'train': 1, 'AutoTranspose': True, 'SingleInstance': False, 'bit': 64, 'normalize': True,
                   'minmax': None, 'pillow': None, 'pillow_type': 'percent'}


class FoKL:
    def __init__(self, **kwargs):
        """Hyper-parameters and defaults exactly as the reference (FR:111-246):

            kernel='Cubic Splines', phis=f(kernel), relats_in=[], a=4, b=f(a, data), atau=4, btau=f(atau, data),
            tolerance=3, burnin=1000, draws=1000, gimmie=False, way3=False, threshav=0.05, threshstda=0.5,
            threshstdb=2, aic=False, sigsqd0=0.5, burn=500, update=False, built=False,
            UserWarnings=True, ConsoleOutput=True
        """
        self.hypers = ['kernel', 'phis', 'relats_in', 'a', 'b', 'atau', 'btau', 'tolerance', 'burnin', 'draws',
                       'gimmie', 'way3', 'threshav', 'threshstda', 'threshstdb', 'aic', 'update', 'built']
        self.settings = ['UserWarnings', 'ConsoleOutput']
        self.kernels = ['Cubic Splines', 'Bernoulli Polynomials']
        self.keep = ['keep', 'hypers', 'settings', 'kernels'] + self.hypers + self.settings + self.kernels

        default = {'kernel': 'Cubic Splines', 'phis': None, 'relats_in': [], 'a': 4, 'b': None, 'atau': 4,
                   'btau': None, 'tolerance': 3, 'burnin': 1000, 'draws': 1000, 'gimmie': False, 'way3': False,
                   'threshav': 0.05, 'threshstda': 0.5, 'threshstdb': 2, 'aic': False,
                   'sigsqd0': 0.5, 'burn': 500, 'update': False, 'built': False,
                   'UserWarnings': True, 'ConsoleOutput': True}
        current = _process_kwargs(default, kwargs)
        for boolean in ['gimmie', 'way3', 'aic', 'UserWarnings', 'ConsoleOutput']:
            if not (current[boolean] is False or current[boolean] is True):
                current[boolean] = _str_to_bool(current[boolean])

        if isinstance(current['kernel'], int):
            current['kernel'] = self.kernels[current['kernel']]
        if current['phis'] is None:
            if current['kernel'] == self.kernels[0]:
                current['phis'] = getKernels.sp500()
            elif current['kernel'] == self.kernels[1]:
                current['phis'] = getKernels.bernoulli()
            elif isinstance(current['kernel'], str):
                raise ValueError(f"The user-provided kernel '{current['phis']}' is not supported.")
            else:
                raise ValueError("The user-provided kernel is not supported.")

        if current['UserWarnings']:
            warnings.filterwarnings("default", category=UserWarning)
        else:
            warnings.filterwarnings("ignore", category=UserWarning)

        for key, value in current.items():
            setattr(self, key, value)
        self.setnos = None

    # `inputs` is stored like any other attribute (same key in __dict__ and in the pickle as the reference); the
    # property only materialises a device-resident normalised dataset on first access.
    @property
    def inputs(self):
        try:
            v = self.__dict__['inputs']
        except KeyError:
            raise AttributeError("'FoKL' object has no attribute 'inputs'") from None
        if isinstance(v, _DeviceInputs):
            v = v.to_numpy()
            self.__dict__['inputs'] = v
        return v

    @inputs.setter
    def inputs(self, value):
        self.__dict__['inputs'] = value

    @inputs.deleter
    def inputs(self):
        try:
            del self.__dict__['inputs']
        except KeyError:
            raise AttributeError('inputs') from None

    def __getstate__(self):
        state = dict(self.__dict__)
        if isinstance(state.get('inputs'), _DeviceInputs):
            state['inputs'] = self.inputs
        return state

    # ------------------------------------------------------------------------------------------------
    # dataset formatting (host side; FR:248-542)
    # ------------------------------------------------------------------------------------------------
    def _format(self, inputs, data=None, AutoTranspose=True, SingleInstance=False, bit=64, _copy=True, _widen=True):
        """inputs -> [n x m] ndarray, data -> [n x 1] ndarray (FR:248-316).  _widen=False: float32 inputs are returned
        as float32 (with the same warning) for the caller to widen on the device, where the conversion is exact too."""
        import pandas as pd
        AutoTranspose = _str_to_bool(AutoTranspose)
        SingleInstance = _str_to_bool(SingleInstance)
        bits = {16: np.float16, 32: np.float32, 64: np.float64}
        if SingleInstance is True:
            AutoTranspose = False
        if bit not in bits:
            warnings.warn(f"Keyword 'bit={bit}' limited to values of 16, 32, or 64. Assuming default value of 64.",
                          category=UserWarning)
            bit = 64
        datatype = bits[bit]

        if isinstance(inputs, (pd.DataFrame, pd.Series)):
            inputs = inputs.to_numpy()
            warnings.warn("'inputs' was auto-converted to numpy. Convert manually for assured accuracy.",
                          category=UserWarning)
        if data is not None and isinstance(data, (pd.DataFrame, pd.Series)):
            data = data.to_numpy()
            warnings.warn("'data' was auto-converted to numpy. Convert manually for assured accuracy.",
                          category=UserWarning)

        inputs = np.array(inputs) if _copy else np.asarray(inputs)
        if inputs.ndim > 2:
            inputs = np.squeeze(inputs)
        if inputs.dtype != datatype:
            if _widen or not (inputs.dtype == np.float32 and datatype == np.float64):
                inputs = np.array(inputs, dtype=datatype)
            warnings.warn(f"'inputs' was converted to float{bit}. May require user-confirmation that "
                          f"values did not get corrupted.", category=UserWarning)
        if inputs.ndim == 1:
            inputs = inputs[np.newaxis, :] if SingleInstance is True else inputs[:, np.newaxis]
        if AutoTranspose is True and SingleInstance is False:
            if inputs.shape[1] > inputs.shape[0]:
                inputs = inputs.transpose()
                warnings.warn("'inputs' was transposed. Ignore if more datapoints than input variables, else set "
                              "'AutoTranspose=False' to disable.", category=UserWarning)

        if data is not None:
            data = np.squeeze(np.array(data) if _copy else np.asarray(data))
            if data.dtype != datatype:
                data = np.array(data, dtype=datatype)
                warnings.warn(f"'data' was converted to float{bit}. May require user-confirmation that "
                              f"values did not get corrupted.", category=UserWarning)
            if data.ndim == 1:
                data = data[:, np.newaxis]
            else:
                n, m = data.shape[0], data.shape[1]
                if (m != 1 and n != 1) or (m == 1 and n == 1):
                    raise ValueError("Error: 'data' must be a vector.")
                elif m != 1 and n == 1:
                    data = data.transpose()
                    warnings.warn("'data' was transposed to match FoKL formatting.", category=UserWarning)
        return inputs, data

    def _normalize(self, inputs, minmax=None, pillow=None, pillow_type='percent'):
        """Min-max normalise the columns of `inputs` in place; updates self.minmax (FR:318-439)."""
        mm = inputs.shape[1]
        minmax = self._normalize_bounds(mm, lambda: _column_minmax_host(inputs), minmax, pillow, pillow_type)
        for m in range(mm):
            inputs[:, m] = (inputs[:, m] - minmax[m][0]) / (minmax[m][1] - minmax[m][0])
        return inputs

    def _normalize_bounds(self, mm, column_minmax, minmax=None, pillow=None, pillow_type='percent'):
        """The [min, max] pair per input that `_normalize` applies (FR:318-435): user `minmax`, else the model's, else
        the data's (`column_minmax()` -> [[min, max], ...], evaluated only when needed), widened by `pillow`.
        Sets self.minmax."""
        pillow_types = ['percent', 'absolute']
        if isinstance(pillow_type, str):
            pillow_type = [pillow_type] * mm
        elif isinstance(pillow_type, list) and len(pillow_type) != mm:
            raise ValueError("Input 'pillow_type' must be string or correspond to input variables (i.e., columns of 'inputs').")
        for pt in pillow_type:
            if pt not in pillow_types:
                raise ValueError(f"'pillow_type' is limited to {pillow_types}.")

        skip_pillow = pillow is None
        if skip_pillow:
            pillow = 0.0
        if isinstance(pillow, int):
            pillow = float(pillow)
        if isinstance(pillow, float):
            pillow = [[pillow, pillow]] * mm
        elif isinstance(pillow[0], (int, float)):
            lp = len(pillow)
            if lp == 2:
                pillow = [[float(pillow[0]), float(pillow[1])]]
                lp = 1
            if lp != int(mm * 2):
                raise ValueError("Input 'pillow' must correspond to input variables (i.e., columns of 'inputs').")
            vals = copy.deepcopy(pillow)
            pillow = [[float(vals[i]), float(vals[i + 1])] for i in range(0, lp, 2)]

        def _minmax_error():
            raise ValueError("Input 'minmax' must correspond to input variables (i.e., columns of 'inputs').")

        if minmax is None:
            if hasattr(self, 'minmax'):
                minmax = self.minmax
            else:
                minmax = column_minmax()
        else:
            if isinstance(minmax[0], (int, float)):
                lm = len(minmax)
                if lm == 2:
                    minmax = [minmax]
                    lm = 1
                if lm != int(mm * 2):
                    _minmax_error()
                else:
                    vals = copy.deepcopy(minmax)
                    minmax = [[vals[i], vals[i + 1]] for i in range(0, lm, 2)]
            elif len(minmax) != mm:
                _minmax_error()

        if pillow is not None and skip_pillow is False:
            vals = copy.deepcopy(minmax)
            minmax = []
            for m in range(mm):
                x_min, x_max = vals[m][0], vals[m][1]
                span = x_max - x_min
                if pillow_type[m] == 'percent':
                    minmax.append([x_min - span * pillow[m][0], x_max + span * pillow[m][1]])
                else:  # 'absolute': choose [min, max] so that the data span maps onto [q, 1 - p]
                    q, p1 = pillow[m][0], pillow[m][1]
                    lo = x_min if q == 0 else (x_min * (1 - p1) - x_max * q) / (1 - p1 - q)
                    if p1 == 0:
                        hi = x_max
                    elif q == 0:
                        hi = (x_max - p1 * lo) / (1 - p1)
                    else:
                        hi = (x_min - lo) / q + lo
                    minmax.append([lo, hi])

        if hasattr(self, 'minmax'):
            if any(minmax[m] == self.minmax[m] for m in range(mm)) is False:
                warnings.warn("The model already contains normalization [min, max] bounds, so the currently trained "
                              "model will not be valid for the new bounds requested. Train a new model with these "
                              "new bounds.", category=UserWarning)
        self.minmax = minmax
        return minmax

    def clean(self, inputs, data=None, kwargs_from_other=None, _setattr=False, **kwargs):
        """Format and (by default) normalise a dataset; see the reference for the keywords (FR:441-507):
        train, AutoTranspose, SingleInstance, bit, normalize, minmax, pillow, pillow_type."""
        default = dict(_CLEAN_DEFAULTS)
        if kwargs_from_other is not None:
            kwargs = _merge_dicts(kwargs, kwargs_from_other)
        current = _process_kwargs(default, kwargs)
        current['normalize'] = _str_to_bool(current['normalize'])

        inputs, data = self._format(inputs, data, current['AutoTranspose'], current['SingleInstance'], current['bit'])
        if current['normalize'] is True:
            inputs = self._normalize(inputs, current['minmax'], current['pillow'], current['pillow_type'])
            # (the reference's capping of values outside [0, 1] is dead code -- `np.max(...) is True`, FR:488)

        if hasattr(self, 'inputs') is False or _setattr is True:
            trainlog, _ = self._shard_trainlog(current['train'], inputs.shape[0])
            self.inputs, self.data, self.trainlog = inputs, data, trainlog

        if data is None:
            return inputs
        return inputs, data

    def generate_trainlog(self, train, n=None):
        """Random logical vector of length n with `train` percent True, or None for "all" (FR:509-530)."""
        if train < 1:
            if n is None:
                n = self.inputs.shape[0]
            keep = _device_trainlog(train, n)
            if keep is not None:
                return keep.cpu().numpy().view(bool)
            l_log = max(int(n * train), 2)
            idx = np.array([], dtype=int)
            while len(idx) < l_log:
                idx = np.append(idx, np.random.randint(1, n + 1, size=l_log) - 1)
                idx = np.unique(idx)
                np.random.shuffle(idx)
            idx = idx[0:l_log]
            trainlog = np.zeros(n, dtype=bool)
            trainlog[idx] = True
            return trainlog
        return None

    def _shard_trainlog(self, train, n):
        """`generate_trainlog(train, n)` for the n rows `clean` was given: (host bool mask or None, the same mask as a
        device uint8 tensor when it was drawn there, else None).  Under torch.distributed every rank holds a row shard
        of one dataset, in rank order: the shard sizes are gathered, rank 0's numpy RNG state is broadcast, every rank
        draws the split of all N rows (in HBM from _TRAINLOG_ON_DEVICE_MIN_ROWS rows on, as a single process would) and
        keeps its own rows.  So the shards' masks concatenate to the single-process mask, and every rank's RNG ends in
        the single process's state."""
        if not train < 1:
            return None, None
        dist = _dist_world()
        lo, total = 0, n
        if dist is not None:
            import torch
            dev = torch.device('cuda', torch.cuda.current_device()) if dist.get_backend() == 'nccl' else torch.device('cpu')
            mine = torch.tensor([n], dtype=torch.int64, device=dev)
            sizes = [torch.zeros_like(mine) for _ in range(dist.get_world_size())]
            dist.all_gather(sizes, mine)
            sizes = [int(t.item()) for t in sizes]
            lo, total = sum(sizes[:dist.get_rank()]), sum(sizes)
            st = np.random.get_state()
            packed = np.concatenate([np.asarray(st[1], dtype=np.int64), [st[2], st[3]],
                                     np.array([st[4]], dtype=np.float64).view(np.int64)])
            t = torch.from_numpy(packed).to(dev)
            dist.broadcast(t, src=0)
            packed = t.cpu().numpy()
            np.random.set_state(('MT19937', packed[:624].astype(np.uint32), int(packed[624]), int(packed[625]),
                                 float(packed[626:627].view(np.float64)[0])))
        keep = _device_trainlog(train, total)
        if keep is None:
            mask = self.generate_trainlog(train, total)
            return (mask if dist is None else mask[lo:lo + n].copy()), None
        keep = keep[lo:lo + n]
        return keep.cpu().numpy().view(bool), keep

    def trainset(self):
        """Train inputs and data after `clean` (FR:532-542)."""
        if self.trainlog is None:
            return self.inputs, self.data
        return self.inputs[self.trainlog, :], self.data[self.trainlog]

    def _inputs_to_phind(self, inputs, phis=None, kernel=None):
        """Piece index and local coordinate of the cubic splines (FR:544-592); host numpy helper kept for API
        compatibility -- the fit path recomputes both inside the basis kernel."""
        if kernel is None:
            kernel = self.kernel
        if phis is None:
            phis = self.phis
        if kernel == self.kernels[1]:
            warnings.warn("Twice normalization of inputs is not required for the 'Bernoulli Polynomials' kernel",
                          category=UserWarning)
            return inputs, [], []
        l_phis = len(phis[0][0])
        phind = np.array(np.ceil(inputs * l_phis), dtype=np.uint16)
        if phind.ndim == 1:
            phind = phind[:, np.newaxis]
        phind = phind + (phind == 0)
        try:
            inputs.dtype
        except AttributeError:
            raise AttributeError("Inputs must be a numpy array, to process automatically try making clean = True")
        r = 1 / l_phis
        xmin = np.array((phind - 1) * r, dtype=inputs.dtype)
        X = (inputs - xmin) / r
        phind = phind - 1
        xsm = np.array(l_phis * inputs - phind, dtype=inputs.dtype)
        if np.max(phind) > 499 or np.min(phind) < 0:
            raise ValueError('Inputs are not normalized correctly, try calling clean=True within evaluate to '
                             'evaluate with normalization of model training')
        return X, phind, xsm

    def evaluate_basis(self, c, x, kernel=None, d=0):
        """One basis function (or its 1st/2nd derivative) at x from coefficients c (FR:807-849)."""
        if kernel is None:
            kernel = self.kernel
        elif isinstance(kernel, int):
            kernel = self.kernels[kernel]
        if kernel not in self.kernels:
            raise ValueError(f"The kernel {kernel} is not currently supported. Please select from the following: "
                             f"{self.kernels}.")
        if kernel == self.kernels[0]:
            if d == 0:
                basis = c[0] + c[1] * x + c[2] * (x ** 2) + c[3] * (x ** 3)
            elif d == 1:
                basis = c[1] + 2 * c[2] * x + 3 * c[3] * (x ** 2)
            elif d == 2:
                basis = 2 * c[2] + 6 * c[3] * x
        else:
            if d == 0:
                basis = c[0] + sum(c[k] * (x ** k) for k in range(1, len(c)))
            elif d == 1:
                basis = c[1] + sum(k * c[k] * (x ** (k - 1)) for k in range(2, len(c)))
            elif d == 2:
                basis = sum((k - 1) * k * c[k] * (x ** (k - 2)) for k in range(2, len(c)))
        return basis

    # ------------------------------------------------------------------------------------------------
    # prediction (FR:851-1200)
    # ------------------------------------------------------------------------------------------------
    def evaluate(self, inputs=None, betas=None, mtx=None, draws=None, **kwargs):
        """Evaluate the model at `inputs`; optionally return 95 % bounds (FR:851-980).  The design matrix and
        the X @ betas' product run on the device (K1 + fokl_predict_draws)."""
        if not hasattr(self, 'minmax'):
            raise ValueError("To set minmax manually call model.minmax = ([input_min, input_max],[data_min, data_max],...)"
                             " or set clean=True to automtically define min and max from model.inputs")
        default = {'minmax': None, 'draws': self.draws, 'clean': False, 'ReturnBounds': False,
                   '_suppress_normalization_warning': False, 'betas': self.betas, 'mtx': self.mtx}
        default_for_clean = dict(_CLEAN_DEFAULTS)
        default_for_clean['minmax'] = self.minmax
        current = _process_kwargs(_merge_dicts(default, default_for_clean), kwargs)
        for boolean in ['clean', 'ReturnBounds']:
            current[boolean] = _str_to_bool(current[boolean])
        kwargs_to_clean = {}
        for kwarg in default_for_clean.keys():
            kwargs_to_clean[kwarg] = current[kwarg]
            del current[kwarg]
        if current['draws'] < 40 and current['ReturnBounds']:
            warnings.warn("'draws' must be greater than or equal to 40 to calculate 95% confidence interval bounds.'.")
        if betas is None:
            betas = self.betas
        if draws is None:
            draws = self.draws
        elif betas.shape[0] < draws:
            raise ValueError(f"The number of draws: {draws}  exceeds the number of draws in betas: {betas.shape[0]}"
                             f", \n       draws must be < betas.")
        if mtx is None:
            mtx = self.mtx
        else:
            if isinstance(mtx, int):
                mtx = [mtx]
            mtx = np.array(mtx)
            if mtx.ndim == 1:
                mtx = mtx[np.newaxis, :]
                warnings.warn("Assuming 'mtx' represents a single model. If meant to represent several models, then "
                              "explicitly enter a 2D numpy array where rows correspond to models.")

        if inputs is None:
            if current['clean']:
                warnings.warn("Cleaning was already performed on default 'inputs', so overriding 'clean' to False.",
                              category=UserWarning)
                current['clean'] = False
            resident = self._resident_inputs()
            normputs = resident if resident is not None else self.inputs
        elif current['clean']:
            normputs = self._evaluate_clean(inputs, kwargs_to_clean, draws)
        else:
            normputs = np.array(inputs)

        betas = np.asarray(betas, dtype=np.float64)
        m, mbets = np.shape(betas)
        if isinstance(normputs, _DeviceInputs):
            n, mputs = normputs.ds.n, normputs.ds.m
        else:
            normputs = np.asarray(normputs, dtype=np.float64)
            n = np.shape(normputs)[0]
            mputs = int(np.size(normputs) / n)
            normputs = normputs.reshape(n, mputs)

        if self.setnos is None:
            setnos = np.random.choice(m, draws, replace=False)
            self.setnos = setnos
        else:
            setnos = self.setnos
        if draws == 1:
            setnos = [0]

        terms = np.asarray(mtx, dtype=np.float64).reshape(mbets - 1, mputs) if mbets > 1 else np.zeros((0, mputs))
        eng = _engine()
        betas_sel = betas[np.asarray(setnos)[:draws], :]
        if draws >= 2 and betas_sel.shape[0] == draws and n * draws >= _PREDICT_SUMMARY_MIN_CELLS:
            cut = int(np.floor(draws * 0.025) + 1)
            with_bounds = current['ReturnBounds'] == True  # noqa: E712
            mean, lo, hi = eng_predict_summary(eng, self.phis, self.kernel, normputs, terms, betas_sel,
                                               (cut, draws - cut) if with_bounds else None)
            if with_bounds:
                bounds = np.zeros((n, 2))
                bounds[:, 0] = lo
                bounds[:, 1] = hi
                return mean, bounds
            return mean
        if isinstance(normputs, _DeviceInputs):
            normputs = self.inputs if normputs is self.__dict__.get('inputs') else normputs.to_numpy()
        modells = eng_predict(eng, self.phis, self.kernel, normputs, terms, betas_sel)
        mean = np.mean(modells, 1)

        if current['ReturnBounds'] == True:  # noqa: E712  (reference semantics: 1 == True)
            bounds = np.zeros((n, 2))
            cut = int(np.floor(draws * 0.025) + 1)
            srt = np.sort(modells, axis=1)
            bounds[:, 0] = srt[:, cut]
            bounds[:, 1] = srt[:, draws - cut]
            return mean, bounds
        return mean

    def _resident_inputs(self):
        """The default inputs when they live only in HBM (fit(clean=True) on a large dataset) and this process is the only
        rank, so evaluate may read them there; None otherwise."""
        v = self.__dict__.get('inputs')
        if isinstance(v, _DeviceInputs) and _engine().world == 1:
            return v
        return None

    def coverage3(self, **kwargs):
        """Validation: predicted mean, confidence bounds and 'rmse' over a dataset (FR:982-1200).
        Plotting needs matplotlib and is skipped with a warning when it is not installed."""
        try:
            self.draws
        except Exception:
            raise ValueError("self.draws is undefined, specify number of draws to evaluate as kwarg: draws = ")
        default = {'inputs': None, 'data': None, 'draws': self.draws, 'betas': self.betas,
                   'plot': False, 'bounds': True, 'xaxis': False, 'labels': True, 'xlabel': 'Index', 'ylabel': 'Data',
                   'title': 'FoKL', 'legend': True, 'LegendLabelFoKL': 'FoKL', 'LegendLabelData': 'Data',
                   'LegendLabelBounds': 'Bounds', 'ReturnBounds': True,
                   'PlotTypeFoKL': 'b', 'PlotSizeFoKL': 2, 'PlotTypeBounds': 'k--', 'PlotSizeBounds': 2,
                   'PlotTypeData': 'ro', 'PlotSizeData': 2}
        current = _process_kwargs(default, kwargs)
        if isinstance(current['plot'], str):
            if current['plot'].lower() in ['sort', 'sorted', 'order', 'ordered']:
                current['plot'] = 'sorted'
                if current['xlabel'] == 'Index':
                    current['xlabel'] = 'Index (Sorted)'
            else:
                warnings.warn("Keyword input 'plot' is limited to True, False, or 'sorted'.", category=UserWarning)
                current['plot'] = False
        else:
            current['plot'] = _str_to_bool(current['plot'])
        for boolean in ['bounds', 'labels', 'legend']:
            current[boolean] = _str_to_bool(current[boolean])
        # device-resident default inputs: evaluate(None) reads them in HBM; the plot materialises them only for `xaxis`
        resident = current['inputs'] is None and self._resident_inputs() is not None

        warn_plot = ' and ignoring plot.' if current['plot'] else '.'
        for this, other in (('inputs', 'data'), ('data', 'inputs')):
            if current[this] is not None and current[other] is None:
                warnings.warn(f"Keyword argument '{other}' should be defined to align with user-defined '{this}'. "
                              f"Ignoring RMSE calculation{warn_plot}", category=UserWarning)
                current['data'] = False
        if current['data'] is False and current['plot'] == 'sorted':
            warnings.warn("Keyword argument 'data' must correspond with 'inputs' if requesting a sorted plot. "
                          "Returning a regular plot instead.", category=UserWarning)
            current['plot'] = True

        if current['inputs'] is None and not resident:
            current['inputs'] = self.inputs
        if current['data'] is None:
            current['data'] = self.data

        normputs = current['inputs']
        data = current['data']
        draws = current['draws']
        if draws > np.shape(current['betas'])[0]:
            raise ValueError(f"Number of draws called ({draws}) exceeds number of rows of betas "
                             f"({np.shape(current['betas'])[0]}) ")
        bounds = None
        if current['ReturnBounds'] == True:  # noqa: E712
            mean, bounds = self.evaluate(normputs, betas=current['betas'], draws=draws, ReturnBounds=1,
                                         _suppress_normalization_warning=True)
        else:
            mean = self.evaluate(normputs, betas=current['betas'], draws=draws, ReturnBounds=0,
                                 _suppress_normalization_warning=True)

        if current['plot']:
            if resident and current['xaxis'] is not False and isinstance(current['xaxis'], int):
                normputs = self.inputs
            self._plot_coverage(current, normputs, data, mean, bounds)

        if data is not False:
            d = np.asarray(data)
            if d.ndim == 2 and d.shape[1] == 1 and np.size(mean) * d.shape[0] > _PREDICT_SUMMARY_MIN_CELLS:
                # the reference's expression (FR:1193) broadcasts (n,) - (n, 1) to an n x n array; the mean of
                # mean_c - data_r over all (r, c) is mean(mean) - mean(data), equal up to the last bits
                rmse = np.abs(np.mean(mean) - np.mean(d))
            else:
                # reference quirk kept (FR:1193): (n,) - (n, 1) broadcasts to n x n; equals |mean(mean) - mean(data)|
                rmse = np.sqrt(np.mean(mean - data) ** 2)
        else:
            rmse = []
        if current['ReturnBounds'] == True:  # noqa: E712
            return mean, bounds, rmse
        return mean, rmse

    def _plot_coverage(self, current, normputs, data, mean, bounds):
        try:
            import matplotlib.pyplot as plt
        except ImportError:
            warnings.warn("matplotlib is not installed; skipping the coverage3 plot.", category=UserWarning)
            return
        n = len(mean)
        if current['xaxis'] is False:
            plt_x = np.linspace(0, n - 1, n)
        elif isinstance(current['xaxis'], int):
            lo, hi = self.minmax[current['xaxis']]
            plt_x = np.array(normputs)[:, current['xaxis']] * (hi - lo) + lo
        else:
            plt_x = current['xaxis']
        plt_mean, plt_bounds, plt_data = mean, bounds, data
        if current['plot'] == 'sorted':
            sort_id = np.argsort(np.squeeze(data))
            plt_mean, plt_data = mean[sort_id], data[sort_id]
            plt_bounds = bounds[sort_id] if bounds is not None else None
        plt.figure()
        plt.plot(plt_x, plt_mean, current['PlotTypeFoKL'], linewidth=current['PlotSizeFoKL'],
                 label=current['LegendLabelFoKL'])
        if data is not False:
            plt.plot(plt_x, plt_data, current['PlotTypeData'], markersize=current['PlotSizeData'],
                     label=current['LegendLabelData'])
        if current['bounds'] and plt_bounds is not None:
            plt.plot(plt_x, plt_bounds[:, 0], current['PlotTypeBounds'], linewidth=current['PlotSizeBounds'],
                     label=current['LegendLabelBounds'])
            plt.plot(plt_x, plt_bounds[:, 1], current['PlotTypeBounds'], linewidth=current['PlotSizeBounds'])
        if current['labels']:
            for fn, key in ((plt.xlabel, 'xlabel'), (plt.ylabel, 'ylabel'), (plt.title, 'title')):
                if current[key]:
                    fn(str(current[key]))
        if current['legend']:
            plt.legend()
        plt.show()

    def _device_raw_inputs(self, inputs, current):
        """The raw `inputs` of a `clean` request (keywords resolved in `current`) that may be formatted and normalised in
        HBM without a host pass over them: float32 / float64 numpy arrays, and pandas frames of one such dtype (their
        block goes up as it is), of at least _CLEAN_ON_DEVICE_MIN_CELLS cells, with bit=64 and normalize=True.  None
        for anything else (mixed-dtype or object frames, other dtypes, small datasets): that takes the host path."""
        if current['bit'] != 64 or _str_to_bool(current['normalize']) is not True:
            return None
        floats = (np.dtype(np.float32), np.dtype(np.float64))
        try:
            import pandas as pd
            if isinstance(inputs, pd.DataFrame):
                dtypes = set(inputs.dtypes)
                ok = len(dtypes) == 1 and dtypes.pop() in floats
                return inputs if ok and inputs.size >= _CLEAN_ON_DEVICE_MIN_CELLS else None
            if isinstance(inputs, pd.Series):
                return None
        except ImportError:
            pass
        raw = np.asarray(inputs)
        if raw.dtype not in floats or raw.size < _CLEAN_ON_DEVICE_MIN_CELLS:
            return None
        return raw

    def _clean_on_device(self, inputs, data, kwargs_to_clean):
        """`clean` for `fit(clean=True)` done in HBM (FR:248-542): `_format`'s checks and warnings run on the host
        unchanged, but the raw inputs go to the device as they are (float32 widened, a column-major block transposed
        there), the per-column min / max and (x - min) / (max - min) run there (bit-identical to the host expression),
        and a train split (`_shard_trainlog`; a mask drawn in HBM goes to the kernel as it is) keeps its rows with
        fokl_rows_compact.  Sets
        `inputs` (the train rows, materialised on the host only if somebody reads them), `data` (the train rows) and
        `trainlog` as the host path's `fit` leaves them.  Returns (DeviceDataset of the train rows, moments_on_device)
        or None when the request needs the host path (_device_raw_inputs).  moments_on_device: the b / btau defaults
        come from the device's sum(y), sum(y^2) -- only for the float64 numpy, train == 1, <= 32 input datasets that
        took this path before the other forms did; every other form keeps the host path's np.var / np.mean of the train
        data, so that its fit stays bit-identical to the host path."""
        current = _process_kwargs(dict(_CLEAN_DEFAULTS), dict(kwargs_to_clean))
        raw = self._device_raw_inputs(inputs, current)
        if raw is None:
            return None
        numpy_f64 = isinstance(raw, np.ndarray) and raw.dtype == np.float64 and not hasattr(data, 'to_numpy') \
            and np.asarray(data).dtype == np.float64
        raw, data = self._format(raw, data, current['AutoTranspose'], current['SingleInstance'], current['bit'],
                                 _copy=False, _widen=False)
        n, mm = raw.shape
        if data.shape[0] != n:
            return None
        eng = _engine()
        ds = eng.upload_clean(raw, data, lambda column_minmax: self._normalize_bounds(
            mm, column_minmax, current['minmax'], current['pillow'], current['pillow_type']))
        trainlog, keep = self._shard_trainlog(current['train'], n)
        if trainlog is not None:
            ds = eng.rows_compact(ds, trainlog) if keep is None else \
                eng.rows_compact(ds, keep, int(np.count_nonzero(trainlog)))
            data = data[trainlog]
        self.__dict__['inputs'] = _DeviceInputs(ds)
        self.data = data
        self.trainlog = trainlog
        return ds, numpy_f64 and mm <= 32 and trainlog is None

    def _evaluate_clean(self, inputs, kwargs_to_clean, draws):
        """`self.clean(inputs, ...)` for `evaluate(inputs, clean=True)` on a model that already has `inputs` (so clean
        sets no attribute and draws no random number).  When the prediction will be reduced on the device
        (fokl_predict_summary) the raw rows are normalised in HBM with the bounds `_normalize_bounds` resolves (same
        warnings, same self.minmax update) and returned as _DeviceInputs; otherwise the formatted rows are normalised on
        the host as `clean` does."""
        current = _process_kwargs(dict(_CLEAN_DEFAULTS), dict(kwargs_to_clean))
        raw = self._device_raw_inputs(inputs, current) if 'inputs' in self.__dict__ and draws >= 2 else None
        if raw is None or _engine().world != 1:
            return self.clean(inputs, kwargs_from_other=kwargs_to_clean)
        raw, _ = self._format(raw, None, current['AutoTranspose'], current['SingleInstance'], current['bit'],
                              _copy=False, _widen=False)
        n, mm = raw.shape
        if n * draws < _PREDICT_SUMMARY_MIN_CELLS:
            return self._normalize(np.array(raw, dtype=np.float64), current['minmax'], current['pillow'],
                                   current['pillow_type'])
        ds = _engine().upload_clean(raw, np.zeros(n), lambda column_minmax: self._normalize_bounds(
            mm, column_minmax, current['minmax'], current['pillow'], current['pillow_type']))
        return _DeviceInputs(ds)

    # ------------------------------------------------------------------------------------------------
    # training hot path (FR:1202-1760)
    # ------------------------------------------------------------------------------------------------
    def fit(self, inputs=None, data=None, **kwargs):
        """Train the model: forward selection over BSS-ANOVA terms, each candidate scored by BIC and sampled by
        a Gibbs chain (FR:1202-1760).  Returns (betas, mtx, evs) as numpy arrays and sets self.betas,
        self.avg_betas, self.mtx, self.evs.

        Keywords: any hyper-parameter of the constructor, `clean` (default False), `ConsoleOutput`, and the
        keywords of `clean`.  `inputs` may also be a FoKL._engine.DeviceDataset (already normalised and resident
        in HBM), in which case no host-to-device copy happens."""
        from ._engine import DeviceDataset
        from ._selection import forward_select

        default_for_fit = {'ConsoleOutput': _str_to_bool(kwargs.get('ConsoleOutput', self.ConsoleOutput)),
                           'clean': _str_to_bool(kwargs.get('clean', False))}
        default_for_clean = dict(_CLEAN_DEFAULTS)
        expected = self.hypers + list(default_for_fit.keys()) + list(default_for_clean.keys())
        kwargs = _process_kwargs(expected, kwargs)
        if default_for_fit['clean'] is False:
            if any(kwarg in default_for_clean for kwarg in kwargs):
                warnings.warn("Keywords for automatic cleaning were defined but clean=False.")
            default_for_clean = {}

        kwargs_to_clean = {}
        for kwarg, value in kwargs.items():
            if kwarg in self.hypers:
                setattr(self, kwarg, _str_to_bool(value) if kwarg in ['gimmie', 'way3', 'aic'] else value)
            elif kwarg in default_for_clean:
                kwargs_to_clean[kwarg] = value
        self.ConsoleOutput = default_for_fit['ConsoleOutput']

        resident = isinstance(inputs, DeviceDataset)
        ds = None
        device_moments = resident      # b / btau defaults from the device's sum(y), sum(y^2) instead of host np.var
        if not resident and default_for_fit['clean'] is True and inputs is not None and data is not None:
            cleaned = self._clean_on_device(inputs, data, kwargs_to_clean)
            if cleaned is not None:
                ds, device_moments = cleaned
        if ds is not None:
            data = self.data
        elif not resident:
            failed = False
            if default_for_fit['clean'] is True:
                try:
                    if inputs is None:
                        inputs, _ = self.trainset()
                    if data is None:
                        _, data = self.trainset()
                except Exception:
                    failed = True
                if not failed:
                    self.clean(inputs, data, kwargs_from_other=kwargs_to_clean, _setattr=True)
            else:
                try:
                    if inputs is None:
                        inputs, _ = self.trainset()
                    if data is None:
                        _, data = self.trainset()
                except Exception:
                    warnings.warn("Keyword 'clean' was set to False but is required prior to or during 'fit'. "
                                  "Assuming 'clean' is True.", category=UserWarning)
                    if inputs is None or data is None:
                        failed = True
                    else:
                        self.clean(inputs, data, kwargs_from_other=kwargs_to_clean, _setattr=True)
            if failed:
                raise ValueError("'inputs' and/or 'data' were not provided so 'clean' could not be performed.")
            try:
                inputs, data = self.trainset()
            except Exception:
                warnings.warn("If not calling 'clean' prior to 'fit' or within the argument of 'fit', then this is the "
                              "likely source of any subsequent errors. To troubleshoot, simply include 'clean=True' "
                              "within the argument of 'fit'.", category=UserWarning)
                if np.ndim(data) != 2:
                    # upstream goes on with the raw arguments and fails on `dtd[0][0]` of a scalar data'data (FR:1374-1378)
                    raise IndexError("'data' must be an [n x 1] array when 'clean' was never performed on this model "
                                     "(invalid index to scalar variable upstream); include 'clean=True'.")
                inputs, data = self._format(inputs, data)
            self.inputs = inputs
            self.data = data
            if np.asarray(inputs).dtype != np.float64 or np.asarray(data).dtype != np.float64:
                raise NotImplementedError("the B200 build supports clean(bit=64) datasets only (float64)")

        # relats_in: only "exclude nothing" works upstream (np.zeros(a, b) at FR:1631 raises otherwise)
        relats_in = self.relats_in
        if np.logical_not(all([isinstance(index, int) for index in relats_in])):
            mrel = sum(np.logical_not(relats_in)).all() if len(relats_in) else 0
        else:
            mrel = sum(np.logical_not(relats_in))
        if mrel != 0:
            raise TypeError("relats_in with excluded terms is not supported (it raises upstream as well: "
                            "np.zeros(a, b) at FoKLRoutines.py:1631)")

        eng = _engine()
        eng.set_phis(self.phis, self.kernel)
        if resident:
            ds = inputs
        elif ds is None:
            ds = eng.upload(inputs, data)
        eng.begin_fit(ds)
        n = eng.n_global

        # b / btau defaults from the data moments (FR:1322-1348: np.var ddof 0, |mean|)
        a, b, atau, btau = self.a, self.b, self.atau, self.btau
        if btau is None or b is None:
            if device_moments or eng.world > 1:   # row shards: only the all-reduced moments describe the whole dataset
                data_mean = eng.sum_y / n
                sigmasq = eng.yty / n - data_mean ** 2
            else:
                sigmasq = np.var(data)
                data_mean = np.mean(data)
            if sigmasq == math.inf:
                warnings.warn("The dataset is too large such that 'sigmasq=inf' even as 64-bit. Consider training "
                              "on a smaller percentage of the dataset.", category=UserWarning)
            if b is None:
                b = sigmasq * (a + 1)
                self.b = b
            if btau is None:
                btau = (np.abs(data_mean) / sigmasq) * (atau + 1)
                self.btau = btau

        if self.update == True:  # noqa: E712   (FR:1365-1367)
            self.betas, self.mtx, self.evs = self._fitupdate_device(eng, ds)
            return self.betas, self.mtx, self.evs

        hy = dict(a=a, b=b, atau=atau, btau=btau, tolerance=self.tolerance, total_draws=self.burnin + self.draws,
                  gimmie=self.gimmie, way3=self.way3, threshav=self.threshav, threshstda=self.threshstda,
                  threshstdb=self.threshstdb, aic=self.aic, nested_chains=B200_CONFIG.get('nested_chains', True),
                  nested_min_p=B200_CONFIG.get('nested_min_p', 256),
                  kill_from_eig=B200_CONFIG.get('kill_from_eig', True))
        t0 = time.perf_counter()
        launches0 = eng.launch_count()
        work0 = dict(eng.work)
        out = forward_select(eng, hy, ds.m, len(self.phis), console=self.ConsoleOutput, rng=B200_CONFIG['rng'],
                             eager=B200_CONFIG['eager_chains'], pipeline=B200_CONFIG['pipeline'],
                             prefetch=B200_CONFIG.get('prefetch', False))
        eng.synchronize()
        LAST_FIT_INFO.clear()
        LAST_FIT_INFO.update(n_gibbs=out['n_gibbs'], n_batches=out['n_batches'], seconds=time.perf_counter() - t0,
                             launches=eng.launch_count() - launches0, n=n, m=ds.m, terms=out['mtx'].shape[0],
                             substages=len(out['evs']), **{k: v - work0[k] for k, v in eng.work.items()})

        betas = out['betas']
        self.betas = betas[-self.draws::, :]
        self.avg_betas = np.mean(self.betas, axis=0)
        self.mtx = out['mtx']
        self.evs = out['evs']
        return betas[-self.draws::, :], self.mtx, self.evs

    # ------------------------------------------------------------------------------------------------
    def clear(self, keep=None, clear=None, all=False):
        """Delete attributes except hyper-parameters and settings (FR:1762-1794)."""
        if all is not False:
            all = _str_to_bool(all)
        if all is False:
            attrs_to_keep = self.keep
            if isinstance(keep, (list, str)):
                attrs_to_keep += keep
                attrs_to_keep = list(np.unique(attrs_to_keep))
            if isinstance(clear, (list, str)):
                for attr in clear:
                    attrs_to_keep.remove(attr)
        else:
            attrs_to_keep = []
        for attr in list(vars(self).keys()):
            if attr not in attrs_to_keep:
                delattr(self, attr)

    def to_pyomo(self, xvars, yvars, m=None, xfix=None, yfix=None, truescale=True, std=True, draws=None):
        raise ImportError("Pyomo export (reference fokl_to_pyomo.py) is outside the B200 hot path; use the "
                          "reference package on the saved model (same pickle layout).")

    def bss_derivatives(self, **kwargs):
        """Gradient (or chosen first / second partial derivatives) of the fitted function with respect to the inputs
        (FR:594-805).  Keywords as upstream: inputs, kernel, d1, d2, draws, betas, phis, mtx, minmax, IndividualDraws,
        ReturnFullArray, ReturnBasis.  The derivative design matrices come from the derivative form of the basis
        kernel (fokl_basis_build_deriv) and the products with the draws from fokl_predict_draws, both on the device.
        Once N * draws >= _DERIV_SUMMARY_MIN_CELLS (draws > 1) the rows stream through fokl_deriv_summary in chunks
        instead (same bits), and device-resident default inputs (fit(clean=True)) are read in place."""
        default = {'inputs': None, 'kernel': self.kernel, 'd1': None, 'd2': None, 'draws': self.draws, 'betas': None,
                   'phis': None, 'mtx': self.mtx, 'minmax': self.minmax, 'IndividualDraws': False,
                   'ReturnFullArray': False, 'ReturnBasis': False}
        current = _process_kwargs(default, kwargs)
        for boolean in ['IndividualDraws', 'ReturnFullArray', 'ReturnBasis']:
            current[boolean] = _str_to_bool(current[boolean])
        resident = self._resident_inputs() if current['inputs'] is None else None
        inputs = resident if resident is not None else (self.inputs if current['inputs'] is None else current['inputs'])
        betas = self.betas if current['betas'] is None else current['betas']
        phis = self.phis if current['phis'] is None else current['phis']
        kernel, draws, span = current['kernel'], current['draws'], current['minmax']
        if isinstance(kernel, int):
            kernel = self.kernels[kernel]

        if isinstance(betas, list):
            betas = np.array(betas)
            if betas.ndim == 1:
                betas = betas[:, np.newaxis]
        mtx = current['mtx']
        if isinstance(mtx, int):
            mtx = np.array(mtx)[np.newaxis, np.newaxis]
        else:
            mtx = np.array(mtx)
            if mtx.ndim == 1:
                mtx = mtx[:, np.newaxis]
        if len(span) == 2 and not isinstance(span[0], (list, np.ndarray)):
            span = [span]
        if resident is not None and not (draws > 1 and resident.ds.n * draws >= _DERIV_SUMMARY_MIN_CELLS
                                         and resident.ds.m == np.shape(mtx)[1] and not current['ReturnBasis']):
            resident, inputs = None, self.inputs        # a path that reads the inputs on the host
        if resident is None:
            inputs = np.array(inputs)
            if inputs.ndim == 1:
                inputs = inputs[:, np.newaxis]
        if resident is not None:
            xr = resident.ds.x[:, :resident.ds.n]
            outside = bool(xr.max() > 1) or bool(xr.min() < 0)
            N = resident.ds.n
        else:
            outside = np.max(np.max(inputs)) > 1 or np.min(np.min(inputs)) < 0
            N = np.shape(inputs)[0]
        if outside:
            warnings.warn("Input 'inputs' should be normalized (0-1). Auto-normalization is in-development.",
                          category=UserWarning)
        B, M = np.shape(mtx)
        betas = np.asarray(betas, dtype=np.float64)
        if B != np.shape(betas)[1] - 1:
            betas = np.transpose(betas)
            if B != np.shape(betas)[1] - 1:
                raise ValueError(
                    "The shape of 'betas' does not align with the shape of 'mtx'. Transposing did not fix this.")

        def as_mask(di, second):
            """d1 / d2 keyword -> boolean row over the inputs (FR:686-725)."""
            if di is None:
                return np.zeros(M, dtype=bool) if second else np.ones(M, dtype=bool)
            if isinstance(di, str):
                return np.ones(M, dtype=bool) if _str_to_bool(di) else np.zeros(M, dtype=bool)
            if isinstance(di, list):
                if len(di) == 1:
                    di = di[0]
                elif len(di) == M:
                    return np.array(di) != 0
                else:
                    raise ValueError("Keyword input 'd1' and/or 'd2', if entered as a list, must be of equal length to "
                                     "the number of input variables.")
            if isinstance(di, bool):
                return np.ones(M, dtype=bool) * di
            if isinstance(di, int):
                row = np.zeros(M, dtype=bool)
                row[di] = True
                return row
            raise ValueError(
                "Keyword input 'd1' and/or 'd2' is limited to an integer indexing an input variable, or to a list "
                "of booleans corresponding to the input variables.")

        derv = [as_mask(current['d1'], False), as_mask(current['d2'], True)]
        if not any(derv[0]) and not any(derv[1]):
            warnings.warn("Function 'bss_derivatives' was called but no derivatives were requested.",
                          category=UserWarning)
            return

        cubic = kernel == self.kernels[0]
        if not cubic and kernel != self.kernels[1]:
            raise ValueError(f"The kernel {kernel} is not currently supported. Please select from the following: "
                             f"{self.kernels}.")
        L_phis = len(phis[0][0]) if cubic else 1
        divisors = np.ones((M, 3))
        for m in range(M):
            span_L = (span[m][1] - span[m][0]) / L_phis
            divisors[m] = [1, span_L, span_L ** 2]

        # one launch of the derivative basis kernel for every requested (input, derivative order) pair: the terms that
        # contain the input, with that input's factor differentiated (the other terms contribute exactly 0, FR:785-787)
        terms_i = np.asarray(mtx, dtype=np.int64)
        pairs, t_rows, d_rows = [], [], []
        for m in range(M):
            for di in (0, 1):
                if not derv[di][m]:
                    continue
                idx = np.nonzero(terms_i[:, m] != 0)[0]
                pairs.append((m, di, idx, sum(len(r) for r in t_rows) if t_rows else 0))
                if len(idx):
                    t_rows.append(terms_i[idx])
                    dr = np.zeros((len(idx), M), dtype=np.uint8)
                    dr[:, m] = di + 1
                    d_rows.append(dr)
        # the rows in chunks through fokl_deriv_summary, which also averages over the draws unless IndividualDraws
        streamed = draws > 1 and N * draws >= _DERIV_SUMMARY_MIN_CELLS
        # the mean over the draws on the device, without the N x M x 2 x draws array (same bits as np.mean on axis 3)
        mean_only = not current['IndividualDraws'] and draws > 1 and (
            streamed or N * draws >= _PREDICT_SUMMARY_MIN_CELLS)
        dy = np.zeros([N, M, 2, 1 if mean_only else draws])
        bsel = np.ascontiguousarray(betas[-draws:, :], dtype=np.float64)
        if t_rows and bsel.shape[0] != draws:
            # upstream fails here as well: `betas[-draws:, b + 1] * phi` does not broadcast into dy's draws axis (FR:789)
            raise ValueError(f"operands could not be broadcast together with shapes ({draws},) ({bsel.shape[0]},): "
                             f"'betas' holds fewer than draws={draws} rows.")
        if t_rows and streamed:
            eng_derivative_summary(_engine(), phis, kernel, inputs, np.concatenate(t_rows, axis=0),
                                   np.concatenate(d_rows, axis=0), divisors, pairs, bsel, dy)
        elif t_rows:
            eng_derivative_draws(_engine(), phis, kernel, inputs, np.concatenate(t_rows, axis=0),
                                 np.concatenate(d_rows, axis=0), divisors, pairs, bsel, dy, mean_only)

        if not current['IndividualDraws'] and draws > 1 and not mean_only:
            dy = np.mean(dy, axis=3)[:, :, :, np.newaxis]
        if not current['ReturnFullArray']:
            dy = np.concatenate([dy[:, :, 0, :], dy[:, :, 1, :]], axis=1)
            dy = dy[:, ~np.all(dy == 0, axis=0)]
        dy = np.squeeze(dy)

        if current['ReturnBasis']:
            # development option of the reference (FR:782-783): the plain basis value of the last factor its loops visit
            basis = np.zeros(N)
            m_last, di_last = max((m, di) for m, di, _, _ in pairs)
            if cubic:
                Xe, phind, _ = self._inputs_to_phind(np.asarray(inputs, dtype=np.float64), phis, kernel)
            else:
                Xe, phind = np.asarray(inputs, dtype=np.float64), None
            for b_ in range(B - 1, -1, -1):
                row = terms_i[b_]
                upto = M if row[m_last] else m_last        # the md loop stops at the differentiated input if absent
                visited = [md for md in range(upto) if row[md]]
                if visited:
                    md = visited[-1]
                    num = int(row[md]) - 1
                    for n_ in range(N):
                        c = [phis[num][k][int(phind[n_, md])] for k in range(4)] if cubic else phis[num]
                        basis[n_] = self.evaluate_basis(c, Xe[n_, md], kernel=kernel)
                    break
            return dy, basis
        return dy

    def fitupdate(self, inputs, data):
        """Update fit (FR:1850-2583) on already-normalised `inputs` / `data`: the first call (model not `built`) selects
        and samples a model from scratch with the evidence taken as the maximum log-likelihood over the draws; later
        calls use the previous draws (rows `burn` .. -1) as a Gaussian prior on the old coefficients and test further
        terms next to them.  Returns (betas, mtx, evs) with the reference's types (all burnin + draws rows of betas)."""
        eng = _engine()
        eng.set_phis(self.phis, self.kernel)
        inputs, data = self._format(inputs, data)
        ds = eng.upload(inputs, data)
        eng.begin_fit(ds)
        return self._fitupdate_device(eng, ds)

    def _fitupdate_device(self, eng, ds):
        from ._update import model_prior, update_select
        # relats_in: FR:2459-2478 only handles "exclude nothing" (the same np.zeros(a, b) defect as FR:1631)
        if len(self.relats_in) != 0:
            raise TypeError("relats_in with excluded terms is not supported (it raises upstream as well)")
        prior = model_prior(self.betas, self.burn) if self.built else None             # FR:1939-1948
        hy = dict(a=self.a, b=self.b, atau=self.atau, btau=self.btau, tolerance=self.tolerance,
                  total_draws=self.burnin + self.draws, gimmie=self.gimmie, aic=self.aic, sigsqd0=self.sigsqd0)
        t0 = time.perf_counter()
        launches0 = eng.launch_count()
        out = update_select(eng, hy, ds.m, len(self.phis), prior=prior, console=self.ConsoleOutput,
                            rng=B200_CONFIG['rng'])
        eng.synchronize()
        if out['built']:
            self.built = True                                                            # FR:2565
        LAST_FIT_INFO.clear()
        LAST_FIT_INFO.update(n_gibbs=out['n_gibbs'], n_batches=out['n_gibbs'], seconds=time.perf_counter() - t0,
                             launches=eng.launch_count() - launches0, n=eng.n_global, m=ds.m,
                             terms=out['mtx'].shape[0], substages=len(out['evs']))
        return out['betas'], out['mtx'], out['evs']

    def save(self, filename=None, directory=None):
        """Pickle the model to '<filename>.fokl'; returns the path (FR:1807-1846)."""
        if filename is None:
            t = time.gmtime()
            filename = "model_" + str(t[0]) + "".join("%02d" % t[i] for i in range(1, 6)) + ".fokl"
        elif filename[-5::] != ".fokl":
            filename = filename + ".fokl"
        filepath = os.path.join(directory, filename) if directory is not None else filename
        with open(filepath, "wb") as file:
            pickle.dump(self, file)
        time.sleep(1)  # so that the next saved model is guaranteed a different default filename
        return filepath


def eng_derivative_draws(eng, phis, kernel, inputs, term_rows, deriv_rows, divisors, pairs, bsel, dy, mean_only=False):
    """dy[:, m, di, :] = (derivative design columns of the terms idx that contain input m) @ bsel[:, idx + 1]' for every
    (m, di, idx, off) of `pairs`, on the device: one fokl_basis_build_deriv over all rows of term_rows / deriv_rows (the
    columns of a pair start at row `off`), one fokl_predict_draws per pair (FR:727-795).  mean_only: dy[:, m, di, 0] =
    the mean over the draws instead, from fokl_predict_summary."""
    import torch
    N, M, draws = np.shape(inputs)[0], np.shape(term_rows)[1], bsel.shape[0]
    eng.set_phis(phis, kernel)
    x64 = np.ascontiguousarray(inputs, dtype=np.float64)
    ds = eng.upload(x64, np.zeros(N))
    t16 = np.ascontiguousarray(term_rows, dtype=np.int16)
    d8 = np.ascontiguousarray(deriv_rows, dtype=np.uint8)
    dv = np.ascontiguousarray(divisors, dtype=np.float64)
    X = torch.empty((t16.shape[0], ds.ldx), dtype=torch.float64, device=eng.device)
    eng._ck(eng.lib.fokl_basis_build_deriv(eng.ctx, eng.kernel_id, ds.x.data_ptr(), N, ds.ldx, M,
                                           t16.ctypes.data, d8.ctypes.data, dv.ctypes.data, t16.shape[0],
                                           X.data_ptr(), ds.ldx))
    eng.synchronize()       # surfaces the out-of-range flag (inputs outside [0, 1]) as ValueError
    for m, di, idx, off in pairs:
        if not len(idx):
            continue
        b = torch.from_numpy(np.ascontiguousarray(bsel[:, idx + 1])).to(eng.device)
        if mean_only:
            mean = torch.empty((N,), dtype=torch.float64, device=eng.device)
            eng._ck(eng.lib.fokl_predict_summary(eng.ctx, X[off].data_ptr(), ds.ldx, N, len(idx), b.data_ptr(), draws,
                                                 -1, -1, mean.data_ptr(), None, None))
            dy[:, m, di, 0] = mean.cpu().numpy()
            continue
        out = torch.empty((N, draws), dtype=torch.float64, device=eng.device)
        eng._ck(eng.lib.fokl_predict_draws(eng.ctx, X[off].data_ptr(), ds.ldx, N, len(idx), b.data_ptr(), draws,
                                           out.data_ptr()))
        dy[:, m, di, :] = out.cpu().numpy()


def eng_derivative_summary(eng, phis, kernel, inputs, term_rows, deriv_rows, divisors, pairs, bsel, dy):
    """dy as eng_derivative_draws fills it -- the same bits -- with the rows streamed through fokl_deriv_summary: per
    chunk one call builds the chunk's derivative columns and forms every pair's values (dy of shape (N, M, 2, draws)) or
    their mean over the draws (dy of shape (N, M, 2, 1)), in dy's layout on the device; one copy per chunk brings the
    slice dy[r0:r0 + rows] back.  inputs is a host array or device-resident _DeviceInputs.  Device memory: the inputs,
    the betas blocks, one chunk of dy (at most _DERIV_CHUNK_BYTES) and the library's chunk workspace."""
    import torch
    N, M, _, depth = dy.shape
    draws = bsel.shape[0]
    eng.set_phis(phis, kernel)
    if isinstance(inputs, _DeviceInputs):
        ds = inputs.ds
    else:
        ds = eng.upload(np.ascontiguousarray(inputs, dtype=np.float64), np.zeros(N))
    t16 = np.ascontiguousarray(term_rows, dtype=np.int16)
    d8 = np.ascontiguousarray(deriv_rows, dtype=np.uint8)
    dv = np.ascontiguousarray(divisors, dtype=np.float64)
    table, blocks, boff = [], [], 0
    for m, di, idx, off in pairs:
        table.append((off, len(idx), boff, m, di))
        blocks.append(np.ascontiguousarray(bsel[:, idx + 1]).ravel())
        boff += draws * len(idx)
    table = np.ascontiguousarray(table, dtype=np.int64)
    b = torch.from_numpy(np.concatenate(blocks)).to(eng.device)
    per_row = M * 2 * depth
    rows = max(16, min(_PREDICT_CHUNK_ROWS, _DERIV_CHUNK_BYTES // (8 * per_row)) // 16 * 16)
    rows = min(rows, (N + 15) // 16 * 16)
    out = torch.empty((rows * per_row,), dtype=torch.float64, device=eng.device)
    cuda = out.device.type == 'cuda'
    # two pinned buffers: the host copies chunk k - 1 into dy while the device works on chunk k
    host = [torch.empty((rows * per_row,), dtype=torch.float64, pin_memory=cuda) for _ in range(2)]
    pending = [None, None]
    flat = dy.reshape(N, per_row)

    def drain(s):
        if pending[s] is not None:
            r0, nr, done = pending[s]
            if done is not None:
                done.synchronize()
            flat[r0:r0 + nr] = host[s][:nr * per_row].numpy().reshape(nr, per_row)
            pending[s] = None

    for k, r0 in enumerate(range(0, N, rows)):
        nr, s = min(rows, N - r0), k % 2
        drain(s)
        eng._ck(eng.lib.fokl_deriv_summary(eng.ctx, eng.kernel_id, ds.x.data_ptr(), ds.ldx, M, r0, nr,
                                           t16.ctypes.data, d8.ctypes.data, dv.ctypes.data, t16.shape[0],
                                           table.ctypes.data, len(table), b.data_ptr(), draws,
                                           1 if depth == 1 else 0, out.data_ptr()))
        host[s][:nr * per_row].copy_(out[:nr * per_row], non_blocking=cuda)
        done = None
        if cuda:
            done = torch.cuda.Event()
            done.record()
        pending[s] = (r0, nr, done)
    eng.synchronize()       # surfaces the out-of-range flag (inputs outside [0, 1]) as ValueError
    drain(0)
    drain(1)


def eng_predict(eng, phis, kernel, normputs, terms, betas_sel):
    """modells[i, d] = X(normputs)[i, :] @ betas_sel[d, :] on the device (FR:950-968)."""
    import torch
    from . import _lib
    eng.set_phis(phis, kernel)
    ds = eng.upload(normputs, np.zeros(normputs.shape[0]))
    n, p = ds.n, terms.shape[0] + 1
    X = torch.empty((p, ds.ldx), dtype=torch.float64, device=eng.device)
    eng._ck(eng.lib.fokl_fill_ones(eng.ctx, X.data_ptr(), n))
    if p > 1:
        t16 = np.ascontiguousarray(terms, dtype=np.int16)
        eng._ck(eng.lib.fokl_basis_build(eng.ctx, eng.kernel_id, ds.x.data_ptr(), n, ds.ldx, ds.m, t16.ctypes.data,
                                         p - 1, X[1].data_ptr(), ds.ldx))
    b = torch.from_numpy(np.ascontiguousarray(betas_sel, dtype=np.float64)).to(eng.device)
    out = torch.empty((n, b.shape[0]), dtype=torch.float64, device=eng.device)
    eng._ck(eng.lib.fokl_predict_draws(eng.ctx, X.data_ptr(), ds.ldx, n, p, b.data_ptr(), b.shape[0], out.data_ptr()))
    eng.synchronize()
    return out.cpu().numpy()


def eng_predict_summary(eng, phis, kernel, normputs_or_ds, terms, betas_sel, ranks):
    """Per row i of X(normputs) @ betas_sel': (mean over the draws, value at ascending rank ranks[0], at ranks[1]), the
    bits of np.mean(modells, 1) and np.sort(modells, 1)[:, k] (only the sign of a zero may differ); the last two are
    None when `ranks` is None.  normputs_or_ds is a host array or device-resident _DeviceInputs.  The design matrix is
    built _PREDICT_CHUNK_ROWS rows at a time and the product is reduced on the device, so device memory does not grow
    with N beyond the inputs and the three output columns."""
    import torch
    eng.set_phis(phis, kernel)
    if isinstance(normputs_or_ds, _DeviceInputs):
        ds = normputs_or_ds.ds
    else:
        ds = eng.upload(normputs_or_ds, np.zeros(normputs_or_ds.shape[0]))
    n, p = ds.n, terms.shape[0] + 1
    b = torch.from_numpy(np.ascontiguousarray(betas_sel, dtype=np.float64)).to(eng.device)
    rank_lo, rank_hi = ranks if ranks is not None else (-1, -1)
    out = torch.empty((1 if ranks is None else 3, n), dtype=torch.float64, device=eng.device)
    rows = min(_PREDICT_CHUNK_ROWS, (n + 15) // 16 * 16)
    X = torch.empty((p, rows), dtype=torch.float64, device=eng.device)
    eng._ck(eng.lib.fokl_fill_ones(eng.ctx, X.data_ptr(), rows))
    t16 = np.ascontiguousarray(terms, dtype=np.int16)
    for r0 in range(0, n, rows):
        nr = min(rows, n - r0)
        if p > 1:
            eng._ck(eng.lib.fokl_basis_build(eng.ctx, eng.kernel_id, ds.x.data_ptr() + 8 * r0, nr, ds.ldx, ds.m,
                                             t16.ctypes.data, p - 1, X[1].data_ptr(), rows))
        lo_ptr, hi_ptr = (None, None) if ranks is None else (out[1].data_ptr() + 8 * r0, out[2].data_ptr() + 8 * r0)
        eng._ck(eng.lib.fokl_predict_summary(eng.ctx, X.data_ptr(), rows, nr, p, b.data_ptr(), b.shape[0], rank_lo,
                                             rank_hi, out[0].data_ptr() + 8 * r0, lo_ptr, hi_ptr))
    eng.synchronize()
    res = out.cpu().numpy()
    if ranks is None:
        return res[0], None, None
    return res[0], res[1], res[2]
