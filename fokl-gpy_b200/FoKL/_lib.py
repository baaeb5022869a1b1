"""ctypes binding of the C ABI declared in include/fokl_b200.h.

There is deliberately NO fallback: if libfokl_b200.so is missing or fails to load, every entry point
of the hot path raises.  Build it with `python __graft_entry__.py` (or `build_library()` below)."""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(_HERE), 'csrc')
SO_PATH = os.path.join(CSRC, 'libfokl_b200.so')
if os.environ.get('FOKL_B200_LIB'):        # kernel-variant experiments (tools/): another build of the same sources
    SO_PATH = os.path.abspath(os.environ['FOKL_B200_LIB'])
SOURCES = ['ctx.cu', 'basis.cu', 'gram.cu', 'candidates.cu', 'nested.cu', 'update.cu', 'predict.cu', 'trainlog.cu']
HEADERS = ['fokl_ctx.cuh', 'fokl_math.cuh', 'cand_math.cuh', 'gram_plan.h', 'eigbig.cuh', 'killbig.cuh', 'update_math.cuh', 'predict_math.cuh', 'trainlog_math.cuh']

ABI_VERSION = 4
KERNEL_CUBIC, KERNEL_BERNOULLI = 0, 1
RNG_NONE, RNG_INJECTED, RNG_PHILOX = 0, 1, 2
ERANGE = -4
GRAM_CROSS_ONLY = 1

_vp = ctypes.c_void_p
_i64 = ctypes.c_int64
_i32 = ctypes.c_int
_u64 = ctypes.c_uint64


class Hypers(ctypes.Structure):
    """struct fokl_hypers (include/fokl_b200.h)."""
    _fields_ = [('a', ctypes.c_double), ('b', ctypes.c_double), ('atau', ctypes.c_double),
                ('btau', ctypes.c_double), ('sigsqd0', ctypes.c_double), ('tausqd0', ctypes.c_double),
                ('yty', ctypes.c_double), ('sum_y', ctypes.c_double), ('n', ctypes.c_int64),
                ('draws', ctypes.c_int32), ('stat_from0', ctypes.c_int32), ('stat_from1', ctypes.c_int32),
                ('reserved', ctypes.c_int32)]


class KillParams(ctypes.Structure):
    """struct fokl_kill_params (include/fokl_b200.h)."""
    _fields_ = [('threshav', ctypes.c_double), ('threshstda', ctypes.c_double), ('threshstdb', ctypes.c_double),
                ('icpt', ctypes.c_double), ('evmin', ctypes.c_double), ('aic_adj', ctypes.c_double),
                ('start', ctypes.c_int32), ('reserved', ctypes.c_int32), ('lamb', ctypes.c_void_p),
                ('Qt', ctypes.c_void_p)]


class UpdateModel(ctypes.Structure):
    """struct fokl_update_model (include/fokl_b200.h)."""
    _fields_ = [('mode', ctypes.c_int32), ('po', ctypes.c_int32), ('pn', ctypes.c_int32), ('draws', ctypes.c_int32),
                ('a_star', ctypes.c_double), ('atau_star', ctypes.c_double), ('b', ctypes.c_double),
                ('btau', ctypes.c_double), ('sigsqd0', ctypes.c_double), ('yty', ctypes.c_double),
                ('squerr', ctypes.c_double), ('n', ctypes.c_int64)]


PROTOTYPES = {
    'fokl_abi_version': (_i32, []),
    'fokl_ctx_create': (_i32, [ctypes.POINTER(_vp), _i32, _vp]),
    'fokl_ctx_destroy': (_i32, [_vp]),
    'fokl_last_error': (ctypes.c_char_p, [_vp]),
    'fokl_ctx_synchronize': (_i32, [_vp]),
    'fokl_launch_count': (_i64, [_vp]),
    'fokl_set_phis_cubic': (_i32, [_vp, _vp, _i32, _i32]),
    'fokl_set_phis_bernoulli': (_i32, [_vp, _vp, _i32, _i32]),
    'fokl_basis_build': (_i32, [_vp, _i32, _vp, _i64, _i64, _i32, _vp, _i32, _vp, _i64]),
    'fokl_basis_build_deriv': (_i32, [_vp, _i32, _vp, _i64, _i64, _i32, _vp, _vp, _vp, _i32, _vp, _i64]),
    'fokl_ctx_set_sm_budget': (_i32, [_vp, _i32]),
    'fokl_ctx_set_high_priority': (_i32, [_vp, _i32]),
    'fokl_ctx_wait_eig': (_i32, [_vp, _vp]),
    'fokl_fill_ones': (_i32, [_vp, _vp, _i64]),
    'fokl_gram_update': (_i32, [_vp, _vp, _i64, _i64, _i32, _i32, _vp, _vp]),
    'fokl_gram_update_ex': (_i32, [_vp, _vp, _i64, _i64, _i32, _i32, _i32, _i32, _vp, _vp]),
    'fokl_gram_last_config': (_i32, [_vp, _vp]),
    'fokl_y_moments': (_i32, [_vp, _vp, _i64, _vp]),
    'fokl_gram_scatter': (_i32, [_vp, _vp, _i32, _i32, _vp, _i64, _vp]),
    'fokl_gram_compact': (_i32, [_vp, _vp, _i64, _vp, _vp, _i32, _vp, _i64, _vp]),
    'fokl_columns_compact': (_i32, [_vp, _vp, _i64, _i64, _vp, _i32]),
    'fokl_candidates_eval': (_i32, [_vp, _vp, _i64, _vp, _vp, _vp, _i32, ctypes.POINTER(Hypers), _vp, _i32, _u64,
                                    _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'fokl_secular_step': (_i32, [_vp, _vp, _vp, _i32, _vp, _vp, _i64, _vp, _vp]),
    'fokl_chain_icpt': (_i32, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, ctypes.POINTER(Hypers), _u64, _vp, _vp]),
    'fokl_update_chain': (_i32, [_vp, ctypes.POINTER(UpdateModel), _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32,
                                 _u64, _u64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'fokl_kill_scores': (_i32, [_vp, _vp, _i64, _vp, _vp, _i32, _vp, _i32, ctypes.POINTER(Hypers), _vp, _vp]),
    'fokl_kill_loop': (_i32, [_vp, _vp, _i64, _vp, _vp, _i32, _vp, _vp, _vp, _i32, ctypes.POINTER(Hypers),
                              ctypes.POINTER(KillParams), _vp, _vp]),
    'fokl_residual_moments': (_i32, [_vp, _vp, _i64, _i64, _i32, _vp, _vp, _vp, _vp]),
    'fokl_predict_draws': (_i32, [_vp, _vp, _i64, _i64, _i32, _vp, _i32, _vp]),
    'fokl_predict_summary': (_i32, [_vp, _vp, _i64, _i64, _i32, _vp, _i32, _i32, _i32, _vp, _vp, _vp]),
    'fokl_deriv_summary': (_i32, [_vp, _i32, _vp, _i64, _i32, _i64, _i64, _vp, _vp, _vp, _i32, _vp, _i32, _vp, _i32,
                                  _i32, _vp]),
    'fokl_column_minmax': (_i32, [_vp, _vp, _i64, _i64, _i32, _vp]),
    'fokl_normalize': (_i32, [_vp, _vp, _i64, _i64, _i32, _vp]),
    'fokl_rows_compact': (_i32, [_vp, _vp, _vp, _i64, _i64, _i32, _vp, _vp, _vp, _i64, ctypes.POINTER(_i64)]),
    'fokl_trainlog': (_i32, [_vp, _vp, _i32, _i64, _i64, _vp, _vp, ctypes.POINTER(_i32), ctypes.POINTER(_i64)]),
}

_lib = None


class FoklLibraryError(RuntimeError):
    pass


def nvcc_command(out=SO_PATH, extra=()):
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    return ['nvcc', '-O3', '-std=c++17', '-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo',
            '-Xcompiler', '-fPIC', '-shared', '-o', out] + list(extra) + srcs


def needs_build():
    if not os.path.exists(SO_PATH):
        return True
    t = os.path.getmtime(SO_PATH)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS]
    deps.append(os.path.join(os.path.dirname(os.path.dirname(_HERE)), 'include', 'fokl_b200.h'))
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build_library(force=False, verbose=False):
    """Compile csrc/*.cu for sm_100a into csrc/libfokl_b200.so (nvcc cross-compiles without a GPU)."""
    if not force and not needs_build():
        return SO_PATH
    cmd = nvcc_command()
    if verbose:
        print(' '.join(cmd))
    subprocess.check_call(cmd)
    return SO_PATH


def load():
    """Load libfokl_b200.so and bind every symbol of include/fokl_b200.h.  Raises if unavailable."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise FoklLibraryError(
            "libfokl_b200.so not found at %s: the CUDA extension is required (no CPU fallback). "
            "Build it with `python __graft_entry__.py` or FoKL._lib.build_library()." % SO_PATH)
    try:
        lib = ctypes.CDLL(SO_PATH)
    except OSError as exc:
        raise FoklLibraryError("failed to load %s: %s" % (SO_PATH, exc))
    for name, (res, args) in PROTOTYPES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            raise FoklLibraryError("libfokl_b200.so does not export %s (stale build?)" % name)
        fn.restype = res
        fn.argtypes = args
    if lib.fokl_abi_version() != ABI_VERSION:
        raise FoklLibraryError("libfokl_b200.so ABI version mismatch")
    _lib = lib
    return lib
