"""Derivatives at training-set scale: bss_derivatives(d1 and d2 on every input) on a cfg4-shaped model (N = 1e7,
8 inputs, 52 cubic 3-way terms, 1000 draws) through fokl_deriv_summary, end to end, and the default coverage3() on
the same model with an (N, 1) data column; then the existing path (eng_derivative_draws) alternated with the streamed
one at --old-n rows, outputs compared.  The card's name and power limit are read in the same run.  Prints one JSON
line; writes nothing into the tree.

    python tools/deriv_bench.py [--n 10000000] [--old-n 1000000] [--reps 3]
"""
import argparse
import json
import os
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'fokl-gpy_b200'))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

from predict_bench import card, model_of  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--n', type=int, default=10_000_000)
    ap.add_argument('--old-n', type=int, default=1_000_000)
    ap.add_argument('--reps', type=int, default=3)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('deriv_bench needs a CUDA device')
    from FoKL import FoKLRoutines as FR
    import bench
    phis = bench.load_phis(argparse.Namespace(workload='cfg4'))
    model = model_of(FR, phis)
    rng = np.random.default_rng(1)
    x = rng.random((a.n, 8))
    model.inputs, model.data = x, rng.standard_normal((a.n, 1))
    terms_i = np.asarray(model.mtx, dtype=np.int64)
    cols = int(2 * np.count_nonzero(terms_i))            # derivative columns of d1 and d2 on every input
    res = {'card': card(), 'n': a.n, 'terms': terms_i.shape[0], 'draws': model.draws, 'deriv_columns': cols}
    warnings.simplefilter('ignore')
    kw = dict(d1=True, d2=True)

    model.bss_derivatives(inputs=x[:200_000], **kw)                # warm-up: module load, scratch
    times = []
    for _ in range(a.reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        dy = model.bss_derivatives(**kw)
        times.append(time.perf_counter() - t0)
    res['bss_derivatives_s'] = times
    res['bss_derivatives_tflops_end_to_end'] = 2.0 * a.n * cols * model.draws / min(times) / 1e12
    np.random.seed(0)
    times = []
    for _ in range(a.reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _, _, rmse = model.coverage3()
        times.append(time.perf_counter() - t0)
    res['coverage3_s'] = times
    res['coverage3_rmse_finite'] = bool(np.isfinite(rmse))

    # the existing path against the streamed one on the same rows, alternating
    xo = x[:a.old_n]
    old_t, new_t, equal = [], [], True
    for _ in range(2):
        for path in ('old', 'new'):
            FR._DERIV_SUMMARY_MIN_CELLS = (1 << 62) if path == 'old' else 0
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = model.bss_derivatives(inputs=xo, **kw)
            (old_t if path == 'old' else new_t).append(time.perf_counter() - t0)
            if path == 'old':
                ref = r
            else:
                equal = equal and bool(np.array_equal(r.view(np.uint64), ref.view(np.uint64)))
    FR._DERIV_SUMMARY_MIN_CELLS = 1 << 24
    res.update(old_n=a.old_n, old_path_s=old_t, new_path_s=new_t, old_new_equal=equal,
               full_n_sample_equal=bool(np.array_equal(dy[:a.old_n].view(np.uint64), ref.view(np.uint64))))
    print(json.dumps(res))


if __name__ == '__main__':
    main()
