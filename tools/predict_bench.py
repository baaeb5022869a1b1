"""Prediction at training-set scale: evaluate(ReturnBounds=1) on a cfg4-shaped model (N = 1e7, 8 inputs, 52 cubic
3-way terms, 1000 draws) through fokl_predict_summary, its two kernels, cuBLAS DGEMM on the same product shape, and the
old path (fokl_predict_draws + numpy on the host) at the largest N where it fits, alternated with the new path on the
same rows.  Prints one JSON line; writes nothing into the tree.

    python tools/predict_bench.py [--n 10000000] [--old-n 1000000] [--reps 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'fokl-gpy_b200'))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm',
                              '--format=csv,noheader'], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as exc:            # the measurement is still valid; say what is missing
        out = 'nvidia-smi unavailable: %s' % exc
    return out


def model_of(FR, phis, n_terms=52, draws=1000, seed=44):
    rng = np.random.default_rng(seed)
    mtx = np.zeros((n_terms, 8))
    for t in range(n_terms):
        k = 1 + t % 3
        mtx[t, rng.choice(8, k, replace=False)] = rng.integers(1, 6, k)
    model = FR.FoKL(phis=phis, draws=draws, UserWarnings=False)
    model.mtx, model.minmax = mtx, [[0.0, 1.0]] * 8
    model.betas = rng.standard_normal((draws, n_terms + 1)) * np.geomspace(1, 1e-3, n_terms + 1)
    return model


def same(a, b):
    return bool(np.array_equal(a, b, equal_nan=True))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--n', type=int, default=10_000_000)
    ap.add_argument('--old-n', type=int, default=1_000_000)
    ap.add_argument('--reps', type=int, default=3)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('predict_bench needs a CUDA device')
    from FoKL import FoKLRoutines as FR
    import bench
    phis = bench.load_phis(argparse.Namespace(workload='cfg4'))
    dev = torch.device('cuda', 0)
    eng = FR._engine()
    model = model_of(FR, phis)
    draws, p = model.draws, model.mtx.shape[0] + 1
    rng = np.random.default_rng(1)
    x = rng.random((a.n, 8))
    res = {'card': card(), 'n': a.n, 'p': p, 'draws': draws}
    warnings.simplefilter('ignore')

    # end to end, default threshold (host arrays in, host arrays out; includes the 640 MB upload)
    np.random.seed(0)
    model.evaluate(x[:200_000], ReturnBounds=1)                  # warm-up: module load, scratch, setnos
    times = []
    for _ in range(a.reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        mean, bounds = model.evaluate(x, ReturnBounds=1)
        times.append(time.perf_counter() - t0)
    res['evaluate_s'] = times
    flops = 2.0 * a.n * p * draws
    res['evaluate_tflops_end_to_end'] = flops / min(times) / 1e12

    # the two kernels: fokl_predict_summary on one 65536-row design-matrix chunk, CUDA events over many launches
    rows = FR._PREDICT_CHUNK_ROWS
    ds = eng.upload(x[:rows], np.zeros(rows))
    X = torch.empty((p, rows), dtype=torch.float64, device=dev)
    eng._ck(eng.lib.fokl_fill_ones(eng.ctx, X.data_ptr(), rows))
    t16 = np.ascontiguousarray(model.mtx, dtype=np.int16)
    eng._ck(eng.lib.fokl_basis_build(eng.ctx, eng.kernel_id, ds.x.data_ptr(), rows, ds.ldx, ds.m, t16.ctypes.data,
                                     p - 1, X[1].data_ptr(), rows))
    b = torch.from_numpy(np.ascontiguousarray(model.betas[model.setnos[:draws]])).to(dev)
    out = torch.empty((3, rows), dtype=torch.float64, device=dev)
    cut = int(np.floor(draws * 0.025) + 1)

    def call(rlo, rhi):
        eng._ck(eng.lib.fokl_predict_summary(eng.ctx, X.data_ptr(), rows, rows, p, b.data_ptr(), draws, rlo, rhi,
                                             out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr()))

    def timed(fn, k=20):
        fn()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(k):
            fn()
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e) / k * 1e-3

    t_call = timed(lambda: call(cut, draws - cut))
    t_mean = timed(lambda: call(-1, -1))
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(10):
            call(cut, draws - cut)
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.key_averages():
        for tag in ('predict_tile_kernel', 'predict_summary_kernel'):
            if tag in ev.key:
                kern[tag] = getattr(ev, 'device_time_total', getattr(ev, 'cuda_time_total', 0.0)) / 10 * 1e-6
    chunk_flops = 2.0 * rows * p * draws
    res['chunk_rows'] = rows
    res['summary_call_s'] = t_call
    res['summary_call_mean_only_s'] = t_mean
    res['product_kernel_s'] = kern.get('predict_tile_kernel')
    res['summary_kernel_s'] = kern.get('predict_summary_kernel')
    if kern.get('predict_tile_kernel'):
        res['product_kernel_tflops'] = chunk_flops / kern['predict_tile_kernel'] / 1e12
    res['summary_call_tflops'] = chunk_flops / t_call / 1e12
    A = X[:, :rows].t().contiguous()
    Bt = b.t().contiguous()
    t_gemm = timed(lambda: torch.matmul(A, Bt))
    res['cublas_dgemm_same_shape_s'] = t_gemm
    res['cublas_dgemm_same_shape_tflops'] = chunk_flops / t_gemm / 1e12
    del A, Bt, X, out, ds

    # old path against the new one on the same rows, alternating
    xo = x[:a.old_n]
    old_t, new_t, equal = [], [], True
    for _ in range(2):
        for path in ('old', 'new'):
            FR._PREDICT_SUMMARY_MIN_CELLS = (1 << 62) if path == 'old' else 0
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = model.evaluate(xo, ReturnBounds=1)
            (old_t if path == 'old' else new_t).append(time.perf_counter() - t0)
            if path == 'old':
                ref = r
            else:
                equal = equal and same(r[0], ref[0]) and same(r[1], ref[1])
    FR._PREDICT_SUMMARY_MIN_CELLS = 1 << 24
    res.update(old_n=a.old_n, old_path_s=old_t, new_path_s=new_t, old_new_equal=equal,
               full_n_sample_equal=same(mean[:a.old_n], ref[0]) and same(bounds[:a.old_n], ref[1]))
    print(json.dumps(res))


if __name__ == '__main__':
    main()
