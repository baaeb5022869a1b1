"""`clean` on the host against `clean` in HBM, end to end, at N = 10^7 rows and 8 inputs on one GPU.

For each form that reaches the device path (pandas frame, float32 array, train split, more than 32 inputs,
evaluate(raw_inputs, clean=True, ReturnBounds=1)) the host path (forced by raising _CLEAN_ON_DEVICE_MIN_CELLS) and the
device path run alternately in one process on the same seeded data, and their outputs are compared bit for bit.  The
more-than-32-inputs form runs at 40 inputs and N = 2 * 10^6 (the same 8 * 10^7 cells).  fokl_rows_compact is timed
with CUDA events against the HBM bandwidth of a device-to-device copy measured in the same run; generate_trainlog, which
stays on the host, is timed on its own.  Prints one JSON object (and writes it to --out)."""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, 'fokl-gpy_b200'), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else 'unknown'


def same(a, b):
    a, b = np.ascontiguousarray(np.atleast_1d(a)), np.ascontiguousarray(np.atleast_1d(b))
    return bool(a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--n', type=int, default=10 ** 7)
    ap.add_argument('--reps', type=int, default=2)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    import pandas as pd
    import torch
    import bench_data
    from FoKL import FoKLRoutines as FR
    from FoKL import getKernels
    assert torch.cuda.is_available(), 'clean_bench needs a GPU'
    phis = getKernels.sp500()
    n = a.n
    x, y = bench_data.make_rows('cfg4', 0, n, n_total=n)
    raw = x * np.arange(1.0, 9.0) - 2.0
    del x
    wide_n = n // 5
    rng = np.random.default_rng(3)
    raw40 = rng.random((wide_n, 40)) * 5.0 - 1.0
    y40 = np.sin(raw40[:, 0]) + raw40[:, 1] * raw40[:, 39] + 0.05 * rng.standard_normal(wide_n)
    hy = dict(phis=phis, way3=True, UserWarnings=False, ConsoleOutput=False)
    forms = {
        'pandas_f64': lambda: (pd.DataFrame(raw), pd.Series(y), {}),
        'numpy_f32': lambda: (raw.astype(np.float32), y.astype(np.float32), {}),
        'split_0.8': lambda: (raw, y, dict(train=0.8)),
        'inputs_40': lambda: (raw40, y40, {}),
    }

    def fit_once(form, cells):
        xi, yi, kw = forms[form]()
        FR._CLEAN_ON_DEVICE_MIN_CELLS = cells
        model = FR.FoKL(**hy) if form != 'inputs_40' else FR.FoKL(phis=phis, UserWarnings=False, ConsoleOutput=False)
        np.random.seed(5)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            out = model.fit(xi, yi, clean=True, **kw)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, model, out

    res = dict(card=card(), n=n, m=8, wide=dict(n=wide_n, m=40), forms={})
    for form in forms:
        t = {'host': [], 'device': []}
        keep = {}
        for r in range(a.reps):
            for path, cells in (('host', 1 << 62), ('device', 0)):
                dt, model, out = fit_once(form, cells)
                t[path].append(dt)
                if r == 0:
                    keep[path] = (out, model.inputs, model.data, model.minmax, model.trainlog, model.b, model.btau)
        h, d = keep['host'], keep['device']
        ident = all(same(u, v) for u, v in zip(h[0], d[0])) and same(h[1], d[1]) and same(h[2], d[2]) \
            and h[3] == d[3] and (h[4] is None and d[4] is None or same(h[4], d[4])) and same(h[5], d[5]) \
            and same(h[6], d[6])
        res['forms'][form] = dict(host_s=t['host'], device_s=t['device'], identical=bool(ident))
        print(form, res['forms'][form], flush=True)

    # evaluate(raw, clean=True, ReturnBounds=1) with a model fitted on the device path
    FR._CLEAN_ON_DEVICE_MIN_CELLS = 0
    model = FR.FoKL(**hy)
    np.random.seed(5)
    model.fit(raw, y, clean=True)
    t = {'host': [], 'device': []}
    outs = {}
    for r in range(a.reps):
        for path, cells in (('host', 1 << 62), ('device', 0)):
            FR._CLEAN_ON_DEVICE_MIN_CELLS = cells
            model.setnos = None
            np.random.seed(9)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            outs[path] = model.evaluate(raw, clean=True, ReturnBounds=1)
            torch.cuda.synchronize()
            t[path].append(time.perf_counter() - t0)
    ident = same(outs['host'][0], outs['device'][0]) and same(outs['host'][1], outs['device'][1])
    res['forms']['evaluate_clean'] = dict(host_s=t['host'], device_s=t['device'], identical=bool(ident))
    print('evaluate_clean', res['forms']['evaluate_clean'], flush=True)

    # fokl_rows_compact alone, and the HBM bandwidth of a device-to-device copy for scale
    eng = FR._engine()
    ds = eng.upload(raw, y)
    mask = np.random.default_rng(1).random(n) < 0.8
    kept = int(mask.sum())
    for _ in range(3):
        eng.rows_compact(ds, mask)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    reps = 20
    ms = []
    for _ in range(reps):
        ev[0].record()
        eng.rows_compact(ds, mask)
        ev[1].record()
        torch.cuda.synchronize()
        ms.append(ev[0].elapsed_time(ev[1]))
    m = ds.m
    alg_bytes = n + 8 * n * (m + 1) + 8 * kept * (m + 1)
    src = torch.empty(1 << 29, dtype=torch.float64, device='cuda')      # 4 GB, well past the L2
    dst = torch.empty_like(src)
    for _ in range(3):
        dst.copy_(src)
    cms = []
    for _ in range(10):
        ev[0].record()
        dst.copy_(src)
        ev[1].record()
        torch.cuda.synchronize()
        cms.append(ev[0].elapsed_time(ev[1]))
    peak = 2 * src.numel() * 8 / (min(cms) / 1e3)
    med = float(np.median(ms))
    res['rows_compact'] = dict(n=n, m=m, kept=kept, bytes=alg_bytes, ms_median=med, ms_min=float(min(ms)),
                               gb_per_s=alg_bytes / (med / 1e3) / 1e9, copy_peak_gb_per_s=peak / 1e9,
                               fraction_of_copy_peak=alg_bytes / (med / 1e3) / peak,
                               note='event window includes the host read of the kept count (one stream sync); '
                                    'the mask upload (N bytes) is inside the window too')
    print('rows_compact', res['rows_compact'], flush=True)

    t0 = time.perf_counter()
    np.random.seed(5)
    FR.FoKL().generate_trainlog(0.8, n)
    res['generate_trainlog_s'] = time.perf_counter() - t0
    print(json.dumps(res))
    if a.out:
        with open(a.out, 'w') as f:
            json.dump(res, f)


if __name__ == '__main__':
    main()
