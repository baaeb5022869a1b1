"""`generate_trainlog(0.8, N)` on the host against fokl_trainlog, and the end-to-end `fit(clean=True, train=0.8)` with
either split, at N = 10^7 rows (cfg4's shape) on one GPU.

The host loop (forced by raising _TRAINLOG_ON_DEVICE_MIN_ROWS) and the device split alternate in one process from the
same numpy state; masks and RNG end states are compared bit for bit, and so are the two fits' betas / mtx / evs.  A
separate pass under torch.profiler (CUDA activities) divides one device split's kernel time between MT19937 generation
(trainlog_mt_gen), the parse of the words (trainlog_parse) and the set / permutation work (the other trainlog_*
kernels).  Prints one JSON object (and writes it to --out)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, 'fokl-gpy_b200'), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

HOST = 1 << 62


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else 'unknown'


def same_state(s, t):
    return bool(s[0] == t[0] and np.array_equal(s[1], t[1]) and s[2:] == t[2:])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--n', type=int, default=10 ** 7)
    ap.add_argument('--train', type=float, default=0.8)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--fit-reps', type=int, default=2)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    import torch
    import bench_data
    from FoKL import FoKLRoutines as FR
    from FoKL import getKernels
    assert torch.cuda.is_available(), 'trainlog_bench needs a GPU'
    n, train = a.n, a.train
    device_min = FR._TRAINLOG_ON_DEVICE_MIN_ROWS
    res = dict(card=card(), n=n, train=train, l_log=max(int(n * train), 2))

    def split(where, seed):
        FR._TRAINLOG_ON_DEVICE_MIN_ROWS = where
        np.random.seed(seed)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        mask = FR.FoKL().generate_trainlog(train, n)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, mask, np.random.get_state()

    split(device_min, 0)                                   # module load, context, allocator pools
    host_s, dev_s, equal = [], [], True
    for r in range(a.reps):
        th, mh, sh = split(HOST, 100 + r)
        td, md, sd = split(device_min, 100 + r)
        host_s.append(th)
        dev_s.append(td)
        equal = equal and bool(np.array_equal(mh, md)) and same_state(sh, sd)
    res['generate_trainlog_s'] = dict(host=host_s, device=dev_s, equal=equal)

    FR._TRAINLOG_ON_DEVICE_MIN_ROWS = device_min
    state = np.random.get_state()
    _, key, pos, words = FR._engine().trainlog(state[1], state[2], n, max(int(n * train), 2))
    res['words_consumed'] = int(words)

    # kernel time of one device split, by stage (a run of its own: the profiler slows the host)
    from torch.profiler import ProfilerActivity, profile
    np.random.seed(7)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        FR.FoKL().generate_trainlog(train, n)
        torch.cuda.synchronize()
    stages = {'generation': 0.0, 'parse': 0.0, 'set_and_permutation': 0.0}
    launches = {}
    for ev in prof.key_averages():
        name = ev.key
        if 'trainlog_' not in name:
            continue
        us = getattr(ev, 'device_time_total', None)
        if us is None:
            us = ev.cuda_time_total
        short = name[name.index('trainlog_'):].split('(')[0]
        launches[short] = launches.get(short, 0) + ev.count
        stage = 'generation' if short == 'trainlog_mt_gen' else 'parse' if short == 'trainlog_parse' \
            else 'set_and_permutation'
        stages[stage] += us / 1e3
    res['device_kernel_ms'] = stages
    res['device_launches'] = launches

    # end to end: fit(clean=True, train=0.8) at cfg4's shape with either split
    x, y = bench_data.make_rows('cfg4', 0, n, n_total=n)
    raw = x * np.arange(1.0, 9.0) - 2.0
    del x
    phis = getKernels.sp500()
    fits = {'host': [], 'device': []}
    outs = {}
    for r in range(a.fit_reps + 1):
        for name, where in (('host', HOST), ('device', device_min)):
            FR._TRAINLOG_ON_DEVICE_MIN_ROWS = where
            np.random.seed(21)
            model = FR.FoKL(phis=phis, way3=True, UserWarnings=False, ConsoleOutput=False)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = model.fit(raw, y, clean=True, train=train)
            torch.cuda.synchronize()
            if r > 0:                                      # the first round warms every shape up
                fits[name].append(time.perf_counter() - t0)
            outs[name] = out + (model.trainlog, np.random.get_state())
    h, d = outs['host'], outs['device']
    res['fit_s'] = fits
    res['fit_equal'] = bool(all(np.array_equal(h[k], d[k]) for k in range(4)) and same_state(h[4], d[4]))
    FR._TRAINLOG_ON_DEVICE_MIN_ROWS = device_min
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            json.dump(res, f)


if __name__ == '__main__':
    main()
