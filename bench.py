#!/usr/bin/env python
"""bench.py -- FoKL.fit throughput on B200 (BASELINE.json metric: candidate-models/sec; basis-matrix GB/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg4] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = one complete `FoKL.fit` (forward selection: basis build -> Gram -> per-candidate spectral
factorisation + Gibbs chain -> BIC) on the synthetic workload of BASELINE.json `configs[3]` (cfg4: N = 10M rows,
8 inputs, 3-way interactions, cubic splines, 1000 + 1000 draws), rows sharded over the N GPUs (strong scaling of the
fixed 10M-row problem, one NCCL allreduce of the new Gram block per substage).  One "candidate model" = one `gibbs`
invocation of the reference (FoKLRoutines.py:1650 / :1681).

    value  candidate-models/sec with the normalised dataset already resident in HBM (fit(DeviceDataset))
    e2e    the same through the public API with HOST numpy buffers: FoKL.fit(inputs, data, clean=True) -- host
           formatting, host->device copies and the device->host read of betas/mtx/evs inside the timed region
    roofline      K1 basis kernel (HBM-bound): algorithmic bytes 8*N*(M + C) per launch / CUDA-event time, against
                  MEASURED_PEAKS.json hbm_gbs; `roofline_gram` the K2 FP64 DMMA Gram against an in-run cuBLAS DGEMM
    cpu_baseline  the CPU oracle (oracle/fokl_oracle.py, a numpy restatement of the reference) on a bounded sample
`--impl reference` times that CPU oracle alone (rank 0), same metric / config keys.
Timing: CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks.
`--dump-outputs DIR` writes what the last timed resident fit returned (betas, mtx, evs) as DIR/<name>.npy in float64, so
that two builds can be compared output for output on the same seeded inputs.  Apart from DIR the benchmark writes no
files: it may run from a read-only tree.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (os.path.join(ROOT, 'fokl-gpy_b200'), ROOT):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

import bench_data  # noqa: E402

METRIC = 'FoKL.fit candidate-models/sec'
UNIT = 'candidate-models/s'


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='cfg4', choices=sorted(bench_data.CONFIGS))
    ap.add_argument('--n', type=int, default=0, help='override the number of rows (debugging only)')
    ap.add_argument('--draws', type=int, default=1000)
    ap.add_argument('--cpu-rows', type=int, default=0, help='rows of the reduced-N CPU fit (default: 10^4; 2*10^4 for cfg3)')
    ap.add_argument('--cpu-seconds', type=float, default=240.0,
                    help='--impl reference: total wall-time bound; complete fits are repeated until --steps or this')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write betas / mtx / evs of the last timed fit to DIR/<name>.npy (float64, at most 64 MB)')
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error('--steps must be >= 1 and --warmup >= 0')
    if a.dump_outputs and a.impl != 'b200':
        ap.error('--dump-outputs writes the device fit: it needs --impl b200')
    return a


DUMP_BYTES = 60 << 20      # array data; keeps the files, headers included, under 64 MB


def dump_outputs(out_dir, arrays):
    """arrays: name -> array.  Each is written as out_dir/<name>.npy in float64.  If they would exceed DUMP_BYTES in all,
    the rows of betas (one per draw) are cut to a sample fixed by seed 0, kept in draw order, so that the files stay
    comparable between runs."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    over = sum(v.nbytes for v in arrays.values()) - DUMP_BYTES
    if over > 0:
        betas = arrays['betas']
        keep = betas.shape[0] - -(-over // (betas.shape[1] * 8))
        assert keep > 0, 'the outputs other than betas alone exceed the %d-byte dump budget' % DUMP_BYTES
        rows = np.sort(np.random.default_rng(0).choice(betas.shape[0], size=keep, replace=False))
        arrays['betas'] = betas[rows]
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + '.npy'), v)


def config_dict(a, n_total, world, extra=None):
    c = bench_data.CONFIGS[a.workload]
    d = {'workload': '%s: synthetic N=%d, M=%d, %s, %s, burnin+draws=%d+%d' % (
        a.workload, n_total, c['m'], '3-way' if c['way3'] else '2-way', c['kernel'], a.draws, a.draws),
        'rows': n_total, 'inputs': c['m'], 'way3': c['way3'], 'kernel': c['kernel'],
        'sharding': 'rows/%d' % world, 'l2': 'inputs_exceed_l2 (%.0f MB per rank)' % (n_total / world * c['m'] * 8 / 1e6)}
    if extra:
        d.update(extra)
    return d


# ---------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ---------------------------------------------------------------------------------------------------
class Clocks:
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.samples, self.stop_flag, self.th = index, [], threading.Event(), None

    def _run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                      '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=10).stdout
                parts = [s.strip() for s in out.strip().split(',')]
                if len(parts) >= 6:
                    self.samples.append(parts)
            except Exception:
                pass
            self.stop_flag.wait(0.5)

    def start(self):
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()

    def stop(self):
        self.stop_flag.set()
        if self.th is not None:
            self.th.join(timeout=15)
        sm, mx, reasons = [], 0.0, set()
        for p in self.samples:
            try:
                sm.append(float(p[0]))
                mx = max(mx, float(p[1]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), p[2:6]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': mx or None, 'reasons': sorted(reasons),
                'samples': len(sm)}


# ---------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (a numpy / OpenBLAS / LAPACK restatement of the reference + a C basis helper), run TO
# COMPLETION on a reduced-N instance of the same workload -- the value does not depend on a time budget
# ---------------------------------------------------------------------------------------------------
CPU_ROWS_DEFAULT = {'cfg3': 20000, 'cfg4': 10000, 'cfg5': 10000}      # BASELINE.md section 3 / SURVEY 8(d)


class _CpuBudget(Exception):
    pass


def cpu_rows(a):
    return a.cpu_rows or CPU_ROWS_DEFAULT[a.workload]


def cpu_fit_complete(a, phis, rows, guard_s=600.0):
    """One complete oracle fit of the workload at `rows` rows, all host threads.  Returns a dict with the number of
    `gibbs` calls, seconds, design-matrix cells built, draws made, model widths and the time spent in the basis helper.
    guard_s is a safety net only (never reached at the default sizes): a fit cut by it is flagged complete=False."""
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import fokl_oracle as fo
    c = bench_data.CONFIGS[a.workload]
    x, y = bench_data.make_rows(a.workload, 0, rows, n_total=rows)
    np.random.seed(c['seed'])
    threads = os.cpu_count() or 1
    st = dict(calls=0, t=0.0, pmax=0, cells=0, t_basis=0.0, draws=0, psum=0, p2sum=0, complete=True)
    real_basis = fo.basis_columns

    def timed_basis(x_, terms, *args, **kw):
        t = time.perf_counter()
        out = real_basis(x_, terms, *args, **kw)
        st['t_basis'] += time.perf_counter() - t
        st['cells'] += out.size
        return out

    t0 = time.perf_counter()

    def on_gibbs(info):
        st['calls'] = info['call']
        st['t'] = time.perf_counter() - t0
        p = info['discmtx'].shape[0] + 1
        st['pmax'] = max(st['pmax'], p)
        st['psum'] += p
        st['p2sum'] += p * p
        st['draws'] += 2 * a.draws
        if guard_s and st['t'] > guard_s:
            raise _CpuBudget()

    fo.basis_columns = timed_basis
    # all host threads for BLAS / LAPACK whatever the launcher exported: torchrun sets OMP_NUM_THREADS=1 for its workers,
    # which would make this arm single-threaded at N > 1 and multi-threaded at N = 1
    import scipy.linalg  # noqa: F401  (loads scipy's OpenBLAS so that the limit below covers it too)
    import threadpoolctl
    limits = threadpoolctl.threadpool_limits(limits=threads)
    st['blas_threads'] = sorted({int(d['num_threads']) for d in threadpoolctl.threadpool_info()}) or [1]
    try:
        r = fo.fit(x, y, phis, kernel=c['kernel'], way3=c['way3'], draws=a.draws, burnin=a.draws, threads=threads,
                   on_gibbs=on_gibbs)
        st['terms'], st['substages'] = int(r.mtx.shape[0]), int(len(r.evs))
        st['t'] = time.perf_counter() - t0
    except _CpuBudget:
        st['complete'] = False
    finally:
        fo.basis_columns = real_basis
    st['threads'], st['rows'] = threads, rows
    # X'X, X'y (FR:1492-1494) are recomputed in full by every call: 2 N p^2 flops each, at the BLAS rate measured here
    A = np.random.default_rng(0).random((rows, 128))
    A.T.dot(A)
    tg = time.perf_counter()
    for _ in range(5):
        A.T.dot(A)
    rate = 5 * 2.0 * rows * 128 * 128 / (time.perf_counter() - tg)
    st['gram_flops'] = 2.0 * rows * st['p2sum']
    st['t_gram_est'] = st['gram_flops'] / rate
    st['gram_gflops_rate'] = rate / 1e9
    limits.restore_original_limits()
    return st


def cpu_python_loop_cost(a, phis, seconds=3.0):
    """us per design-matrix cell of the reference's literal Python triple loop (FR:1446-1485; oracle basis='py'),
    measured on a few hundred rows of the workload's 3-way / 2-way terms for ~`seconds` s."""
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import fokl_oracle as fo
    c = bench_data.CONFIGS[a.workload]
    x, _ = bench_data.make_rows(a.workload, 0, 512, n_total=512)
    part = ([1, 1, 1] if c['way3'] else [1, 1]) + [0] * (c['m'] - (3 if c['way3'] else 2))
    terms = fo.distinct_perms(part).astype(int)[:8]
    rows, cells, t0 = 16, 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        fo.basis_columns_py(x[:rows], terms, phis, c['kernel'])
        cells += rows * terms.shape[0]
    return 1e6 * (time.perf_counter() - t0) / cells


def cpu_report(a, st, n_full, py_us):
    """The numbers SURVEY 8(d) asks for next to the CPU value, plus the linear-in-N extrapolation LABELLED as such."""
    t, tb = st['t'], st['t_basis']
    cells_s = st['cells'] / tb if tb > 0 else None
    scale = n_full / st['rows']
    rep = {
        'rows': st['rows'], 'complete_fit': st['complete'], 'seconds': t, 'gibbs_calls': st['calls'],
        'blas_threads': st.get('blas_threads'),
        'terms_selected': st.get('terms'), 'substages': st.get('substages'), 'max_model_width': st['pmax'],
        'cells_built': st['cells'], 'basis_seconds_c_helper': tb, 'cells_per_s_c_helper': cells_s,
        'gram_flops': st['gram_flops'], 'gram_seconds_estimate': st['t_gram_est'], 'gram_gflops_rate': st['gram_gflops_rate'],
        'draws': st['draws'], 'draws_per_s': st['draws'] / max(t - tb - st['t_gram_est'], 1e-9),
        'python_loop_us_per_cell': py_us,
        'reference_as_shipped_seconds_estimate': (t - tb) + st['cells'] * py_us * 1e-6 if py_us else None,
        'extrapolation_to_full_N': {
            'note': 'LABELLED EXTRAPOLATION, not a measurement: the same %d gibbs calls at N=%d, basis and Gram time '
                    'scaled linearly in N, draw loop unchanged; the real N=%d fit keeps more terms and makes more calls'
                    % (st['calls'], n_full, n_full),
            'seconds_port_c_helper': (t - tb - st['t_gram_est']) + (tb + st['t_gram_est']) * scale,
            'seconds_reference_python_loop': ((t - tb - st['t_gram_est']) + (st['t_gram_est'] + st['cells'] * py_us * 1e-6) * scale)
            if py_us else None}}
    return rep


def cpu_sample_desc(a, st):
    return ('oracle port (numpy/OpenBLAS/LAPACK like the reference + a C basis helper, i.e. faster than the reference, '
            'whose basis build is a Python triple loop) of the %s fit at N=%d rows, %d+%d draws, run to completion: '
            '%d gibbs calls in %.1f s (model width up to %d columns)%s'
            % (a.workload, st['rows'], a.draws, a.draws, st['calls'], st['t'], st['pmax'],
               '' if st['complete'] else ' -- CUT by the safety guard'))


def run_reference(a):
    """`--impl reference`: complete CPU fits of the reduced-N workload on rank 0.  The TOTAL wall time is bounded
    independently of --steps: fits are repeated until `--steps` are done or --cpu-seconds (default 240 s) are used up,
    whichever comes first, and at least one fit always completes; warm-up is one import + one tiny fit."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    phis = load_phis(a)
    n_total = a.n or bench_data.CONFIGS[a.workload]['n']
    rows = cpu_rows(a)
    t_start = time.perf_counter()
    if a.warmup:
        cpu_fit_complete(a, phis, 300, guard_s=20.0)          # page in numpy / LAPACK / the C helper
    py_us = cpu_python_loop_cost(a, phis)
    fits = []
    while len(fits) < max(a.steps, 1):
        fits.append(cpu_fit_complete(a, phis, rows))
        if time.perf_counter() - t_start + fits[-1]['t'] > a.cpu_seconds:
            break
    tot_models = sum(f['calls'] for f in fits)
    tot_s = sum(f['t'] for f in fits)
    v = tot_models / tot_s
    st = fits[-1]
    line = {'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': UNIT, 'n_gpus': a.gpus, 'steps': a.steps,
            'steps_run': len(fits), 'warmup': a.warmup, 'ms_per_step': 1e3 * tot_s / len(fits),
            'higher_is_better': True, 'scaling': 'strong',
            'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': config_dict(a, n_total, 1, {'cpu_sample_rows': rows}),
            'cpu_baseline': {'value': v, 'unit': UNIT, 'cores': st['threads'], 'kind': 'port',
                             'sample': cpu_sample_desc(a, st), 'detail': cpu_report(a, st, n_total, py_us)},
            'e2e': {'value': v, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line), flush=True)


def load_phis(a):
    import warnings
    from FoKL import getKernels
    if bench_data.CONFIGS[a.workload]['kernel'] == 'Cubic Splines':
        if not os.path.exists(os.path.join(getKernels._KDIR, getKernels.UPSTREAM_SPLINE_FILE)):
            # the table sp500() would fall back to, built from the current code: no cache file written into the
            # package, and never one left behind by another build
            return getKernels._to_phis(getKernels.regenerate_spline_table(500))
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            return getKernels.sp500()
    return getKernels.bernoulli()


# ---------------------------------------------------------------------------------------------------
def measure_fp64_peak(torch, dev):
    """cuBLAS DGEMM ceiling on this box (MEASURED_PEAKS.json has no FP64 figure): 4096^3, best of 5."""
    n = 4096
    A = torch.randn(n, n, dtype=torch.float64, device=dev)
    B = torch.randn(n, n, dtype=torch.float64, device=dev)
    torch.matmul(A, B)
    best = float('inf')
    for _ in range(5):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        torch.matmul(A, B)
        e.record()
        torch.cuda.synchronize(dev)
        best = min(best, s.elapsed_time(e))
    del A, B
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12


def main():
    a = parse()
    if a.impl == 'reference':
        run_reference(a)
        return
    import torch
    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (the B200 path has no CPU fallback); use --impl reference for the CPU arm')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
    from FoKL import FoKLRoutines as FR

    c = bench_data.CONFIGS[a.workload]
    n_total = a.n or c['n']
    per = -(-n_total // world)
    lo, hi = rank * per, min((rank + 1) * per, n_total)
    x_host, y_host = bench_data.make_rows(a.workload, lo, hi, n_total=n_total)
    # pinned host buffers (the e2e arm copies from these every step)
    x_pin = torch.from_numpy(x_host).pin_memory()
    y_pin = torch.from_numpy(y_host).pin_memory()
    x_host, y_host = x_pin.numpy(), y_pin.numpy()
    phis = load_phis(a)
    m = c['m']
    unit_minmax = [[0.0, 1.0]] * m      # the generator draws inputs in [0, 1): global bounds, identical on every rank

    eng = FR._engine()
    eng.set_phis(phis, c['kernel'])

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def new_model():
        return bench_data.make_model(FR, a.workload, draws=a.draws, phis=phis)

    ds = eng.upload(x_host, y_host)
    last_fit = {}

    def step_resident():
        np.random.seed(c['seed'])
        model = new_model()
        last_fit['betas'], last_fit['mtx'], last_fit['evs'] = model.fit(ds, None)
        return dict(FR.LAST_FIT_INFO)

    def step_e2e():
        np.random.seed(c['seed'])
        model = new_model()
        betas, mtx, evs = model.fit(x_host, y_host, clean=True, minmax=unit_minmax, AutoTranspose=False)
        info = dict(FR.LAST_FIT_INFO)
        info['d2h'] = betas.nbytes + mtx.nbytes + evs.nbytes
        return info

    def timed(fn, steps, profile):
        barrier()
        eng.profile = {} if profile else None
        l0 = eng.launch_count()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        s.record()
        infos = [fn() for _ in range(steps)]
        e.record()
        barrier()
        wall = time.perf_counter() - t0
        ms = s.elapsed_time(e)
        t = torch.tensor([ms, wall * 1e3], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        prof = eng.profile_summary() if profile else {}
        eng.profile = None
        return infos, float(t[0].item()), float(t[1].item()), eng.launch_count() - l0, prof

    fp64_peak = measure_fp64_peak(torch, dev) if rank == 0 else None

    for _ in range(a.warmup):
        step_resident()
    clocks = Clocks(local)
    if rank == 0:
        clocks.start()
    infos, ms, wall_ms, launches, prof = timed(step_resident, a.steps, True)
    clk = clocks.stop() if rank == 0 else None
    models = sum(i['n_gibbs'] for i in infos)
    value = models / (ms * 1e-3)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, last_fit)

    e2e = None
    if not a.no_e2e:
        step_e2e()
        einfos, ems, ewall, _, _ = timed(step_e2e, a.steps, False)
        emodels = sum(i['n_gibbs'] for i in einfos)
        e2e = {'value': emodels / (ems * 1e-3), 'unit': UNIT,
               'h2d_bytes_per_step': int(x_host.nbytes + y_host.nbytes), 'd2h_bytes_per_step': int(einfos[-1]['d2h']),
               'ms_per_step': ems / a.steps}

    # the same call with ordinary (pageable) numpy arrays, as a user who never heard of pinned memory passes them
    e2e_pageable = None
    if not a.no_e2e:
        x_page, y_page = np.array(x_host, copy=True), np.array(y_host, copy=True)

        def step_pageable():
            np.random.seed(c['seed'])
            model = new_model()
            model.fit(x_page, y_page, clean=True, minmax=unit_minmax, AutoTranspose=False)
            return dict(FR.LAST_FIT_INFO)

        step_pageable()
        pinfos, pms, _, _, _ = timed(step_pageable, max(1, min(a.steps, 3)), False)
        e2e_pageable = {'value': sum(i['n_gibbs'] for i in pinfos) / (pms * 1e-3), 'unit': UNIT,
                        'ms_per_step': pms / len(pinfos), 'host_buffers': 'pageable numpy arrays'}
        del x_page, y_page
    if e2e is not None:
        e2e['host_buffers'] = 'pinned (torch pin_memory)'
        e2e['pageable'] = e2e_pageable

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm_peak = float(peaks.get('hbm_gbs', 6650.0))
    hbm_src = 'MEASURED_PEAKS.json hbm_gbs (of measured)' if 'hbm_gbs' in peaks else '6650 GB/s (of fallback)'

    def stage(name):
        return prof.get(name, {'ms': 0.0, 'calls': 0})

    # DRAM traffic per launch from the committed `ncu --set full` capture of this same command (tools/ncu_traffic.py
    # over the .ncu-rep of one cfg4 fit); a number taken under the profiler is evidence, not a timing
    traffic, traffic_src = {}, None
    for name in ('r02_ncu_traffic.json', 'r01_ncu_traffic.json'):      # newest capture first (tools/gpurun/gpu_final_r2.sh)
        try:
            with open(os.path.join(ROOT, 'profiles', name)) as f:
                traffic = json.load(f)
            traffic_src = 'profiles/' + name + (' @ ' + traffic['_commit'] if '_commit' in traffic else '')
            break
        except Exception:
            continue

    def traffic_of(kernel):
        if a.workload != 'cfg4' or a.n or world != 1:
            return None
        parts = [v for k, v in traffic.items() if isinstance(v, dict) and k.startswith(kernel)]
        if not parts:
            return None
        return sum(v['dram_read_bytes'] + v['dram_write_bytes'] for v in parts) / sum(v['launches'] for v in parts)

    tot_ms = ms
    shares = {k: v['ms'] / tot_ms for k, v in prof.items()}
    b = stage('basis')
    roof = None
    if b['calls']:
        ach = b['bytes'] / (b['ms'] * 1e-3) / 1e9
        roof = {'kernel': 'basis_kernel (K1)', 'bound': 'hbm', 'achieved': ach, 'peak': hbm_peak, 'unit': 'GB/s',
                'frac': ach / hbm_peak, 'traffic': traffic_of('basis_kernel'), 'traffic_source': traffic_src,
                'peak_source': hbm_src,
                'launches': b['calls'],
                'avg_launch_ms': b['ms'] / b['calls'], 'bytes_per_launch': b['bytes'] / b['calls'],
                'share_of_step': shares.get('basis')}
    g = stage('gram')
    roof_g = None
    if g['calls'] and fp64_peak:
        ach = g['flops'] / (g['ms'] * 1e-3) / 1e12
        roof_g = {'kernel': 'gram_kernel (K2, FP64 DMMA)', 'bound': 'tensor', 'achieved': ach, 'peak': fp64_peak,
                  'unit': 'TFLOP/s', 'frac': ach / fp64_peak, 'traffic': traffic_of('gram_kernel'),
                  'peak_source': 'in-run cuBLAS DGEMM 4096^3 (torch.matmul f64), best of 5', 'launches': g['calls'],
                  'avg_launch_ms': g['ms'] / g['calls'], 'share_of_step': shares.get('gram')}

    cpu = None
    if world == 1 and not a.no_cpu_baseline:
        st = cpu_fit_complete(a, phis, cpu_rows(a))
        cpu = {'value': st['calls'] / st['t'], 'unit': UNIT, 'cores': st['threads'], 'kind': 'port',
               'sample': cpu_sample_desc(a, st), 'seconds': st['t'],
               'detail': cpu_report(a, st, n_total, cpu_python_loop_cost(a, phis))}

    line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': a.steps, 'warmup': a.warmup,
            'ms_per_step': ms / a.steps, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
            'dtype': 'f64', 'data': 'synthetic', 'config': config_dict(a, n_total, world, {'cpu_sample_rows': cpu_rows(a)}),
            'candidate_models_per_step': models / a.steps,
            'work_per_step': {
                'note': "candidate_models_per_step counts the reference's `gibbs` invocations (FR:1650 full models + "
                        "FR:1681 one per kill proposal).  Here a kill proposal's BIC is an O(1) score from the "
                        "sweep-operator tableau of the model's Gram (kill_proposals_scored); an eigensolve + Gibbs chain "
                        "is run only for the full models and for the accepted models whose chain can influence a later "
                        "decision (eig_solves / chains_run)",
                **{k: sum(i.get(k, 0) for i in infos) / a.steps
                   for k in ('eig_solves', 'chains_run', 'secular_steps', 'kill_loops', 'kill_proposals_scored')}},
            'terms_selected': infos[-1]['terms'],
            'substages': infos[-1]['substages'], 'wall_ms_per_step': wall_ms / a.steps,
            'e2e': e2e, 'gpu_launches': int(launches), 'clocks': clk, 'roofline': roof, 'roofline_gram': roof_g,
            'roofline_note': "roofline = the basis-matrix kernel BASELINE.json's metric names (HBM-bound); "
                             "roofline_gram = the kernel with the largest share of the step (FP64 tensor pipe)",
            'stage_ms_per_step': {k: v['ms'] / a.steps for k, v in prof.items()},
            'cpu_baseline': cpu}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
