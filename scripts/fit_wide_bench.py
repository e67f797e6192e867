"""Warm PolyModel.fit at 64 < input_size <= 128 and up to P = 16381 parameters: quadratic n = 72 / 96 / 128 and cubic-2 n = 64 / 104,
N = 2 P rows from the host.  Per case, the best of three:
  - fit_s:   the whole PolyModel.fit call (host copies, Gram, solve, bound ellipsoid, f_mu);
  - gram_ms: gram_kernel + gram_reduce_kernel (CUDA events around the accumulation), and N P (P + 1) / gram_ms in TFLOP/s;
  - solve_s: bfb_fit_solve (equilibration, Cholesky, triangular solves, refinement; it ends in a device synchronise).
One torch.profiler pass per case then sums the device time of each solve kernel (cholesky_ms, trsv_ms).
Prints the GPU's name and power limit; writes one JSON object to --out.

    python scripts/fit_wide_bench.py --out fit_wide_bench.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np

CASES = (('quadratic', 72), ('quadratic', 96), ('quadratic', 128), ('cubic-2', 64), ('cubic-2', 104))


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
    return q.stdout.strip()


def problem(n, N, seed):
    rng = np.random.default_rng(seed)
    x = rng.normal(size=(N, n))
    y = (-0.5 * np.sum(x**2, axis=1) + 0.1 * x[:, 0] * x[:, -1]**2 + 1e-3 * rng.normal(size=N))[:, None]
    return x, y


def run_case(order, n, reps):
    import torch
    import bayesfast_b200 as bfb
    from bayesfast_b200 import _cabi
    s = bfb.PolyModel(order, input_size=n, output_size=1)
    P = s.n_param
    N = 2 * P
    x, y = problem(n, N, n)
    s.fit(x, y, logp=y[:, 0])                      # warm-up: module load, allocations
    fit_s = []
    for _ in range(reps):
        t0 = time.perf_counter()
        s.fit(x, y, logp=y[:, 0])
        fit_s.append(time.perf_counter() - t0)
    h, L = s._dev(), _cabi.lib()
    gram_ms, solve_s = [], []
    out, rr = np.empty(P), C.c_double(0.)
    for _ in range(reps):
        _cabi.check(L.bfb_fit_begin(h._h, None))
        _cabi.check(L.bfb_fit_accumulate(h._h, x.ctypes.data, y.ctypes.data, None, N, _cabi.BFB_HOST))
        gram_ms.append(h.last_kernel_ms())
        t0 = time.perf_counter()
        _cabi.check(L.bfb_fit_solve(h._h, out.ctypes.data_as(_cabi._dp), C.byref(rr)))
        solve_s.append(time.perf_counter() - t0)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        _cabi.check(L.bfb_fit_solve(h._h, out.ctypes.data_as(_cabi._dp), C.byref(rr)))
        torch.cuda.synchronize()
    dev_ms = {}
    for e in prof.key_averages():
        t = getattr(e, 'device_time_total', None)
        if t is None:
            t = e.cuda_time_total
        dev_ms[e.key] = dev_ms.get(e.key, 0.) + t / 1e3
    chol = sum(v for k, v in dev_ms.items() if k.startswith(('chol_diag', 'chol_trsm', 'chol_syrk')))
    trsv = sum(v for k, v in dev_ms.items() if 'chol_solve_kernel' in k)
    g = min(gram_ms)
    return dict(order=order, n=n, P=P, N=N, fit_s=min(fit_s), gram_ms=g, gram_tflops=N * P * (P + 1) / (g * 1e-3) / 1e12,
                solve_s=min(solve_s), cholesky_ms=chol, trsv_ms=trsv, rel_resid=rr.value)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--reps', type=int, default=3)
    a = ap.parse_args()
    info = gpu_info()
    print('gpu:', info, flush=True)
    rows = []
    for order, n in CASES:
        r = run_case(order, n, a.reps)
        print(json.dumps(r), flush=True)
        rows.append(r)
    res = dict(gpu=info, rows=rows)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
