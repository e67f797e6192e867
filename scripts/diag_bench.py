"""Split-R-hat / ESS on the device (csrc/bfb_diag.cu): the kernels alone on a resident [4096, 1000, 26] array, the cost they add to the
headline sample() call, and min / median ESS per second of the tensor-core diagonal-metric run against the dense-metric generic run.
Headline workload: d = 26 cubic-2 (synthetic.des_shaped), 4096 chains, n_iter 1500, n_warmup 500.  Prints one JSON line per
measurement; --out FILE also writes them all to FILE.

    python scripts/diag_bench.py [--reps 3] [--out diag_bench.json]
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import bayesfast_b200 as bfb
from bayesfast_b200 import _cabi, synthetic

REPS = int(sys.argv[sys.argv.index('--reps') + 1]) if '--reps' in sys.argv else 3
OUT = sys.argv[sys.argv.index('--out') + 1] if '--out' in sys.argv else None
N_DIM, C, N_ITER, N_WARMUP, SEED = 26, 4096, 1500, 500, 7
rows = []


def emit(**kw):
    rows.append(kw)
    print(json.dumps(kw), flush=True)


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return [s.strip() for s in q.split(',')]
    except Exception as exc:
        return ['unknown ({})'.format(exc)]


def flops(Mp, L, n):
    """Gram form: the upper triangle of every M' x L Gram, M' L (L + 1) n flops.  FFT form for comparison: per half-chain and
    coordinate a real forward and inverse FFT of the zero-padded length 2^ceil(log2(2L)) (2.5 P log2 P flops each) and the power
    spectrum (3 P)"""
    P = 1 << int(np.ceil(np.log2(2 * L)))
    return Mp * L * (L + 1) * n, Mp * n * (2 * 2.5 * P * np.log2(P) + 3 * P)


def main():
    import torch
    info = gpu_info()
    emit(what='gpu', name=info[0], power_limit=info[1] if len(info) > 1 else None, max_sm_clock=info[2] if len(info) > 2 else None)
    prob = synthetic.des_shaped(N_DIM, seed=1, n_chain=C, order='cubic-2')
    sur = bfb.PolyModel('cubic-2', input_size=N_DIM, output_size=1)
    sur.fit(prob['x_fit'], prob['y_fit'], logp=prob['y_fit'][:, 0])
    den = bfb.Density(sur)
    h = den._sync(False)
    kw = dict(n_chain=C, n_iter=N_ITER, n_warmup=N_WARMUP, x_0=prob['x_0'], random_generator=SEED)

    # ---- end to end: sample(keep='post_warmup') with and without the diagnostics, alternated ----
    walls = {'post_warmup': [], 'post_warmup+diagnostics': [], 'fields=()+summaries+diagnostics': []}
    kms = {k: [] for k in walls}
    tt = None
    for rep in range(REPS + 1):                       # the first round warms up every shape
        for name, extra in (('post_warmup', {}), ('post_warmup+diagnostics', dict(diagnostics=True)),
                            ('fields=()+summaries+diagnostics', dict(fields=(), summaries=True, diagnostics=True))):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = bfb.sample(den, dict(kw), verbose=False, keep='post_warmup', **extra)
            dt = time.perf_counter() - t0
            if rep:
                walls[name].append(dt)
                kms[name].append(r.kernel_ms)
            if name == 'post_warmup+diagnostics':
                tt = r
    base = np.median(walls['post_warmup'])
    for name in walls:
        emit(what='e2e', call=name, wall_s_median=float(np.median(walls[name])), wall_s_all=walls[name],
             sampling_kernel_ms_median=float(np.median(kms[name])), over_post_warmup=float(np.median(walls[name]) / base - 1.))

    # ---- the kernels alone on the resident post-warm-up samples of that run ----
    x = torch.from_numpy(np.ascontiguousarray(tt.samples)).cuda()
    torch.cuda.synchronize()
    Cc, N, n = x.shape
    L = N // 2
    h.chain_diagnostics(x.data_ptr(), Cc, N, 0, N, n, _cabi.BFB_DEVICE)      # warm-up (workspace, module load)
    ms = []
    for _ in range(20):
        P = h.chain_diagnostics(x.data_ptr(), Cc, N, 0, N, n, _cabi.BFB_DEVICE)
        ms.append(h.last_kernel_ms())
    same = bfb.diag.finish(P)
    assert all(np.array_equal(same[k], tt.diagnostics[k]) for k in ('rhat', 'ess'))
    peak = max(h.fp64_peak(1) for _ in range(2))      # DMMA m8n8k4, TFLOP/s, measured now on this GPU
    fg, ff = flops(2 * Cc, L, n)
    t = float(np.median(ms))
    emit(what='kernels', shape=[Cc, N, n], ms_median=t, ms_min=float(min(ms)), gram_flops=fg, tflops=fg / t * 1e-9,
         fp64_dmma_peak_tflops=peak, fraction_of_peak=fg / t * 1e-9 / peak, fft_form_flops=ff, gram_over_fft_flops=fg / ff,
         input_bytes=8 * Cc * N * n, workspace_bytes=8 * n * 2 * Cc * ((L + 63) // 64 * 64))

    # ---- ESS per second: tensor-core diagonal metric vs the dense metric on the generic kernel ----
    for name, extra in (('diag/tensor-core', {}), ('dense/generic', dict(metric='full'))):
        r = bfb.sample(den, dict(kw, **extra), verbose=False, keep='post_warmup', fields=(), diagnostics=True)
        ess = r.diagnostics['ess']
        s = r.kernel_ms * 1e-3
        emit(what='ess_per_s', run=name, path=h.sampler_last_path(), sampling_kernel_ms=r.kernel_ms, min_ess=float(ess.min()),
             median_ess=float(np.median(ess)), min_ess_per_s=float(ess.min() / s), median_ess_per_s=float(np.median(ess) / s),
             max_rhat=float(r.diagnostics['rhat'].max()), leapfrogs=r.total_tree_size)
    if OUT:
        os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
        with open(OUT, 'w') as f:
            json.dump(rows, f, indent=1)


if __name__ == '__main__':
    main()
