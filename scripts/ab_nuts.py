"""A/B kernel time of the headline NUTS launch for two builds of the library, alternating them in separate processes.

usage: ab_nuts.py OLD_LIB NEW_LIB [--rounds 3] [--warm 2] [--launches 5] [--timing]

Each round runs OLD then NEW, each in a process of its own (BFB200_LIB selects the library).  A process times the bench.py
step: the 4096-chain, 1500-iteration launch of the d = 26 cubic-2 workload with bench.py's inputs and seed, every output
written to device memory, the 256 MiB L2 flush before each launch, `--warm` untimed launches first, then `--launches` timed
ones (CUDA events around the kernel, bfb_last_kernel_ms).  Prints one JSON line per process and a summary line: median,
min / max of each build over all its timed launches, the relative change of the medians, and the GPU's name and power
limit.  --timing sets BFB200_DEBUG=1, so builds with -DBFB_DMMA_TIMING print their per-section cycles of a round."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def child(warm, launches):
    import numpy as np
    import torch
    import bayesfast_b200 as bfb
    from bayesfast_b200 import _cabi, synthetic
    from bench import N_DIM, ORDER, CHAINS_PER_GPU as C, N_ITER, N_WARMUP, SEED
    prob = synthetic.des_shaped(N_DIM, seed=1, n_chain=C, order=ORDER)
    sur = bfb.PolyModel(ORDER, input_size=N_DIM, output_size=1, device=0)
    sur.fit(prob['x_fit'], prob['y_fit'], logp=prob['y_fit'][:, 0])
    h = bfb.Density(sur)._sync(False)
    x0 = np.ascontiguousarray(prob['x_0'][:C])
    cfg = bfb.NTrace(n_chain=C, n_iter=N_ITER, n_warmup=N_WARMUP, x_0=x0, random_generator=SEED)._cfg_dict(SEED, 0)
    h.sampler_init(cfg, x0, 1. / N_DIM**0.25, np.ones(N_DIM), x0)
    S = C * N_ITER
    d_out = dict(samples=torch.empty(S * N_DIM, dtype=torch.float64, device='cuda:0'))
    for k in _cabi.FLOAT_STATS:
        d_out[k] = torch.empty(S, dtype=torch.float64, device='cuda:0')
    for k in _cabi.INT_STATS:
        d_out[k] = torch.empty(S, dtype=torch.int32, device='cuda:0')
    ptrs = {k: v.data_ptr() for k, v in d_out.items()}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda:0')
    ms, trees = [], set()
    for i in range(warm + launches):
        flush.zero_()
        torch.cuda.synchronize()
        h.sampler_reset()
        r = h.sampler_run('NUTS', N_ITER, out_ptrs=ptrs)
        h.synchronize()
        if i >= warm:
            ms.append(h.last_kernel_ms())
            trees.add(r['total_tree_size'])
    print(json.dumps(dict(lib=_cabi.LIB_PATH, path=h.sampler_last_path(), kernel_ms=ms, total_tree_size=sorted(trees))),
          flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('old')
    ap.add_argument('new')
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--warm', type=int, default=2)
    ap.add_argument('--launches', type=int, default=5)
    ap.add_argument('--timing', action='store_true')
    ap.add_argument('--child', action='store_true', help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:
        return child(a.warm, a.launches)
    import numpy as np
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                         capture_output=True, text=True).stdout.strip()
    res = {'old': [], 'new': []}
    trees = {'old': set(), 'new': set()}
    for rnd in range(a.rounds):
        for tag in ('old', 'new'):
            env = dict(os.environ, BFB200_LIB=os.path.abspath(getattr(a, tag)))
            if a.timing:
                env['BFB200_DEBUG'] = '1'
            p = subprocess.run([sys.executable, os.path.abspath(__file__), a.old, a.new, '--child', '--warm', str(a.warm),
                                '--launches', str(a.launches)], env=env, capture_output=True, text=True)
            if p.returncode != 0:
                sys.exit('%s build failed (round %d):\n%s' % (tag, rnd, p.stderr[-3000:]))
            line = json.loads(p.stdout.strip().splitlines()[-1])
            res[tag] += line['kernel_ms']
            trees[tag].update(line['total_tree_size'])
            print(json.dumps(dict(round=rnd, build=tag, **line)), flush=True)
            if a.timing:
                for ln in p.stderr.splitlines():
                    if 'cycles per' in ln:
                        print('%s round %d: %s' % (tag, rnd, ln), flush=True)
    med = {k: float(np.median(v)) for k, v in res.items()}
    print(json.dumps(dict(gpu=gpu, rounds=a.rounds, launches_per_process=a.launches,
                          old_ms=dict(median=med['old'], min=min(res['old']), max=max(res['old'])),
                          new_ms=dict(median=med['new'], min=min(res['new']), max=max(res['new'])),
                          change=med['new'] / med['old'] - 1.,
                          same_total_tree_size=trees['old'] == trees['new'], total_tree_size=sorted(trees['new']))))


if __name__ == '__main__':
    main()
