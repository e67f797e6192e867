"""HMC team kernel (8 chains per team of four warps) against the one-warp-per-group kernel: rates at d=26 cubic-2."""
import json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import bayesfast_b200 as bfb
from bayesfast_b200 import synthetic
n = 26
variants = [('team', {}), ('team', {'BFB200_TEAMS_PER_SM': '3'}), ('team', {'BFB200_TEAMS_PER_SM': '5'}), ('dmma', {})]
for C in (4096, 16384):
    prob = synthetic.des_shaped(n, seed=1, n_chain=C)
    sur = bfb.PolyModel('cubic-2', input_size=n, output_size=1)
    sur.fit(prob['x_fit'], prob['y_fit'], logp=prob['y_fit'][:, 0])
    den = bfb.Density(sur)
    h = den._sync(False)
    peak = h.fp64_peak(0)
    for fam, env in variants:
        for k in list(os.environ):
            if k.startswith('BFB200_'):
                del os.environ[k]
        os.environ['BFB200_SAMPLER'] = fam
        os.environ.update(env)
        cfg = bfb.HTrace(n_chain=C, n_iter=300, n_warmup=100, x_0=prob['x_0'], n_int_step=32)._cfg_dict(1, 0)
        h.sampler_init(cfg, prob['x_0'], 1. / n**0.25, np.ones(n), prob['x_0'])
        for k in (100, 200):
            r = h.sampler_run('HMC', k, fields=('tree_depth',))
            ms = h.last_kernel_ms()
            rate = r['total_tree_size'] / ms * 1e3
            print(json.dumps(dict(sampler='HMC', C=C, family=fam, env=env, iters=k, kernel=h.sampler_last_path(), ms=round(ms, 3),
                                  leapfrogs_per_s=rate, frac_fp64=round(rate * (8 * n * n + 24 * n) / 1e12 / peak, 4))), flush=True)
