"""debug: tensor-core NUTS (BFB200_SAMPLER family, default dmma) vs oracle float differences per iteration"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import numpy as np
from oracle import bf_oracle
from bayesfast_b200 import _cabi
from _specs import synthetic_spec, to_device_spec
from test_gpu_sampler import cfg_from, device_draws
bf_oracle.build()
n, order, C, n_iter = 16, 'cubic-2', 70, 40
fam = sys.argv[1] if len(sys.argv) > 1 else 'dmma'
os.environ['BFB200_SAMPLER'] = fam
h = _cabi.Handle(0)
spec, cov = synthetic_spec(n, order, seed=70 + n)
spec['alpha'] = spec['alpha'] / 1.6 * 0.9
h.set_model(to_device_spec(spec))
x0 = (np.linalg.cholesky(cov) @ np.random.default_rng(8).normal(size=(n, C))).T
seed, chain0 = 777, 500
cfg = cfg_from({}, n_iter // 2, seed, chain0)
step0 = 1. / n**0.25
h.sampler_init(cfg, x0, step0, np.ones(n), x0)
out = h.sampler_run('NUTS', n_iter)
print(h.sampler_last_path())
st = h.sampler_state()
U, Z = device_draws(h, seed, st['n_draws'], chain0)
ref = bf_oracle.OracleDensity(spec).run('NUTS', dict(n_iter=n_iter, n_warmup=n_iter // 2), x0, step0, np.ones(n), draws_u=U, draws_z=Z)
for k in ('energy_change', 'energy', 'logp', 'max_energy_change', 'step_size'):
    d = np.abs(out[k] - ref[k]) / (1e-300 + np.maximum(1., np.abs(ref[k])))
    print(k, 'max rel diff per iteration', np.array2string(d.max(axis=0), precision=1, max_line_width=250))
    c = np.unravel_index(np.argmax(d), d.shape)
    print('   worst chain', c, out[k][c], ref[k][c], 'chain row', np.array2string(d[c[0]], precision=1, max_line_width=250))
d = np.abs(out['samples'] - ref['samples']).max(axis=2)
print('samples max abs diff per iteration', np.array2string(d.max(axis=0), precision=1, max_line_width=250))
