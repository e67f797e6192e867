"""Split-R-hat and ESS on the device (csrc/bfb_diag.cu, bayesfast_b200.diagnostics, sample(diagnostics=True)) against the numpy
oracle, across input kinds and sampler paths, bit-identical where the same draws go through the same kernels, and over two ranks."""
import os

import numpy as np
import pytest

from _specs import to_device_spec, synthetic_spec, pack
from test_diagnostics_cpu import _ar1
from _diag_oracle import split_rhat_ess

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def handle():
    from bayesfast_b200 import _cabi
    h = _cabi.Handle(0)
    yield h
    h.close()


def _draws(M, N, n, seed):
    rng = np.random.default_rng(seed)
    if M * N * n > 10**7:                            # the headline shape: AR(1) chains with a different phi per coordinate
        return _ar1(rng, M, N, np.linspace(0.0, 0.95, n), n)
    x = _ar1(rng, M, N, np.linspace(0.1, 0.9, n), n)
    return x * np.linspace(0.5, 3., n) + rng.normal(size=(M, 1, n)) * 0.05 + np.arange(n)


@pytest.mark.parametrize('M,N,n', [(1, 9, 1), (3, 101, 5), (130, 333, 26), (37, 1000, 64), (4096, 1000, 26)])
def test_against_oracle(handle, M, N, n):
    import bayesfast_b200 as bfb
    x = _draws(M, N, n, seed=M + N + n)
    got = bfb.diagnostics(x[:, :, 0] if n == 1 else x, handle=handle)
    rhat, ess = split_rhat_ess(x)
    assert got['rhat'].shape == (n,) and got['ess'].shape == (n,)
    assert np.allclose(got['rhat'], rhat, rtol=1e-10, atol=0)
    assert np.allclose(got['ess'], ess, rtol=1e-9, atol=0)


def test_input_kinds_and_determinism(handle):
    import torch
    import bayesfast_b200 as bfb
    x = _draws(130, 333, 26, seed=3)
    x[5, 17, 4] = np.nan                             # a non-finite draw and a constant coordinate give nan, nothing else changes
    x[:, :, 9] = 1.5
    a = bfb.diagnostics(x, handle=handle)
    b = bfb.diagnostics(torch.from_numpy(x).cuda(), handle=handle)
    c = bfb.diagnostics(x, handle=handle)
    for k in ('rhat', 'ess'):
        assert np.array_equal(a[k], b[k], equal_nan=True) and np.array_equal(a[k], c[k], equal_nan=True)
        assert np.isnan(a[k][4]) and np.isnan(a[k][9]) and np.isfinite(np.delete(a[k], [4, 9])).all()
    rhat, ess = split_rhat_ess(x)
    assert np.allclose(a['rhat'], rhat, rtol=1e-10, equal_nan=True) and np.allclose(a['ess'], ess, rtol=1e-9, equal_nan=True)
    with pytest.raises(ValueError):
        bfb.diagnostics(torch.zeros((4, 3, 2), dtype=torch.float64, device='cuda'), handle=handle)


def test_headline_shape():
    """d = 26 cubic-2, 4096 chains, 1500 iterations: the diagnostics of the single-launch run equal those of its host samples, the
    run's outputs do not change, and a run that brings nothing back (fields=(), thin=10) computes the same diagnostics"""
    import bayesfast_b200 as bfb
    from bayesfast_b200 import synthetic
    n, C = 26, 4096
    prob = synthetic.des_shaped(n, seed=1, n_chain=C, order='cubic-2')
    sur = bfb.PolyModel('cubic-2', input_size=n, output_size=1)
    sur.fit(prob['x_fit'], prob['y_fit'], logp=prob['y_fit'][:, 0])
    den = bfb.Density(sur)
    kw = dict(n_chain=C, n_iter=1500, n_warmup=500, x_0=prob['x_0'], random_generator=7)
    base = bfb.sample(den, dict(kw), verbose=False, keep='post_warmup')
    tt = bfb.sample(den, dict(kw), verbose=False, keep='post_warmup', diagnostics=True)
    assert base.diagnostics is None
    assert set(tt.arrays) == set(base.arrays)
    for k in base.arrays:
        assert np.array_equal(tt.arrays[k], base.arrays[k]), k
    assert tt.total_tree_size == base.total_tree_size
    d = bfb.diagnostics(tt.samples)
    for k in ('rhat', 'ess'):
        assert np.array_equal(tt.diagnostics[k], d[k]), k
    red = bfb.sample(den, dict(kw), verbose=False, keep='post_warmup', fields=(), thin=10, diagnostics=True)
    for k in ('rhat', 'ess'):
        assert np.array_equal(red.diagnostics[k], d[k]), k
    assert np.all(d['rhat'] < 1.05) and np.all(d['ess'] > 0.01 * C * 1000)


def _small_density(n=9):
    import bayesfast_b200 as bfb
    spec, cov = synthetic_spec(n, 'cubic-2', seed=14)
    sur = bfb.PolyModel('cubic-2', input_size=n, output_size=1)
    for conf, cf in zip(sur.configs, spec['configs']):
        conf._set(pack(cf['order'], cf['coef'][0], n), 0)
    sur._mu, sur._hess, sur._alpha, sur._f_mu = spec['mu'], spec['hess'], spec['alpha'], spec['f_mu']
    return bfb.Density(sur), cov


def _small_trace(cov, n=9, C=50, n_iter=173, n_warmup=61):
    x0 = (np.linalg.cholesky(cov) @ np.random.default_rng(1).normal(size=(n, C))).T
    return dict(n_chain=C, n_iter=n_iter, n_warmup=n_warmup, x_0=x0, random_generator=11)


@pytest.mark.parametrize('sampler,extra,out', [('NUTS', {}, dict(keep='all')),
                                               ('NUTS', {}, dict(keep='post_warmup', thin=3, summaries=True)),
                                               ('HMC', {'n_int_step': 5}, dict(keep='all')),
                                               ('HMC', {'n_int_step': 5}, dict(keep='post_warmup', fields=('logp',))),
                                               ('NUTS', {'metric': 'full'}, dict(keep='all')),
                                               ('NUTS', {'metric': 'full'}, dict(keep='post_warmup', thin=2))])
def test_sampler_paths(sampler, extra, out):
    """every path of bfb_sampler_run_ex (single launch, chunked launches, HMC, dense metric, thinning, fields without samples):
    the diagnostics cover the post-warm-up iterations only and equal those of the full run's samples"""
    import bayesfast_b200 as bfb
    den, cov = _small_density()
    kw = dict(_small_trace(cov), **extra)
    full = bfb.sample(den, dict(kw), sampler=sampler, verbose=False)
    post = full.samples[:, 61:]
    ref = bfb.diagnostics(post)
    tt = bfb.sample(den, dict(kw), sampler=sampler, verbose=False, diagnostics=True, **out)
    for k in ('rhat', 'ess'):
        assert np.array_equal(tt.diagnostics[k], ref[k]), k
    rhat, ess = split_rhat_ess(post)
    assert np.allclose(ref['rhat'], rhat, rtol=1e-10) and np.allclose(ref['ess'], ess, rtol=1e-9)
    if out.get('keep') == 'all' and 'thin' not in out:
        assert np.array_equal(tt.samples, full.samples)


def test_continue_and_short_runs():
    import bayesfast_b200 as bfb
    den, cov = _small_density()
    kw = _small_trace(cov)
    full = bfb.sample(den, dict(kw), verbose=False)
    with pytest.raises(ValueError):                  # 2 post-warm-up iterations
        bfb.sample(den, dict(kw), n_run=63, verbose=False, diagnostics=True)
    a = bfb.sample(den, dict(kw), n_run=100, verbose=False, keep='post_warmup', diagnostics=True)
    b = bfb.sample(den, a, n_run=73, verbose=False)
    for k in ('rhat', 'ess'):
        assert np.array_equal(a.diagnostics[k], bfb.diagnostics(full.samples[:, 61:100])[k])
        assert np.array_equal(b.diagnostics[k], bfb.diagnostics(full.samples[:, 100:173])[k])
    with pytest.raises(NotImplementedError):
        bfb.sample(den, bfb.TNTrace(den, 0., **kw), verbose=False, diagnostics=True)


def test_gaussian_target_means_within_measured_ess(handle):
    """the quadratic surrogate of test_full_size_posterior_moments (26-d Gaussian, 4096 chains): R-hat < 1.01 everywhere, and the
    posterior mean is within 5 sd / sqrt(ESS) of the truth with the ESS the device measured"""
    from bayesfast_b200 import diag
    from test_gpu_sampler import cfg_from
    n, C = 26, 4096
    spec, cov = synthetic_spec(n, 'quadratic', seed=11, bound=False)
    mean = cov @ spec['configs'][0]['coef'][0, 1:]
    handle.set_model(to_device_spec(spec))
    x0 = np.random.default_rng(0).normal(size=(C, n))
    handle.sampler_init(cfg_from({}, 150, 2024), x0, 1. / n**0.25, np.ones(n), x0)
    out = handle.sampler_run('NUTS', 250, fields=('samples',), diag_from=150)
    d = diag.finish(out['diag_partials'])
    post = out['samples'][:, 150:]
    assert np.array_equal(d['ess'], diag.diagnostics(post, handle=handle)['ess'])
    assert np.all(d['rhat'] < 1.01)
    sd = np.sqrt(np.diag(cov))
    assert np.all(np.abs(post.reshape(-1, n).mean(axis=0) - mean) < 5. * sd / np.sqrt(d['ess']))


def _two_rank_worker(rank, world, port, q):
    import sys
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    import torch.distributed as dist
    os.environ['MASTER_ADDR'], os.environ['MASTER_PORT'] = '127.0.0.1', str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)        # two ranks share cuda:0
    import bayesfast_b200 as bfb
    from test_gpu_diagnostics import _small_density, _small_trace
    den, cov = _small_density()
    tt = bfb.sample(den, _small_trace(cov), verbose=False, comm=True, keep='post_warmup', diagnostics=True)
    q.put((rank, tt.diagnostics['rhat'], tt.diagnostics['ess'], tt.samples.shape[0]))
    dist.barrier()
    dist.destroy_process_group()


def test_two_ranks_sharing_one_gpu():
    import torch.multiprocessing as mp
    import bayesfast_b200 as bfb
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 33700 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_two_rank_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=300) for _ in procs], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert res[0][3] == 25 and res[1][3] == 25
    assert np.array_equal(res[0][1], res[1][1]) and np.array_equal(res[0][2], res[1][2])
    den, cov = _small_density()
    one = bfb.sample(den, _small_trace(cov), verbose=False, keep='post_warmup', diagnostics=True)
    assert np.allclose(res[0][1], one.diagnostics['rhat'], rtol=1e-12, atol=0)
    assert np.allclose(res[0][2], one.diagnostics['ess'], rtol=1e-12, atol=0)
