"""GPU parity of the lock-step NUTS / HMC kernels vs golden runs of the real reference and vs the oracle."""
import numpy as np
import pytest

import _golden_io as gio
from _specs import to_device_spec, synthetic_spec

pytestmark = pytest.mark.gpu

INT_STATS = ('tree_depth', 'tree_size', 'diverging')
FLT_STATS = ('logp', 'energy', 'mean_tree_accept', 'step_size', 'step_size_bar', 'energy_change', 'max_energy_change')
# floats: tight over the first EARLY iterations, loose later (chaotic amplification of rounding differences through
# step-size / metric adaptation, see tests/test_oracle_golden.py); integer outcomes must be identical throughout.
EARLY, EARLY_TOL, LATE_TOL = 8, 1e-9, 1e-3


def cfg_from(kw, n_warmup, seed, chain0=0):
    d = dict(n_warmup=n_warmup, max_treedepth=10, n_int_step=0, max_change=1000., adapt_step_size=1,
             target_accept=0.8, gamma=0.05, k=0.75, t0=10., adapt_metric=1, initial_weight=10., adapt_window=60,
             update_window=1, doubling=1, seed=seed, chain0=chain0)
    for k, v in kw.items():
        if k in d:
            d[k] = type(d[k])(v)
    return d


@pytest.fixture(scope='module')
def handle():
    from bayesfast_b200 import _cabi
    h = _cabi.Handle(0)
    yield h
    h.close()


def device_draws(handle, seed, n_draws, chain0=0):
    nmax = int(max(n_draws)) + 8
    U = np.zeros((len(n_draws), nmax))
    Z = np.zeros((len(n_draws), nmax))
    for c in range(len(n_draws)):
        U[c], Z[c] = handle.rng_fill(seed, chain0 + c, 0, nmax)
    return U, Z


def check_floats(a, b, tag, late=LATE_TOL):
    assert np.allclose(a[:, :EARLY], b[:, :EARLY], rtol=EARLY_TOL, atol=EARLY_TOL, equal_nan=True), tag
    assert np.allclose(a, b, rtol=late, atol=late, equal_nan=True), tag


@pytest.mark.parametrize('case', gio.load('sampler.npz')['cases'] + gio.load('sampler_d26.npz')['cases'], ids=lambda c: c['name'])
def test_golden_chains(handle, oracle, case):
    """same seeds and draw stream as the recorded runs of the real reference"""
    r, kw = case['result'], case['trace_kw']
    n_iter, n_warmup = int(kw['n_iter']), int(kw['n_warmup'])
    handle.set_model(to_device_spec(case['spec']))
    cfg = cfg_from(kw, n_warmup, int(case['seed']))
    handle.sampler_init(cfg, case['x0'], float(r['step0']), r['var0'], case['x0'])
    out = handle.sampler_run(case['sampler'], n_iter)
    st = handle.sampler_state()
    assert np.all(st['status'] == 0)
    assert np.array_equal(st['n_draws'], r['n_draws'])
    if case['sampler'] == 'NUTS':
        for k in INT_STATS:
            assert np.array_equal(out[k], r[k].astype(np.int32)), k
        for k in FLT_STATS:
            check_floats(out[k], r[k], k)
        assert out['total_tree_size'] == int(r['tree_size'].sum())
    else:
        assert np.array_equal(out['tree_depth'], r['accepted'].astype(np.int32))
        assert np.array_equal(out['diverging'], r['diverging'].astype(np.int32))
        for k, k2 in (('logp', 'logp'), ('energy', 'energy'), ('mean_tree_accept', 'accept_stat'),
                      ('step_size', 'step_size'), ('energy_change', 'energy_change')):
            check_floats(out[k], r[k2], k)
    check_floats(out['samples'], r['samples'], 'samples')
    assert np.allclose(st['final_step'], r['final_step'], rtol=LATE_TOL)
    assert np.allclose(st['final_var'], r['final_var'], rtol=LATE_TOL)


@pytest.mark.parametrize('n,order,C,n_iter', [(26, 'cubic-2', 256, 40), (16, 'cubic-2', 130, 40), (40, 'cubic-3', 6, 12),
                                               (2, 'quadratic', 64, 60), (64, 'cubic-3', 64, 20)])
def test_teacher_forced_vs_oracle(handle, oracle, n, order, C, n_iter):
    """per-chain tree depths / sizes / divergences identical to the oracle fed with the device's own draws"""
    spec, cov = synthetic_spec(n, order, seed=7 + n, decay=True)
    handle.set_model(to_device_spec(spec))
    rng = np.random.default_rng(5)
    x0 = (np.linalg.cholesky(cov) @ rng.normal(size=(n, C))).T
    seed, chain0 = 4242, 1000
    cfg = cfg_from({}, n_iter // 2, seed, chain0)
    step0 = 1. / n**0.25
    handle.sampler_init(cfg, x0, step0, np.ones(n), x0)
    out = handle.sampler_run('NUTS', n_iter)
    st = handle.sampler_state()
    assert np.all(st['status'] == 0)
    U, Z = device_draws(handle, seed, st['n_draws'], chain0)
    ref = oracle.OracleDensity(spec).run('NUTS', dict(n_iter=n_iter, n_warmup=n_iter // 2), x0, step0, np.ones(n),
                                         draws_u=U, draws_z=Z)
    assert np.all(ref['status'] == 0)
    assert np.array_equal(st['n_draws'], ref['n_draws'])
    for k in INT_STATS:
        assert np.array_equal(out[k], ref[k]), k
    check_floats(out['samples'], ref['samples'], 'samples')
    assert out['total_tree_size'] == int(ref['tree_size'].sum())


def test_hmc_vs_oracle(handle, oracle):
    n, C, n_iter = 12, 64, 40
    spec, cov = synthetic_spec(n, 'cubic-2', seed=3)
    handle.set_model(to_device_spec(spec))
    x0 = (np.linalg.cholesky(cov) @ np.random.default_rng(2).normal(size=(n, C))).T
    cfg = cfg_from({'n_int_step': 12}, 20, 77)
    handle.sampler_init(cfg, x0, 0.5, np.ones(n), x0)
    out = handle.sampler_run('HMC', n_iter)
    st = handle.sampler_state()
    U, Z = device_draws(handle, 77, st['n_draws'])
    ref = oracle.OracleDensity(spec).run('HMC', dict(n_iter=n_iter, n_warmup=20, n_int_step=12), x0, 0.5, np.ones(n),
                                         draws_u=U, draws_z=Z)
    assert np.array_equal(out['tree_depth'], ref['tree_depth'])
    assert np.array_equal(out['diverging'], ref['diverging'])
    check_floats(out['samples'], ref['samples'], 'samples')


def test_full_size_posterior_moments(handle):
    """BASELINE config shape (d=26 cubic-2, 4096 chains): size-independent checks on a pure Gaussian surrogate
    whose posterior is known exactly: mean / variance within Monte Carlo error, no divergences after warm-up,
    chains are reproducible (same seed -> same bits) and independent of how they are batched."""
    n, C = 26, 4096
    spec, cov = synthetic_spec(n, 'quadratic', seed=11, bound=False)
    lin = spec['configs'][0]['coef'][0, 1:]
    mean = cov @ lin
    handle.set_model(to_device_spec(spec))
    x0 = np.random.default_rng(0).normal(size=(C, n))
    cfg = cfg_from({}, 150, 2024)
    handle.sampler_init(cfg, x0, 1. / n**0.25, np.ones(n), x0)
    out = handle.sampler_run('NUTS', 250)
    post = out['samples'][:, 150:].reshape(-1, n)
    sd = np.sqrt(np.diag(cov))
    ess = post.shape[0] / 4.
    assert np.all(np.abs(post.mean(axis=0) - mean) < 6. * sd / np.sqrt(ess))
    assert np.all(np.abs(post.var(axis=0) / np.diag(cov) - 1.) < 0.05)
    assert out['diverging'][:, 150:].sum() == 0
    assert np.all(out['tree_size'] <= 2 ** out['tree_depth'] - 1) and np.all(out['tree_size'] >= 2 ** (out['tree_depth'] - 1))
    # reproducibility + batching independence: chains 100..163 alone, with chain0 = 100
    cfg2 = cfg_from({}, 150, 2024, chain0=100)
    handle.sampler_init(cfg2, x0[100:164], 1. / n**0.25, np.ones(n), x0[100:164])
    out2 = handle.sampler_run('NUTS', 250, fields=('samples', 'tree_depth'))
    assert np.array_equal(out2['samples'], out['samples'][100:164])
    assert np.array_equal(out2['tree_depth'], out['tree_depth'][100:164])


def test_sample_api(oracle):
    import bayesfast_b200 as bfb
    n = 6
    spec, cov = synthetic_spec(n, 'cubic-2', seed=4, decay=True, transform=True)
    sur = bfb.PolyModel('cubic-2', input_size=n, output_size=1)
    from _specs import pack
    for conf, cf in zip(sur.configs, spec['configs']):
        conf._set(pack(cf['order'], cf['coef'][0], n), 0)
    sur._mu, sur._hess, sur._alpha, sur._f_mu = spec['mu'], spec['hess'], spec['alpha'], spec['f_mu']
    den = bfb.Density(sur, input_scales=spec['transform_ranges'], hard_bounds=spec['hard_bounds'],
                      decay_options=dict(use_decay=True, alpha=float(np.sqrt(spec['d_alpha2'])), alpha_p=None))
    den._mu, den._hess = spec['d_mu'], spec['d_hess']
    x0 = (np.linalg.cholesky(cov) @ np.random.default_rng(1).normal(size=(n, 16))).T * 0.5
    tt = bfb.sample(den, dict(n_chain=16, n_iter=60, n_warmup=30, x_0=x0, random_generator=5), verbose=False)
    assert tt.n_chain == 16 and tt.samples.shape == (16, 60, n)
    t3 = tt[3]
    assert isinstance(t3, bfb.NTrace) and t3.chain_id == 3 and t3.samples.shape == (60, n)
    assert len(t3.stats._tree_depth) == 60 and t3.stats.n_warmup == 30
    assert tt.get().shape == (16 * 30, n)
    assert np.allclose(t3.samples_original, den.to_original(t3.samples))
    assert t3.n_call == int(np.sum(t3.stats._tree_size[1:])) + 60 + 1
    # vs the oracle with the same stream
    od = oracle.OracleDensity(den.to_spec())
    U, Z = device_draws(den._sync(False), 5, tt._final['n_draws'])
    ref = od.run('NUTS', dict(n_iter=60, n_warmup=30), den.from_original(x0), 1. / n**0.25, np.ones(n), draws_u=U, draws_z=Z)
    assert np.array_equal(tt.arrays['tree_depth'], ref['tree_depth'])
    # resume: the chains are still resident (sample.py:91-98)
    tt2 = bfb.sample(den, tt, n_run=10, verbose=False)
    assert tt2.samples.shape == (16, 70, n) and np.array_equal(tt2.samples[:, :60], tt.samples)
    ref70 = od.run('NUTS', dict(n_iter=70, n_warmup=30), den.from_original(x0), 1. / n**0.25, np.ones(n), draws_u=U, draws_z=Z) \
        if U.shape[1] >= int(tt2._final['n_draws'].max()) else None
    if ref70 is not None:
        assert np.array_equal(tt2.arrays['tree_depth'], ref70['tree_depth'])
    # dense mass matrix through the same API (sample_trace.py:430-431, 445-449): identity start, adapted covariance back
    ttf = bfb.sample(den, dict(n_chain=16, n_iter=60, n_warmup=30, x_0=x0, random_generator=5, metric='full'), verbose=False)
    assert isinstance(ttf[2].metric, bfb.sample_trace.QuadMetricFullAdapt) and ttf[2].metric._cov.shape == (n, n)
    U, Z = device_draws(den._sync(False), 5, ttf._final['n_draws'])
    reff = od.run('NUTS', dict(n_iter=60, n_warmup=30, dense_metric=1), den.from_original(x0), 1. / n**0.25, np.eye(n),
                  draws_u=U, draws_z=Z)
    assert np.array_equal(ttf.arrays['tree_depth'], reff['tree_depth'])
    assert np.allclose(ttf._final['final_var'], reff['final_var'], rtol=1e-3, atol=1e-3 * np.abs(reff['final_var']).max())
    assert bfb.sample_trace._get_metric(ttf, 'full', from_samples=False).shape == (n, n)
    # other chains were started on this density since: the first run cannot be continued any more
    with pytest.raises(RuntimeError):
        bfb.sample(den, tt2, n_run=10, verbose=False)
    # errors surface like the reference's (base_hmc.py:42-46)
    bad = x0.copy()
    bad[2] = np.nan
    with pytest.raises(ValueError):
        bfb.sample(den, dict(n_chain=16, n_iter=20, n_warmup=10, x_0=bad, random_generator=5), verbose=False)


def test_sample_reduced_outputs():
    """sample(keep='post_warmup', thin=k, summaries=True): warm-up records never leave the device, thinned records are the
    same numbers as in the full run, mean / covariance over ALL post-warm-up samples are accumulated on the device
    (SampleTrace.get, sample_trace.py:762-787, only ever hands out post-warm-up samples)"""
    import bayesfast_b200 as bfb
    n, C, n_iter, n_warmup = 9, 50, 173, 61
    spec, cov = synthetic_spec(n, 'cubic-2', seed=14)
    sur = bfb.PolyModel('cubic-2', input_size=n, output_size=1)
    from _specs import pack
    for conf, cf in zip(sur.configs, spec['configs']):
        conf._set(pack(cf['order'], cf['coef'][0], n), 0)
    sur._mu, sur._hess, sur._alpha, sur._f_mu = spec['mu'], spec['hess'], spec['alpha'], spec['f_mu']
    den = bfb.Density(sur)
    x0 = (np.linalg.cholesky(cov) @ np.random.default_rng(1).normal(size=(n, C))).T
    kw = dict(n_chain=C, n_iter=n_iter, n_warmup=n_warmup, x_0=x0, random_generator=11)
    full = bfb.sample(den, dict(kw), verbose=False)
    for sampler, thin in (('NUTS', 3), ('NUTS', 1), ('HMC', 4)):
        if sampler == 'HMC':
            full = bfb.sample(den, dict(kw, n_int_step=5), sampler='HMC', verbose=False)
        red = bfb.sample(den, dict(kw, **({'n_int_step': 5} if sampler == 'HMC' else {})), sampler=sampler, verbose=False,
                         keep='post_warmup', thin=thin, summaries=True)
        sel = np.arange(n_warmup, n_iter, thin)
        assert np.array_equal(red.iters, sel) and red.i_iter == n_iter
        for k in ('samples', 'logp', 'energy', 'tree_depth', 'tree_size', 'diverging', 'step_size'):
            assert np.array_equal(red.arrays[k], full.arrays[k][:, sel]), (sampler, thin, k)
        assert red.total_tree_size == full.total_tree_size
        post = full.samples[:, n_warmup:].reshape(-1, n)
        assert np.allclose(red.summaries['mean'], post.mean(axis=0), rtol=1e-11, atol=1e-12)
        assert np.allclose(red.summaries['cov'], np.cov(post, rowvar=False), rtol=1e-10, atol=1e-13)
        assert np.array_equal(red.get(), full.get()[:: 1].reshape(C, -1, n)[:, ::thin].reshape(-1, n))
        assert red[2].samples.shape == (len(sel), n) and not red[2].stats._warmup.any()
    # a run that ends inside the warm-up brings back nothing, and continues into the kept part
    a = bfb.sample(den, dict(kw), n_run=40, verbose=False, keep='post_warmup', thin=2, fields=('samples', 'logp', 'tree_size'))
    assert a.samples.shape == (C, 0, n) and a.i_iter == 40
    b = bfb.sample(den, a, n_run=60, verbose=False)
    full = bfb.sample(den, dict(kw), verbose=False)
    sel = np.arange(n_warmup, 100, 2)
    assert np.array_equal(b.iters, sel) and np.array_equal(b.samples, full.samples[:, sel]) and b.i_iter == 100
    assert set(b.arrays) == {'samples', 'logp', 'tree_size', 'samples_original', 'logp_original'}
    # ... but `b` cannot be continued any more: other chains were started on the density since
    with pytest.raises(RuntimeError):
        bfb.sample(den, b, n_run=5, verbose=False)


def test_single_launch_host_outputs_match_chunked_launches(handle, monkeypatch):
    """bfb_sampler_run_ex with host outputs: ONE launch whose finished iteration chunks the host copies out while the kernel goes on
    (progress word in mapped pinned memory) against the chunked launches through staging buffers -- same records, bit for bit,
    for full and post-warm-up outputs, ragged chunk counts and a field subset"""
    n, C, n_iter = 26, 203, 150
    spec, cov = synthetic_spec(n, 'cubic-2', seed=21)
    handle.set_model(to_device_spec(spec))
    x0 = (np.linalg.cholesky(cov) @ np.random.default_rng(9).normal(size=(n, C))).T
    cfg = cfg_from({}, 60, 17)
    runs = {}
    for name, env, kw in (('multi', {'BFB200_E2E_MULTI_LAUNCH': '1'}, {}), ('single', {}, {}), ('single7', {'BFB200_E2E_CHUNKS': '7'}, {}),
                          ('multi_post', {'BFB200_E2E_MULTI_LAUNCH': '1'}, dict(skip=60)), ('single_post', {'BFB200_E2E_CHUNKS': '100'}, dict(skip=60)),
                          ('single_sub', {}, dict(fields=('samples', 'tree_depth')))):
        for k in ('BFB200_E2E_MULTI_LAUNCH', 'BFB200_E2E_CHUNKS'):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        handle.sampler_init(cfg, x0, 1. / n**0.25, np.ones(n), x0)
        runs[name] = handle.sampler_run('NUTS', n_iter, **kw)
        assert handle.sampler_last_path() == 'dmma'
        assert np.all(handle.sampler_state()['status'] == 0)
    for a, b in (('single', 'multi'), ('single7', 'multi'), ('single_post', 'multi_post')):
        for k, v in runs[b].items():
            assert np.array_equal(np.asarray(runs[a][k]), np.asarray(v)), (a, k)
    for k in ('samples', 'tree_depth'):
        assert np.array_equal(runs['single_sub'][k], runs['multi'][k]), k
    assert np.array_equal(runs['single_post']['samples'], runs['multi']['samples'][:, 60:])


def test_work_queue_chunking_is_invisible(handle, monkeypatch):
    """the fast path cuts a launch into (chain-group, iteration-chunk) work units handed out by an atomic queue;
    results must not depend on the chunk length (chain state is carried through global memory between units)"""
    n, C, n_iter = 26, 96, 48
    spec, cov = synthetic_spec(n, 'cubic-2', seed=33)
    handle.set_model(to_device_spec(spec))
    x0 = (np.linalg.cholesky(cov) @ np.random.default_rng(5).normal(size=(n, C))).T
    cfg = cfg_from({}, n_iter // 2, 99)
    outs = []
    for chunk in (str(n_iter), '16', '5'):
        monkeypatch.setenv('BFB200_CHUNK_ITERS', chunk)
        handle.sampler_init(cfg, x0, 1. / n**0.25, np.ones(n), x0)
        outs.append(handle.sampler_run('NUTS', n_iter))
    for o in outs[1:]:
        for k in ('samples', 'tree_depth', 'tree_size', 'step_size', 'energy'):
            assert np.array_equal(o[k], outs[0][k]), k


# n, order, chains, iterations, environment of the one-warp (dmma) and pair kernels (n <= 32) ...
NUTS_CASES = [
    (26, 'cubic-2', 203, 40, {}),                                  # ragged: 203 = 25 groups of 8 + 3 chains
    (26, 'cubic-2', 203, 40, {'BFB200_WARPS_PER_SM': '8'}),        # the 8-warps-per-SM launch used above 4736 chains
    (26, 'cubic-2', 64, 48, {'BFB200_STACK_LEVELS_SMEM': '1', 'BFB200_CHUNK_ITERS': '7'}),   # deep stack levels in L2, odd chunks
    (16, 'cubic-2', 70, 40, {}),
    (31, 'cubic-2', 40, 30, {}),
    (5, 'cubic-2', 50, 40, {}),
    (26, 'quadratic', 100, 40, {}),
    (26, 'cubic-2', 203, 40, {'BFB200_STACK_LEVELS_SMEM': '0'}),
    (16, 'quadratic', 33, 40, {'BFB200_CHUNK_ITERS': '9'}),
]
# ... and of the team kernel (32 < n <= 64)
TEAM_NUTS_CASES = [
    (40, 'cubic-2', 203, 40, {}),
    (40, 'cubic-2', 64, 48, {'BFB200_STACK_LEVELS_SMEM': '1', 'BFB200_CHUNK_ITERS': '7'}),
    (48, 'cubic-2', 70, 40, {}),
    (64, 'cubic-2', 40, 30, {}),
    (33, 'cubic-2', 50, 40, {}),
    (40, 'quadratic', 100, 40, {}),
    (40, 'cubic-2', 203, 40, {'BFB200_STACK_LEVELS_SMEM': '0'}),
    (56, 'quadratic', 33, 40, {'BFB200_CHUNK_ITERS': '9'}),
    (40, 'cubic-3', 21, 24, {'BFB200_STACK_LEVELS_SMEM': '2'}),
]


@pytest.mark.parametrize('family,n,order,C,n_iter,env', [
    pytest.param(f, *c, id='%s-%d-%s-%d-%d-env%d' % (f, c[0], c[1], c[2], c[3], i))
    for f, cases in (('dmma', NUTS_CASES), ('pair', NUTS_CASES), ('team', TEAM_NUTS_CASES)) for i, c in enumerate(cases)])
def test_tensor_core_nuts_vs_oracle(handle, oracle, monkeypatch, n, order, C, n_iter, env, family):
    """bfb_sampler_dmma.cu (8 chains per warp) / bfb_sampler_pair.cu (integrator warp + tree warp per 8 chains, speculative
    trajectory) / bfb_sampler_team.cu (8 chains per team of four warps, 32 < n <= 64), the chains as the rows of FP64 DMMAs:
    per-chain tree depths / sizes / divergences and draw counts identical to the oracle fed with the device's own draws, and
    to the generic warp-per-chain kernel"""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    monkeypatch.setenv('BFB200_SAMPLER', family)
    spec, cov = synthetic_spec(n, order, seed=70 + n)              # radial bound, no decay / transform: the headline shape
    spec['alpha'] = spec['alpha'] / 1.6 * 0.9                      # tight bound: many leapfrogs leave the ellipsoid
    handle.set_model(to_device_spec(spec))
    x0 = (np.linalg.cholesky(cov) @ np.random.default_rng(8).normal(size=(n, C))).T
    seed, chain0 = 777, 500
    cfg = cfg_from({}, n_iter // 2, seed, chain0)
    step0 = 1. / n**0.25
    handle.sampler_init(cfg, x0, step0, np.ones(n), x0)
    out = handle.sampler_run('NUTS', n_iter)
    assert handle.sampler_last_path() == family
    st = handle.sampler_state()
    assert np.all(st['status'] == 0)
    U, Z = device_draws(handle, seed, st['n_draws'], chain0)
    ref = oracle.OracleDensity(spec).run('NUTS', dict(n_iter=n_iter, n_warmup=n_iter // 2), x0, step0, np.ones(n),
                                         draws_u=U, draws_z=Z)
    assert np.array_equal(st['n_draws'], ref['n_draws'])
    for k in INT_STATS:
        assert np.array_equal(out[k], ref[k]), k
    # late tolerance: with the tight bound single chains amplify rounding differences ~10x every two iterations (scripts/
    # team_debug.py: 1e-15 at iteration 1, 1e-9 at 10, 1e-3 at 18 for BOTH kernel families against the oracle, which sums in
    # a third order); the decisions above must agree regardless
    for k in FLT_STATS:
        check_floats(out[k], ref[k], k, late=5e-3)
    check_floats(out['samples'], ref['samples'], 'samples', late=5e-3)
    assert out['total_tree_size'] == int(ref['tree_size'].sum())
    assert np.allclose(st['final_var'], ref['final_var'], rtol=5e-3)
    # same run on the generic kernel
    monkeypatch.setenv('BFB200_SAMPLER', 'generic')
    handle.sampler_init(cfg, x0, step0, np.ones(n), x0)
    gen = handle.sampler_run('NUTS', n_iter)
    assert handle.sampler_last_path() == 'generic'
    for k in INT_STATS:
        assert np.array_equal(out[k], gen[k]), k


@pytest.mark.parametrize('family,n,C', [('dmma', 26, 96), ('pair', 26, 96), ('team', 40, 101)],    # 101 chains: a ragged group
                         ids=['dmma', 'pair', 'team-n40'])
def test_tensor_core_nuts_resume_and_reset(handle, monkeypatch, family, n, C):
    """chain state survives between launches (bfb_sampler_run called twice == once), and bfb_sampler_reset restarts it"""
    monkeypatch.setenv('BFB200_SAMPLER', family)
    spec, cov = synthetic_spec(n, 'cubic-2', seed=12)
    handle.set_model(to_device_spec(spec))
    x0 = (np.linalg.cholesky(cov) @ np.random.default_rng(3).normal(size=(n, C))).T
    cfg = cfg_from({}, 30, 31)
    handle.sampler_init(cfg, x0, 1. / n**0.25, np.ones(n), x0)
    a = handle.sampler_run('NUTS', 50)
    assert handle.sampler_last_path() == family
    handle.sampler_reset()
    b1 = handle.sampler_run('NUTS', 20)
    b2 = handle.sampler_run('NUTS', 30)
    for k in ('samples', 'tree_depth', 'energy', 'step_size'):
        assert np.array_equal(np.concatenate([b1[k], b2[k]], axis=1), a[k]), k


@pytest.mark.parametrize('family', ['team', 'dmma'])
@pytest.mark.parametrize('n,order,C,env', [(26, 'cubic-2', 100, {}), (26, 'cubic-2', 100, {'BFB200_WARPS_PER_SM': '8', 'BFB200_TEAMS_PER_SM': '3', 'BFB200_CHUNK_ITERS': '7'}),
                                           (12, 'cubic-2', 37, {}), (30, 'quadratic', 24, {})])
def test_tensor_core_hmc_vs_oracle(handle, oracle, monkeypatch, n, order, C, env, family):
    """hmc_team_kernel (8 chains per team of four warps) / hmc_dmma_kernel (8 chains per warp), lock-step HMC on FP64 DMMA, vs
    the oracle fed with the device's draws and vs the generic kernel: accept / divergence decisions identical, states
    within rounding"""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    monkeypatch.setenv('BFB200_SAMPLER', family)
    n_iter = 40
    spec, cov = synthetic_spec(n, order, seed=90 + n)
    spec['alpha'] = spec['alpha'] / 1.6
    handle.set_model(to_device_spec(spec))
    x0 = (np.linalg.cholesky(cov) @ np.random.default_rng(2).normal(size=(n, C))).T
    cfg = cfg_from({'n_int_step': 12}, 20, 77, chain0=9)
    handle.sampler_init(cfg, x0, 0.5, np.ones(n), x0)
    out = handle.sampler_run('HMC', n_iter)
    assert handle.sampler_last_path() == family
    st = handle.sampler_state()
    assert np.all(st['status'] == 0)
    U, Z = device_draws(handle, 77, st['n_draws'], 9)
    ref = oracle.OracleDensity(spec).run('HMC', dict(n_iter=n_iter, n_warmup=20, n_int_step=12), x0, 0.5, np.ones(n),
                                         draws_u=U, draws_z=Z)
    assert np.array_equal(st['n_draws'], ref['n_draws'])
    assert np.array_equal(out['tree_depth'], ref['tree_depth'])
    assert np.array_equal(out['diverging'], ref['diverging'])
    # the tight bound makes these trajectories chaotic (rounding differences grow ~10x every two iterations, for the generic
    # kernel too: scripts/hmc_debug.py), so the late tolerance is looser than for the NUTS cases; decisions must still agree
    check_floats(out['samples'], ref['samples'], 'samples', late=1e-2)
    ok = ref['diverging'] == 0                      # the end state of a divergent trajectory is chaotic: only its verdict is compared
    check_floats(np.where(ok, out['energy'], 0.), np.where(ok, ref['energy'], 0.), 'energy', late=1e-2)
    assert out['total_tree_size'] == C * n_iter * 12
    monkeypatch.setenv('BFB200_SAMPLER', 'generic')
    handle.sampler_init(cfg, x0, 0.5, np.ones(n), x0)
    gen = handle.sampler_run('HMC', n_iter)
    assert handle.sampler_last_path() == 'generic'
    assert np.array_equal(out['tree_depth'], gen['tree_depth']) and np.array_equal(out['diverging'], gen['diverging'])
    check_floats(out['samples'], gen['samples'], 'samples', late=1e-2)


@pytest.mark.parametrize('n,order,sampler,kw', [(26, 'cubic-2', 'NUTS', dict(decay=True, transform=True)),
                                                (12, 'quadratic', 'NUTS', dict(decay=True)),
                                                (7, 'cubic-2', 'NUTS', dict(transform=True, scales=True)),
                                                (26, 'cubic-2', 'HMC', dict(decay=True, transform=True, scales=True))])
def test_tensor_core_extended_density(handle, oracle, monkeypatch, n, order, sampler, kw):
    """decay ellipsoid, variable transform and module rescale (core/density.py:724-754, core/module.py:80-85) inside the
    tensor-core kernels (model variant bit 1): decisions identical to the oracle and to the generic kernel"""
    scales = kw.pop('scales', False)
    spec, cov = synthetic_spec(n, order, seed=40 + n, **kw)
    if scales:
        rng = np.random.default_rng(1)
        s0, s1 = -0.3 + 0.1 * rng.normal(size=n), 1.5 + 0.2 * rng.random(n)
        spec['input_scales'] = np.stack((s0, s0 + s1), axis=1)
    handle.set_model(to_device_spec(spec))
    C, n_iter = 90, 36
    x0 = (np.linalg.cholesky(cov) @ np.random.default_rng(6).normal(size=(n, C))).T * 0.7
    if spec['transform_ranges'] is not None:
        x0 = np.clip(x0, spec['transform_ranges'][:, 0] * 0.9, spec['transform_ranges'][:, 1] * 0.9)
        x0 = np.array([oracle.from_original(x, spec['transform_ranges'], spec['hard_bounds']) for x in x0])
    cfg = cfg_from({'n_int_step': 10}, n_iter // 2, 321, chain0=3)
    step0 = 0.5 / n**0.25
    ocfg = dict(n_iter=n_iter, n_warmup=n_iter // 2, n_int_step=10)
    handle.sampler_init(cfg, x0, step0, np.ones(n), x0)
    out = handle.sampler_run(sampler, n_iter)
    assert handle.sampler_last_path() == 'dmma'
    st = handle.sampler_state()
    assert np.all(st['status'] == 0)
    U, Z = device_draws(handle, 321, st['n_draws'], 3)
    ref = oracle.OracleDensity(spec).run(sampler, ocfg, x0, step0, np.ones(n), draws_u=U, draws_z=Z)
    assert np.array_equal(st['n_draws'], ref['n_draws'])
    for k in ('tree_depth', 'diverging') + (('tree_size',) if sampler == 'NUTS' else ()):
        assert np.array_equal(out[k], ref[k]), k
    check_floats(out['samples'], ref['samples'], 'samples', late=1e-2)
    check_floats(out['logp'], ref['logp'], 'logp', late=1e-2)
    monkeypatch.setenv('BFB200_SAMPLER', 'generic')
    handle.sampler_init(cfg, x0, step0, np.ones(n), x0)
    gen = handle.sampler_run(sampler, n_iter)
    assert handle.sampler_last_path() == 'generic'
    assert np.array_equal(out['tree_depth'], gen['tree_depth']) and np.array_equal(out['diverging'], gen['diverging'])


@pytest.mark.parametrize('family,n', [('dmma', 26), ('pair', 26), ('team', 40)], ids=['dmma', 'pair', 'team-n40'])
@pytest.mark.parametrize('env', [{}, {'BFB200_STACK_LEVELS_SMEM': '2'}, {'BFB200_STACK_LEVELS_SMEM': '0'}])
def test_tensor_core_nuts_deep_trees(handle, oracle, monkeypatch, env, family, n):
    """tiny fixed step size: trees reach depth 8-10 (up to 1023 leaves), i.e. every stack level, the L2-resident deep
    levels, the proposal-slot pool and the depth cap are exercised; outcomes identical to the oracle.  Stack levels in shared
    memory: the default (team at n = 40: 3), 2, or none but the current subtree (the pair kernel keeps at least one)"""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    monkeypatch.setenv('BFB200_SAMPLER', family)
    C, n_iter = 19, 5
    spec, cov = synthetic_spec(n, 'cubic-2', seed=5)
    handle.set_model(to_device_spec(spec))
    x0 = (np.linalg.cholesky(cov) @ np.random.default_rng(11).normal(size=(n, C))).T
    cfg = cfg_from({'adapt_step_size': 0, 'adapt_metric': 0}, 0, 55)
    step0 = 0.0035
    handle.sampler_init(cfg, x0, step0, np.ones(n), x0)
    out = handle.sampler_run('NUTS', n_iter)
    assert handle.sampler_last_path() == family
    assert out["tree_depth"].max() == 10 and out["tree_depth"].min() >= 8
    st = handle.sampler_state()
    U, Z = device_draws(handle, 55, st['n_draws'])
    ref = oracle.OracleDensity(spec).run('NUTS', dict(n_iter=n_iter, n_warmup=0, adapt_step_size=0, adapt_metric=0), x0, step0,
                                         np.ones(n), draws_u=U, draws_z=Z)
    assert np.array_equal(st['n_draws'], ref['n_draws'])
    for k in INT_STATS:
        assert np.array_equal(out[k], ref[k]), k
    check_floats(out['samples'], ref['samples'], 'samples')


@pytest.mark.parametrize('n,order,sampler,C,n_iter', [(64, 'cubic-3', 'NUTS', 64, 20), (64, 'cubic-3', 'HMC', 40, 16), (40, 'cubic-3', 'NUTS', 21, 24),
                                                       (48, 'cubic-2', 'NUTS', 50, 30), (64, 'quadratic', 'NUTS', 33, 30), (33, 'cubic-2', 'HMC', 17, 20)])
def test_team_kernels_above_32_dimensions(handle, oracle, monkeypatch, n, order, sampler, C, n_iter):
    """32 < n <= 64 (BASELINE configs[3]: 64-D cubic-3): the four-warp team kernels are the tensor-core path -- 16 dimensions per
    warp, the cubic-3 pair-product operand (1 MB at n = 64) streamed from L2 -- and the default; decisions identical to the oracle fed
    with the device's own draws and to the generic warp-per-chain kernel, tight bound so that leapfrogs leave the ellipsoid"""
    spec, cov = synthetic_spec(n, order, seed=80 + n, cubic_scale=0.05)
    spec['alpha'] = spec['alpha'] / 1.6
    handle.set_model(to_device_spec(spec))
    x0 = (np.linalg.cholesky(cov) @ np.random.default_rng(13).normal(size=(n, C))).T
    seed, chain0 = 909, 77
    kw = {'n_int_step': 6} if sampler == 'HMC' else {}
    cfg = cfg_from(kw, n_iter // 2, seed, chain0)
    step0 = 1. / n**0.25
    handle.sampler_init(cfg, x0, step0, np.ones(n), x0)
    out = handle.sampler_run(sampler, n_iter)
    assert handle.sampler_last_path() == 'team'
    st = handle.sampler_state()
    assert np.all(st['status'] == 0)
    U, Z = device_draws(handle, seed, st['n_draws'], chain0)
    ref = oracle.OracleDensity(spec).run(sampler, dict(n_iter=n_iter, n_warmup=n_iter // 2, **kw), x0, step0, np.ones(n), draws_u=U, draws_z=Z)
    assert np.array_equal(st['n_draws'], ref['n_draws'])
    ints = INT_STATS if sampler == 'NUTS' else ('tree_depth', 'diverging')      # HMC: accepted flag, divergence
    for k in ints:
        assert np.array_equal(out[k], ref[k]), k
    if sampler == 'NUTS':
        for k in FLT_STATS:
            check_floats(out[k], ref[k], k, late=5e-3)
        assert out['total_tree_size'] == int(ref['tree_size'].sum())
    check_floats(out['samples'], ref['samples'], 'samples', late=1e-2 if sampler == 'HMC' else 5e-3)
    monkeypatch.setenv('BFB200_SAMPLER', 'generic')
    handle.sampler_init(cfg, x0, step0, np.ones(n), x0)
    gen = handle.sampler_run(sampler, n_iter)
    assert handle.sampler_last_path() == 'generic'
    for k in ints:
        assert np.array_equal(out[k], gen[k]), k


@pytest.mark.parametrize('n,sampler,C', [(26, 'NUTS', 50), (10, 'NUTS', 33), (26, 'HMC', 40)])
def test_tensor_core_cubic3_samplers(handle, oracle, monkeypatch, n, sampler, C):
    """cubic-3 surrogates (n <= 28) on the tensor-core NUTS / HMC kernels: decisions identical to the oracle and the generic kernel"""
    spec, cov = synthetic_spec(n, 'cubic-3', seed=60 + n, cubic_scale=0.05)
    spec['alpha'] = spec['alpha'] / 1.6
    handle.set_model(to_device_spec(spec))
    n_iter = 30
    x0 = (np.linalg.cholesky(cov) @ np.random.default_rng(9).normal(size=(n, C))).T
    cfg = cfg_from({'n_int_step': 10}, n_iter // 2, 909, chain0=2)
    step0 = 0.6 / n**0.25
    handle.sampler_init(cfg, x0, step0, np.ones(n), x0)
    out = handle.sampler_run(sampler, n_iter)
    assert handle.sampler_last_path() == 'dmma'
    st = handle.sampler_state()
    assert np.all(st['status'] == 0)
    U, Z = device_draws(handle, 909, st['n_draws'], 2)
    ref = oracle.OracleDensity(spec).run(sampler, dict(n_iter=n_iter, n_warmup=n_iter // 2, n_int_step=10), x0, step0, np.ones(n),
                                         draws_u=U, draws_z=Z)
    assert np.array_equal(st['n_draws'], ref['n_draws'])
    for k in ('tree_depth', 'diverging') + (('tree_size',) if sampler == 'NUTS' else ()):
        assert np.array_equal(out[k], ref[k]), k
    check_floats(out['samples'], ref['samples'], 'samples', late=1e-2)
    monkeypatch.setenv('BFB200_SAMPLER', 'generic')
    handle.sampler_init(cfg, x0, step0, np.ones(n), x0)
    gen = handle.sampler_run(sampler, n_iter)
    assert handle.sampler_last_path() == 'generic'
    assert np.array_equal(out['tree_depth'], gen['tree_depth']) and np.array_equal(out['diverging'], gen['diverging'])


@pytest.mark.parametrize('family,n,order', [('team', 26, 'cubic-2'), ('pair', 10, 'cubic-3')])
def test_pinned_family_that_cannot_run_the_model_raises(handle, monkeypatch, family, n, order):
    """BFB200_SAMPLER pins a kernel family; one that has no kernel for the model is an error that names the family, not a
    silent run on the generic kernel"""
    from bayesfast_b200._cabi import BfbError
    spec, cov = synthetic_spec(n, order, seed=3, cubic_scale=0.05)
    handle.set_model(to_device_spec(spec))
    C = 16
    x0 = (np.linalg.cholesky(cov) @ np.random.default_rng(4).normal(size=(n, C))).T
    handle.sampler_init(cfg_from({}, 4, 8), x0, 0.5, np.ones(n), x0)
    monkeypatch.setenv('BFB200_SAMPLER', family)
    with pytest.raises(BfbError, match='BFB200_SAMPLER=%s: the %s kernels cannot run this model' % (family, family)):
        handle.sampler_run('NUTS', 8)
    monkeypatch.delenv('BFB200_SAMPLER')
    handle.sampler_run('NUTS', 8)
    assert handle.sampler_last_path() == 'dmma'


# ---------------------------------------------------------------------------------------------------------------------
# dense mass matrix (metric='full'): QuadMetricFull / QuadMetricFullAdapt, hmc_utils/metrics.py:94-132, 240-330
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('case', gio.load('sampler_dense.npz')['cases'], ids=lambda c: c['name'])
def test_golden_chains_dense_metric(handle, case):
    """recorded runs of the real reference with metric='full' (adapted) and a fixed covariance"""
    r, kw = case['result'], case['trace_kw']
    n_iter, n_warmup = int(kw['n_iter']), int(kw['n_warmup'])
    handle.set_model(to_device_spec(case['spec']))
    cfg = cfg_from(kw, n_warmup, int(case['seed']))
    handle.sampler_init(cfg, case['x0'], float(r['step0']), r['var0'], case['x0'], dense=True)
    out = handle.sampler_run(case['sampler'], n_iter)
    assert handle.sampler_last_path() == 'generic'
    st = handle.sampler_state()
    assert np.all(st['status'] == 0) and np.all(st['chol_error'] == 0)
    assert np.array_equal(st['n_draws'], r['n_draws'])
    if case['sampler'] == 'NUTS':
        for k in INT_STATS:
            assert np.array_equal(out[k], r[k].astype(np.int32)), k
        for k in FLT_STATS:
            check_floats(out[k], r[k], k)
    else:
        assert np.array_equal(out['tree_depth'], r['accepted'].astype(np.int32))
        assert np.array_equal(out['diverging'], r['diverging'].astype(np.int32))
        for k, k2 in (('logp', 'logp'), ('energy', 'energy'), ('mean_tree_accept', 'accept_stat'),
                      ('step_size', 'step_size'), ('energy_change', 'energy_change')):
            check_floats(out[k], r[k2], k)
    check_floats(out['samples'], r['samples'], 'samples')
    assert np.allclose(st['final_step'], r['final_step'], rtol=LATE_TOL)
    assert st['final_var'].shape == r['final_var'].shape
    assert np.allclose(st['final_var'], r['final_var'], rtol=LATE_TOL, atol=LATE_TOL * np.abs(r['final_var']).max())


@pytest.mark.parametrize('n,C,n_iter', [(26, 96, 40), (40, 8, 24)])
def test_dense_metric_teacher_forced_vs_oracle(handle, oracle, n, C, n_iter):
    """dense metric, adapted during warm-up: integer outcomes identical to the oracle fed with the device's own draws;
    after bfb_sampler_reset the run repeats bit for bit"""
    spec, cov = synthetic_spec(n, 'cubic-2', seed=7 + n, decay=True)
    handle.set_model(to_device_spec(spec))
    rng = np.random.default_rng(6)
    x0 = (np.linalg.cholesky(cov) @ rng.normal(size=(n, C))).T
    seed, chain0 = 777, 50
    cfg = cfg_from({'adapt_window': 10}, n_iter // 2, seed, chain0)
    step0 = 1. / n**0.25
    cov0 = 0.5 * cov + 0.5 * np.eye(n)
    handle.sampler_init(cfg, x0, step0, cov0, x0, dense=True)
    out = handle.sampler_run('NUTS', n_iter)
    st = handle.sampler_state()
    assert np.all(st['status'] == 0) and np.all(st['chol_error'] == 0)
    U, Z = device_draws(handle, seed, st['n_draws'], chain0)
    ref = oracle.OracleDensity(spec).run('NUTS', dict(n_iter=n_iter, n_warmup=n_iter // 2, adapt_window=10, dense_metric=1),
                                         x0, step0, cov0, draws_u=U, draws_z=Z)
    assert np.all(ref['status'] == 0)
    assert np.array_equal(st['n_draws'], ref['n_draws'])
    for k in INT_STATS:
        assert np.array_equal(out[k], ref[k]), k
    check_floats(out['samples'], ref['samples'], 'samples')
    assert np.allclose(st['final_var'], ref['final_var'], rtol=LATE_TOL, atol=LATE_TOL * np.abs(ref['final_var']).max())
    handle.sampler_reset()
    out2 = handle.sampler_run('NUTS', n_iter)
    assert np.array_equal(out2['samples'], out['samples']) and np.array_equal(out2['tree_size'], out['tree_size'])


def test_dense_metric_rejects_indefinite_covariance(handle):
    from bayesfast_b200 import _cabi
    n = 4
    spec, cov = synthetic_spec(n, 'quadratic', seed=1)
    handle.set_model(to_device_spec(spec))
    bad = np.eye(n)
    bad[0, 0] = -1.
    with pytest.raises(_cabi.BfbError, match='positive definite'):
        handle.sampler_init(cfg_from({}, 5, 1), np.zeros((2, n)), 0.5, bad, np.zeros((2, n)), dense=True)
