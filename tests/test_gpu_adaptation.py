"""Warm-up adaptation in every sampler kernel family -- dual averaging of the step size and the windowed Welford metric with its
foreground / background swap -- with settings away from the defaults, windows that close inside the warm-up, per-chain start
values and tree-depth caps:
  (a) decisions and states identical / close to the oracle fed with the device's own draws;
  (b) the recorded step sizes and the final step-size / metric state equal, to 1e-12, the numpy restatement (tests/_adapt_ref.py)
      applied to the device's own records -- free of chaotic drift, so it runs long warm-ups, the headline shape included;
  (c) launch boundaries inside a window (split runs, short work-queue chunks, the single-launch host-output path, reset) change
      no bit;
  (d) bayesfast_b200.sample with the reference's keyword names."""
import numpy as np
import pytest

import _adapt_ref as ar
from _specs import to_device_spec, synthetic_spec
from test_gpu_sampler import cfg_from, device_draws, check_floats, INT_STATS, FLT_STATS
from test_adaptation_cpu import PROFILES, DEFAULTS, start_values, close

pytestmark = pytest.mark.gpu

# Runs compared bit for bit with themselves: profile W closes windows after warm-up samples 4, 12 and 28, D after every 6th.
N_WARMUP, N_ITER = 40, 56
# Runs compared with the oracle are shorter.  Under these settings the rounding differences between the device and the oracle
# grow about 10x every two iterations, for the generic kernel as much as for the tensor-core ones (1e-13 at the start, 1e-3
# by iteration ~28 for NUTS and ~16 for HMC), and the first different decision follows at iteration ~30 (NUTS) / ~26 (HMC).
# Within these lengths NUTS still sees the three windows of W and four of D, HMC two of each.
PARITY_LEN = {'NUTS': (29, 32), 'TNUTS': (29, 32), 'HMC': (16, 18), 'THMC': (16, 18)}      # (n_warmup, n_iter)


@pytest.fixture(scope='module')
def handles():
    from bayesfast_b200 import _cabi
    h, hb = _cabi.Handle(0), _cabi.Handle(0)
    yield h, hb
    h.close()
    hb.close()


def make_run(handles, monkeypatch, sampler, family, n, order, C, dense, settings, n_warmup, n_iter, seed=4711, chain0=40,
             n_int_step=8, max_treedepth=10):
    """set up the model and chains (per-chain step0 / var0, mean0 != x0) and run them; returns everything the checks need"""
    h, hb = handles
    tempered = sampler in ('TNUTS', 'THMC')
    hmc = sampler in ('HMC', 'THMC')
    if tempered:
        monkeypatch.delenv('BFB200_SAMPLER', raising=False)
    else:
        monkeypatch.setenv('BFB200_SAMPLER', family)
    spec, cov = synthetic_spec(n, order, seed=100 + n, decay=tempered)
    h.set_model(to_device_spec(spec))
    rng = np.random.default_rng(n + C)
    x0, step0, var0, mean0 = start_values(cov, C, rng, dense)
    if hmc:
        step0 = step0 * 0.5
    kw = dict(settings, n_int_step=n_int_step if hmc else 0, max_treedepth=max_treedepth)
    cfg = cfg_from(kw, n_warmup, seed, chain0)
    r = dict(spec=spec, x0=x0, step0=step0, var0=var0, mean0=mean0, cfg=cfg, kw=kw, seed=seed, chain0=chain0,
             n_warmup=n_warmup, n_iter=n_iter, sampler=sampler, base=None)
    if tempered:
        bspec, _ = synthetic_spec(n, 'quadratic', seed=3 + n, cond=4., bound=False)
        for cf in bspec['configs']:
            cf['coef'] = np.asarray(cf['coef']) / 3.
        hb.set_model(to_device_spec(bspec))
        r.update(base=bspec, u0=rng.normal(size=C), logxi=0.25)
        h.tsampler_init(hb, r['logxi'], cfg, x0, r['u0'], step0, var0, mean0)
    else:
        h.sampler_init(cfg, x0, step0, var0, mean0, dense=dense)
    r['out'] = run(h, sampler, n_iter)
    r['path'] = h.sampler_last_path()
    r['st'] = h.sampler_state()
    return r


def run(h, sampler, n_iter, **kw):
    return h.tsampler_run(sampler, n_iter, **kw) if sampler in ('TNUTS', 'THMC') else h.sampler_run(sampler, n_iter, **kw)


def oracle_run(oracle, h, r):
    st = r['st']
    U, Z = device_draws(h, r['seed'], st['n_draws'], r['chain0'])
    ocfg = dict(r['kw'], n_iter=r['n_iter'], n_warmup=r['n_warmup'], dense_metric=int(np.ndim(r['var0']) == 3))
    extra = {}
    if r['base'] is not None:
        extra = dict(base=oracle.OracleDensity(r['base']), logxi=r['logxi'], u0=r['u0'])
    return oracle.OracleDensity(r['spec']).run(r['sampler'], ocfg, r['x0'], r['step0'], r['var0'], r['mean0'],
                                               draws_u=U, draws_z=Z, **extra)


def check_hmc_floats(a, b, tag):
    """HMC: tight over the first 4 iterations, 1e-2 after.  Profile D's step-size adaptation takes the step to ~3 in the second
    iteration, where the leapfrog integration is unstable and rounding differences grow ~30x per iteration (the generic kernel
    reaches 4e-9 against the oracle by iteration 6, the team kernel a little more): the first 8 iterations of check_floats are
    not within 1e-9 for any kernel."""
    assert np.allclose(a[:, :4], b[:, :4], rtol=1e-9, atol=1e-9, equal_nan=True), tag
    assert np.allclose(a, b, rtol=1e-2, atol=1e-2, equal_nan=True), tag


def check_parity(r, ref):
    out, st, sampler = r['out'], r['st'], r['sampler']
    nuts = sampler in ('NUTS', 'TNUTS')
    # THMC ends a chain whose tempering variable ran away ('Bad initial energy'): most do under profile D, the same ones as in the
    # oracle; the others are compared
    assert np.array_equal(st['status'], ref['status'])
    ok = st['status'] == 0
    assert np.all(ok) if sampler != 'THMC' else ok.sum() >= len(ok) // 8
    assert np.array_equal(st['n_draws'], ref['n_draws'])
    for k in (INT_STATS if nuts else ('tree_depth', 'diverging')):
        assert np.array_equal(out[k][ok], ref[k][ok]), k
    late = 5e-3 if nuts else 1e-2
    for k in (FLT_STATS if nuts else ('mean_tree_accept', 'step_size', 'step_size_bar')) + (('u',) if sampler == 'TNUTS' else ()):
        if nuts:
            check_floats(out[k][ok], ref[k][ok], k, late)
        else:
            check_hmc_floats(out[k][ok], ref[k][ok], k)
    if nuts:
        check_floats(out['samples'][ok], ref['samples'][ok], 'samples', late)
    else:
        check_hmc_floats(out['samples'][ok], ref['samples'][ok], 'samples')
    assert np.allclose(st['final_step'][ok], ref['final_step'][ok], rtol=late, atol=late)
    fv, rv = st['final_var'][ok], ref['final_var'][ok]
    assert np.allclose(fv, rv, rtol=late, atol=late * np.abs(rv).max())


def check_restatement(r):
    """the device's adaptation state, rebuilt from its own records (chains that ended with a nonzero status left out)"""
    out, st = r['out'], r['st']
    ok = st['status'] == 0
    assert ok.sum() >= len(ok) // 8
    rec = dict(mean_tree_accept=out['mean_tree_accept'][ok], samples=out['samples'][ok])
    re = ar.adaptation(rec, r['n_warmup'], r['step0'][ok], r['var0'][ok], r['mean0'][ok], r['cfg'])
    for k in ('step_size', 'step_size_bar'):
        assert close(out[k][ok], re[k]), k
    assert close(st['final_step'][ok], re['final_step']), 'final_step'
    assert close(st['final_var'][ok], re['final_var']), 'final_var'
    return re


# sampler, family (BFB200_SAMPLER), n, order, chains, dense metric
FAMILIES = [
    ('NUTS', 'dmma', 26, 'cubic-2', 203, False),       # one-warp NUTS: the adaptation sits in the iteration boundary
    ('NUTS', 'pair', 26, 'cubic-2', 203, False),
    ('NUTS', 'team', 40, 'cubic-2', 101, False),
    ('NUTS', 'team', 64, 'cubic-3', 8, False),
    ('NUTS', 'generic', 26, 'cubic-2', 64, False),
    ('NUTS', 'generic', 96, 'quadratic', 16, False),   # above 64 dimensions only the generic kernel runs
    ('NUTS', 'generic', 16, 'cubic-2', 32, True),      # dense metric
    ('HMC', 'dmma', 26, 'cubic-2', 100, False),
    ('HMC', 'team', 26, 'cubic-2', 100, False),
    ('HMC', 'team', 40, 'cubic-2', 64, False),
    ('HMC', 'generic', 26, 'cubic-2', 64, False),
    ('HMC', 'generic', 16, 'cubic-2', 32, True),
    ('TNUTS', 'generic', 26, 'cubic-2', 64, False),
    ('THMC', 'generic', 26, 'cubic-2', 64, False),
]


def fam_id(c):
    return '%s-%s-n%d-%s-C%d%s' % (c[0], c[1], c[2], c[3], c[4], '-dense' if c[5] else '')


@pytest.mark.parametrize('profile', ['W', 'D'])
@pytest.mark.parametrize('sampler,family,n,order,C,dense', FAMILIES, ids=[fam_id(c) for c in FAMILIES])
def test_adaptation_profile_vs_oracle(handles, oracle, monkeypatch, profile, sampler, family, n, order, C, dense):
    """(a) non-default adaptation settings, windows closing inside the warm-up: integer outcomes identical to the oracle fed with
    the device's own draws, floats within the usual windows, and (b) the adaptation state exact against the restatement"""
    r = make_run(handles, monkeypatch, sampler, family, n, order, C, dense, PROFILES[profile], *PARITY_LEN[sampler])
    assert r['path'] == family
    check_parity(r, oracle_run(oracle, handles[0], r))
    check_restatement(r)


@pytest.mark.parametrize('sampler,family,n,order,C,dense', FAMILIES, ids=[fam_id(c) for c in FAMILIES])
def test_long_warmup_adaptation_vs_restatement(handles, monkeypatch, sampler, family, n, order, C, dense):
    """(b) profile W over 200 warm-up iterations (windows close after samples 4, 12, 28, 60 and 124): the recorded step sizes and
    the final state equal the restatement applied to the device's own records, to 1e-12"""
    C = min(C, 64)
    r = make_run(handles, monkeypatch, sampler, family, n, order, C, dense, PROFILES['W'], 200, 208)
    assert r['path'] == family
    # THMC ends a chain whose tempering variable ran away ('Bad initial energy', as the reference and the oracle do)
    assert sampler == 'THMC' or np.all(r['st']['status'] == 0)
    check_restatement(r)


def test_headline_shape_adaptation_vs_restatement(handles, monkeypatch):
    """(b) the default settings at the headline shape (d = 26 cubic-2, 1024 chains, 500 warm-up iterations): the windows close
    after warm-up samples 60, 180 and 420 on every chain, and the step sizes and metric equal the restatement to 1e-12"""
    h, _ = handles
    monkeypatch.delenv('BFB200_SAMPLER', raising=False)
    n, C, n_warmup, n_iter = 26, 1024, 500, 504
    spec, cov = synthetic_spec(n, 'cubic-2', seed=70 + n)
    h.set_model(to_device_spec(spec))
    x0 = (np.linalg.cholesky(cov) @ np.random.default_rng(8).normal(size=(n, C))).T
    cfg = cfg_from({}, n_warmup, 2024)
    step0, var0 = np.full(C, 1. / n**0.25), np.ones((C, n))
    h.sampler_init(cfg, x0, step0, var0, x0)
    out = h.sampler_run('NUTS', n_iter, fields=('samples', 'mean_tree_accept', 'step_size', 'step_size_bar'))
    assert h.sampler_last_path() == 'dmma'
    st = h.sampler_state()
    assert np.all(st['status'] == 0)
    r = dict(out=out, st=st, n_warmup=n_warmup, step0=step0, var0=var0, mean0=x0, cfg=dict(DEFAULTS))
    check_restatement(r)
    assert ar.windowed_metric(out['samples'][0, :n_warmup], x0[0], var0[0])[2] == [60, 180, 420]


@pytest.mark.parametrize('sampler,family,n,C,cap', [
    ('NUTS', 'dmma', 26, 96, 1), ('NUTS', 'dmma', 26, 96, 3), ('NUTS', 'pair', 26, 96, 1), ('NUTS', 'pair', 26, 96, 3),
    ('NUTS', 'team', 40, 64, 1), ('NUTS', 'team', 40, 64, 3),
    ('HMC', 'dmma', 26, 96, 1), ('HMC', 'dmma', 26, 96, 7), ('HMC', 'team', 26, 96, 1), ('HMC', 'team', 40, 64, 7)])
def test_depth_caps_vs_oracle(handles, oracle, monkeypatch, sampler, family, n, C, cap):
    """max_treedepth 1 / 3 for NUTS (the cap ends most trees), n_int_step 1 / 7 for HMC, with profile W's adaptation"""
    kw = dict(n_int_step=cap) if sampler == 'HMC' else dict(max_treedepth=cap)
    r = make_run(handles, monkeypatch, sampler, family, n, 'cubic-2', C, False, PROFILES['W'], *PARITY_LEN[sampler], **kw)
    assert r['path'] == family
    if sampler == 'NUTS':
        assert r['out']['tree_depth'].max() == cap and r['out']['tree_size'].max() <= 2**cap - 1
    else:
        assert np.all(r['out']['tree_size'] == cap)
    check_parity(r, oracle_run(oracle, handles[0], r))
    check_restatement(r)


def test_tree_depth_above_ten_runs_on_the_generic_kernel(handles, oracle, monkeypatch):
    """the tensor-core NUTS kernels keep at most 10 tree levels: max_treedepth = 11 runs on the generic kernel by default and matches
    the oracle there (a tiny step size makes trees reach depth 11), and pinning a tensor-core family with it is an error"""
    from bayesfast_b200._cabi import BfbError
    h, _ = handles
    monkeypatch.delenv('BFB200_SAMPLER', raising=False)
    n, C, n_iter = 26, 19, 3
    spec, cov = synthetic_spec(n, 'cubic-2', seed=5)
    h.set_model(to_device_spec(spec))
    x0 = (np.linalg.cholesky(cov) @ np.random.default_rng(11).normal(size=(n, C))).T
    cfg = cfg_from({'adapt_step_size': 0, 'adapt_metric': 0, 'max_treedepth': 11}, 0, 55)
    step0 = 0.0035 / 2.
    h.sampler_init(cfg, x0, step0, np.ones(n), x0)
    out = h.sampler_run('NUTS', n_iter)
    assert h.sampler_last_path() == 'generic'
    assert out['tree_depth'].max() == 11
    st = h.sampler_state()
    U, Z = device_draws(h, 55, st['n_draws'])
    ref = oracle.OracleDensity(spec).run('NUTS', dict(n_iter=n_iter, n_warmup=0, adapt_step_size=0, adapt_metric=0, max_treedepth=11),
                                         x0, step0, np.ones(n), draws_u=U, draws_z=Z)
    assert np.array_equal(st['n_draws'], ref['n_draws'])
    for k in INT_STATS:
        assert np.array_equal(out[k], ref[k]), k
    check_floats(out['samples'], ref['samples'], 'samples')
    for family in ('dmma', 'pair'):
        monkeypatch.setenv('BFB200_SAMPLER', family)
        with pytest.raises(BfbError, match='max_treedepth <= 10'):
            h.sampler_run('NUTS', 2)


SPLIT_FAMILIES = [('NUTS', 'dmma', 26, 203), ('NUTS', 'pair', 26, 96), ('NUTS', 'team', 40, 101), ('NUTS', 'generic', 26, 40),
                  ('HMC', 'dmma', 26, 96), ('HMC', 'team', 40, 64), ('TNUTS', 'generic', 26, 40)]
RECORDS = ('samples', 'tree_depth', 'tree_size', 'energy', 'mean_tree_accept', 'step_size', 'step_size_bar')


def same_state(a, b):
    for k in ('final_step', 'final_var', 'q', 'n_draws', 'status'):
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize('sampler,family,n,C', SPLIT_FAMILIES, ids=['%s-%s-n%d' % c[:3] for c in SPLIT_FAMILIES])
def test_launch_boundaries_inside_windows(handles, monkeypatch, sampler, family, n, C):
    """(c) profile W: the same run after bfb_sampler_reset, split over five calls that end inside windows (after iterations 3, 10,
    16 and 29; windows close at 4, 12 and 28), and cut into work-queue chunks of 3 iterations, is bit-identical to one call"""
    h, _ = handles
    r = make_run(handles, monkeypatch, sampler, family, n, 'cubic-2', C, False, PROFILES['W'], N_WARMUP, N_ITER)
    assert r['path'] == family
    full, st = r['out'], r['st']
    h.sampler_reset()
    again = run(h, sampler, N_ITER)
    same_state(h.sampler_state(), st)
    h.sampler_reset()
    parts = [run(h, sampler, k) for k in (3, 7, 6, 13, 27)]
    assert h.sampler_last_path() == family
    same_state(h.sampler_state(), st)
    monkeypatch.setenv('BFB200_CHUNK_ITERS', '3')
    h.sampler_reset()
    chunked = run(h, sampler, N_ITER)
    same_state(h.sampler_state(), st)
    for k in RECORDS:
        assert np.array_equal(again[k], full[k]), ('reset', k)
        assert np.array_equal(np.concatenate([p[k] for p in parts], axis=1), full[k]), ('split', k)
        assert np.array_equal(chunked[k], full[k]), ('chunks', k)


def test_single_launch_host_outputs_inside_windows(handles, monkeypatch):
    """(c) the single-launch host-output path of the one-warp NUTS kernel (copies of finished iteration chunks while the kernel runs)
    against chunked launches through staging buffers, with profile W's windows: same records and state, bit for bit"""
    h, _ = handles
    runs = {}
    for name, env in (('single', {}), ('multi', {'BFB200_E2E_MULTI_LAUNCH': '1'})):
        monkeypatch.delenv('BFB200_E2E_MULTI_LAUNCH', raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        r = make_run(handles, monkeypatch, 'NUTS', 'dmma', 26, 'cubic-2', 203, False, PROFILES['W'], N_WARMUP, 80)
        monkeypatch.delenv('BFB200_SAMPLER')           # the single-launch path is the default one: nothing pinned
        h.sampler_reset()
        r['out'] = h.sampler_run('NUTS', 80)
        assert h.sampler_last_path() == 'dmma'
        runs[name] = (r['out'], h.sampler_state())
        check_restatement(dict(r, st=runs[name][1]))
    for k in RECORDS:
        assert np.array_equal(runs['single'][0][k], runs['multi'][0][k]), k
    same_state(runs['single'][1], runs['multi'][1])


def api_density(n, order, seed, scale=1.):
    import bayesfast_b200 as bfb
    from _specs import pack
    spec, cov = synthetic_spec(n, order, seed=seed, bound=False)
    sur = bfb.PolyModel(order, input_size=n, output_size=1)
    for conf, cf in zip(sur.configs, spec['configs']):
        conf._set(pack(cf['order'], np.asarray(cf['coef'][0]) * scale, n), 0)
    return bfb.Density(sur, decay_options=dict(use_decay=False)), cov


def check_trace_tuple(tt, cfg, step0, var0, mean0, n_warmup):
    """per chain: the step-size object and the metric of tt[i] carry the device's final state, which equals the restatement"""
    fin = tt._final
    for i in range(tt.n_chain):
        da = tt[i].step_size
        assert [da._log_step, da._log_bar, da._hbar, da._count] == [fin['final_step'][i, 0], fin['final_step'][i, 1],
                                                                    fin['final_step'][i, 2], int(fin['final_step'][i, 3])]
        assert np.array_equal(tt[i].metric._var, fin['final_var'][i])
    re = ar.adaptation(dict(mean_tree_accept=tt.arrays['mean_tree_accept'], samples=tt.arrays['samples']), n_warmup, step0,
                       var0, mean0, cfg)
    assert close(fin['final_step'], re['final_step']) and close(fin['final_var'], re['final_var'])
    assert close(tt.arrays['step_size'], re['step_size'])


def test_sample_api_adaptation_keywords(oracle):
    """(d) bayesfast_b200.sample with the reference's keyword names (adapt_window, update_window, doubling, initial_mean,
    initial_weight, target_accept, gamma, k, t_0, max_change, max_treedepth): tree depths equal the oracle's, tt[i].step_size and
    tt[i].metric carry the final state; the same with a TNTrace"""
    import bayesfast_b200 as bfb
    n, C, n_iter, n_warmup = 8, 32, 56, 40
    den, cov = api_density(n, 'cubic-2', 4)
    rng = np.random.default_rng(3)
    x0 = (np.linalg.cholesky(cov) @ rng.normal(size=(n, C))).T * 0.5
    m0 = 0.2 * np.sqrt(np.diag(cov)) * rng.normal(size=n)
    akw = dict(adapt_window=4, update_window=3, doubling=False, initial_mean=m0, initial_weight=2.5, target_accept=0.65,
               gamma=0.1, k=0.6, t_0=4., max_change=40., max_treedepth=8)
    cfg = dict(target_accept=0.65, gamma=0.1, k=0.6, t0=4., initial_weight=2.5, adapt_window=4, update_window=3, doubling=0,
               max_change=40., max_treedepth=8)
    step0, mean0 = np.full(C, 1. / n**0.25), np.broadcast_to(m0, (C, n))
    tt = bfb.sample(den, dict(n_chain=C, n_iter=n_iter, n_warmup=n_warmup, x_0=x0, random_generator=5, **akw), verbose=False)
    U, Z = device_draws(den._sync(False), 5, tt._final['n_draws'])
    ref = oracle.OracleDensity(den.to_spec()).run('NUTS', dict(cfg, n_iter=n_iter, n_warmup=n_warmup), x0, step0, np.ones(n),
                                                  mean0, draws_u=U, draws_z=Z)
    assert np.array_equal(tt.arrays['tree_depth'], ref['tree_depth'])
    assert np.allclose(tt._final['final_var'], ref['final_var'], rtol=5e-3)
    check_trace_tuple(tt, cfg, step0, np.ones((C, n)), mean0, n_warmup)
    # the tempered sampler takes the same keywords through its trace
    base, _ = api_density(n, 'quadratic', 4, 0.4)
    u0 = np.linspace(-1., 1., C)
    tn = bfb.sample(den, bfb.TNTrace(base, 0.1, n_chain=C, n_iter=n_iter, n_warmup=n_warmup, x_0=x0, random_generator=5, u_0=u0,
                                     **akw), verbose=False)
    assert tn.sampler == 'TNUTS'
    U, Z = device_draws(den._sync(False), 5, tn._final['n_draws'])
    ref = oracle.OracleDensity(den.to_spec()).run('TNUTS', dict(cfg, n_iter=n_iter, n_warmup=n_warmup), x0, step0, np.ones(n),
                                                  mean0, draws_u=U, draws_z=Z, base=oracle.OracleDensity(base.to_spec()),
                                                  logxi=0.1, u0=u0)
    assert np.array_equal(tn.arrays['tree_depth'], ref['tree_depth'])
    check_trace_tuple(tn, cfg, step0, np.ones((C, n)), mean0, n_warmup)
