"""Warm-up adaptation of the oracle (oracle/bf_oracle.c: dual averaging, windowed Welford metric) against the independent numpy
restatement in tests/_adapt_ref.py, with settings away from the defaults and windows that close inside the warm-up; a hand-worked
case pins the restatement itself.  No GPU needed."""
import numpy as np
import pytest

import _adapt_ref as ar
from _specs import synthetic_spec

# the reference's defaults, and the two profiles the device kernels are tested with (tests/test_gpu_adaptation.py): W closes
# windows after warm-up samples 4, 12 and 28 and updates the metric every third sample; D keeps a window of 6 and changes
# every setting of the step-size adaptation
DEFAULTS = dict(target_accept=0.8, gamma=0.05, k=0.75, t0=10., initial_weight=10., adapt_window=60, update_window=1, doubling=1,
                max_change=1000.)
PROFILES = {'W': dict(DEFAULTS, adapt_window=4, update_window=3, doubling=1, initial_weight=2.5),
            'D': dict(DEFAULTS, adapt_window=6, doubling=0, update_window=2, target_accept=0.65, gamma=0.1, k=0.6, t0=4.,
                      max_change=40.)}


def close(a, b, rtol=1e-12):
    """relative agreement; entries near zero are measured against the largest magnitude of the row"""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    scale = np.max(np.abs(b).reshape(b.shape[0], -1), axis=1).reshape((-1,) + (1,) * (b.ndim - 1))
    return np.all(np.abs(a - b) <= rtol * np.maximum(np.abs(b), 1e-3 * scale))


def start_values(cov, C, rng, dense=False):
    """per-chain step0, var0 (0.5-2x the diagonal of the covariance, or a perturbed covariance) and mean0 != x0"""
    n = cov.shape[0]
    sd = np.sqrt(np.diag(cov))
    x0 = (np.linalg.cholesky(cov) @ rng.normal(size=(n, C))).T
    step0 = rng.uniform(0.6, 1.2, size=C) / n**0.25
    if dense:
        var0 = np.array([cov * s + np.diag(np.diag(cov)) * 0.5 for s in rng.uniform(0.5, 2., size=C)])
    else:
        var0 = np.diag(cov) * rng.uniform(0.5, 2., size=(C, n))
    mean0 = x0 + 0.3 * sd * rng.normal(size=(C, n))
    return x0, step0, var0, mean0


@pytest.mark.parametrize('profile', ['W', 'D'])
@pytest.mark.parametrize('sampler,dense', [('NUTS', False), ('HMC', False), ('NUTS', True), ('HMC', True), ('TNUTS', False)])
def test_oracle_adaptation_matches_restatement(oracle, profile, sampler, dense):
    """the oracle's recorded step_size / step_size_bar and its final step-size and metric state are rebuilt from its own records"""
    n, C, n_warmup, n_iter = 6, 12, 40, 48
    spec, cov = synthetic_spec(n, 'cubic-2', seed=17, decay=True)
    rng = np.random.default_rng(23)
    x0, step0, var0, mean0 = start_values(cov, C, rng, dense)
    p = PROFILES[profile]
    cfg = dict(p, n_iter=n_iter, n_warmup=n_warmup, max_treedepth=10, n_int_step=6, seed=99, dense_metric=int(dense))
    od = oracle.OracleDensity(spec)
    if sampler == 'TNUTS':
        bspec, _ = synthetic_spec(n, 'quadratic', seed=3, cond=4., bound=False)
        kw = dict(base=oracle.OracleDensity(bspec), logxi=0.2, u0=rng.normal(size=C))
    else:
        kw = {}
    ref = od.run(sampler, cfg, x0, step0, var0, mean0, **kw)
    assert np.all(ref['status'] == 0)
    re = ar.adaptation(ref, n_warmup, step0, var0, mean0, cfg)
    for k in ('step_size', 'step_size_bar', 'final_step', 'final_var'):
        assert close(ref[k], re[k]), k
    # the profile's windows close inside the warm-up (the swap branch of the metric runs) and the metric moved off var0
    closed = ar.windowed_metric(ref['samples'][0, :n_warmup], mean0[0], var0[0], p['initial_weight'], p['adapt_window'],
                                p['update_window'], p['doubling'])[2]
    assert closed == ([4, 12, 28] if profile == 'W' else [6, 12, 18, 24, 30, 36])
    assert not np.allclose(ref['final_var'], var0)


def test_oracle_adaptation_settings_reach_the_result(oracle):
    """each non-default setting changes the oracle's outcome: none of them is ignored on the way in"""
    n, C = 5, 4
    spec, cov = synthetic_spec(n, 'cubic-2', seed=2)
    x0, step0, var0, mean0 = start_values(cov, C, np.random.default_rng(1))
    od = oracle.OracleDensity(spec)
    base = dict(PROFILES['W'], n_iter=30, n_warmup=30, seed=5)
    r0 = od.run('NUTS', base, x0, step0, var0, mean0)
    for k, v in (('adapt_window', 5), ('update_window', 2), ('doubling', 0), ('initial_weight', 3.), ('target_accept', 0.7),
                 ('gamma', 0.06), ('k', 0.7), ('t0', 9.)):
        r = od.run('NUTS', dict(base, **{k: v}), x0, step0, var0, mean0)
        assert not (np.array_equal(r['final_step'], r0['final_step']) and np.array_equal(r['final_var'], r0['final_var'])), k
    r = od.run('NUTS', base, x0, step0, var0, mean0 + 0.1)
    assert not np.array_equal(r['final_var'], r0['final_var'])


def test_windowed_metric_hand_worked():
    """n = 1, initial weight 2 at mean 0 / variance 1, window 2 (doubling), metric updated every second sample of a window.
    Foreground after samples 1, 3: weight 4, mean 1, raw 8 -> variance 2 at the second sample.  The third sample (delta = 2)
    closes the window: the background (weight 13, mean 4/13, raw 114/13) takes over, the window becomes 4.  Sample 2 there
    (delta = 1): weight 14, raw 80/7 -> 40/49.  Sample 5 (delta = 2): no update.  Sample -1 (delta = 3): weight 16, raw 135/4
    -> 135/64."""
    hist, final, closed = ar.windowed_metric(np.array([[1.], [3.], [0.], [2.], [5.], [-1.]]), np.zeros(1), np.ones(1),
                                             initial_weight=2., adapt_window=2, update_window=2, doubling=True)
    assert np.allclose(hist[:, 0], [1., 2., 2., 40. / 49., 40. / 49., 135. / 64.], rtol=1e-14, atol=0)
    assert closed == [2] and np.allclose(final, 135. / 64., rtol=1e-14)
    # dense, 1 x 1: the same numbers up to the swap (after it the foreground is the background, which starts at the identity)
    hd, fd, cd = ar.windowed_metric(np.array([[1.], [3.], [0.]]), np.zeros(1), np.eye(1), initial_weight=2., adapt_window=2,
                                    update_window=2, doubling=True)
    assert cd == [2] and np.allclose(hd[:, 0, 0], [1., 2., 2.], rtol=1e-14)


def test_dual_average_hand_worked():
    """step0 = 0.1 (mu = log(10 step0) = 0), accept statistics 0.5 then 1.0, target 0.8, gamma 0.05, k 0.75, t0 10:
    hbar_1 = 0.3 / 11, log_step_1 = log_bar_1 = -6/11; hbar_2 = 11/12 hbar_1 - 0.2 / 12 = 1/120,
    log_step_2 = -sqrt(2) / 6, log_bar_2 = 2^-0.75 log_step_2 + (1 - 2^-0.75) log_bar_1."""
    s, b, f = ar.dual_average([0.5, 1.0], 0.1, target_accept=0.8, gamma=0.05, k=0.75, t0=10.)
    ls2 = -np.sqrt(2.) / 6.
    lb2 = 2.**-0.75 * ls2 + (1. - 2.**-0.75) * (-6. / 11.)
    assert np.allclose(s, np.exp([-6. / 11., ls2]), rtol=1e-14) and np.allclose(b, np.exp([-6. / 11., lb2]), rtol=1e-14)
    assert np.allclose(f, [ls2, lb2, 1. / 120., 3.], rtol=1e-14)


def test_sample_rejects_bad_adaptation_settings_before_device_work():
    """the reference's keyword checks (sample_trace.py): a bad setting is a ValueError raised before any device handle exists"""
    import bayesfast_b200 as bfb
    from _specs import pack
    n = 4
    spec, cov = synthetic_spec(n, 'cubic-2', seed=4)
    sur = bfb.PolyModel('cubic-2', input_size=n, output_size=1)
    for conf, cf in zip(sur.configs, spec['configs']):
        conf._set(pack(cf['order'], cf['coef'][0], n), 0)
    den = bfb.Density(sur)
    x0 = np.zeros((4, n))
    for bad in (dict(update_window=0), dict(adapt_window=0), dict(initial_weight=0.),
                dict(target_accept=1.), dict(gamma=0.), dict(t_0=-1.), dict(max_change=0.), dict(max_treedepth=0)):
        with pytest.raises(ValueError):
            bfb.sample(den, dict(n_chain=4, n_iter=10, n_warmup=5, x_0=x0, random_generator=1, **bad), verbose=False)
        assert den._handle is None, bad
    with pytest.raises(ValueError):
        bfb.sample(den, dict(n_chain=4, n_iter=10, n_warmup=5, n_int_step=0, x_0=x0, random_generator=1), sampler='HMC',
                   verbose=False)
    assert den._handle is None
