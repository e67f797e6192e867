"""The CPU oracle (oracle/) pinned against vectors produced by the real reference (tests/golden/)."""
import numpy as np
import pytest

import _golden_io as gio

RTOL = 1e-12   # oracle restates the reference's own evaluation order; only BLAS-order sums differ


def _close(a, b, rtol=RTOL):
    """|a-b| <= rtol * max(|b|, 1e-3 * max|b|): elementwise relative, floored against cancellation to ~0."""
    a, b = np.asarray(a, float), np.asarray(b, float)
    assert a.size == b.size
    a, b = a.ravel(), b.ravel()
    return bool(np.all(np.abs(a - b) <= rtol * np.maximum(np.abs(b), 1e-3 * np.max(np.abs(b)) + 1e-300)))


def test_philox_known_answers(oracle):
    # Random123 known-answer vectors for philox4x32-10
    assert oracle.philox_raw([0, 0, 0, 0], [0, 0]) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert oracle.philox_raw([0xffffffff] * 4, [0xffffffff] * 2) == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert oracle.philox_raw([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0]) == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_norminv_against_scipy(oracle):
    from scipy.special import ndtri
    u, z = oracle.rng_fill(3, 7, 0, 200000)
    assert np.all((u > 0) & (u < 1))
    assert np.max(np.abs(z - ndtri(u)) / np.maximum(1., np.abs(z))) < 5e-15
    assert abs(np.mean(z)) < 0.01 and abs(np.std(z) - 1) < 0.01


def test_poly_kat(oracle):
    g = gio.load('poly_kat.npz')
    for tag in ('nologp', 'logp'):
        c = g[tag]
        od = oracle.OracleDensity(c['spec'])
        F, J = od.poly_eval_batch(g['x'])
        assert _close(F[:, 0], c['values'])
        assert np.allclose(F, g['y'], rtol=1e-9, atol=1e-9)
        assert _close(J[0, 0], c['jac0'])
        F, J = od.poly_eval_batch(c['far'][None])
        assert _close(F[0], c['far_f']) and _close(J[0], c['far_j'])
    # SURVEY.md section 8c known answers
    c = g['logp']
    assert abs(c['spec']['alpha'] - 3.557097890322362) < 1e-12
    assert abs(c['spec']['f_mu'][0] - 13.784528300586311) < 1e-10


def test_poly_eval_cases(oracle):
    g = gio.load('poly_eval.npz')
    for c in g['cases']:
        spec = dict(c['spec'])
        od = oracle.OracleDensity(spec)
        F, J = od.poly_eval_batch(c['X'])
        assert _close(F, c['wrapped_f']), c['name']
        assert _close(J, c['wrapped_j']), c['name']
        spec['input_scales'] = None
        F, J = oracle.OracleDensity(spec).poly_eval_batch(c['X'])
        assert _close(F, c['raw_f']), c['name']
        assert _close(J, c['raw_j']), c['name']


def test_density_cases(oracle):
    g = gio.load('density.npz')
    for c in g['cases']:
        od = oracle.OracleDensity(c['spec'])
        lp, gr = od.logp_and_grad_batch(c['X'])
        assert _close(lp, c['logp']), c['name']
        assert _close(gr, c['grad']), c['name']


def test_fit_cases(oracle):
    g = gio.load('fit.npz')
    for c in g['cases']:
        spec = c['spec']
        cfgs = [dict(order=cf['order'], input_mask=cf['input_mask'], output_mask=cf['output_mask'])
                for cf in spec['configs']]
        coefs = oracle.fit(cfgs, int(spec['n']), int(spec['m']), c['x'], c['y'], c['w'])
        for a, cf in zip(coefs, spec['configs']):
            assert np.allclose(a, cf['coef'], rtol=1e-9, atol=1e-11), c['name']
        mu, hess, alpha = oracle.bound_from_points(c['x'], float(c['alpha_p']))
        assert np.allclose(mu, spec['mu'], rtol=1e-13) and np.allclose(hess, spec['hess'], rtol=1e-12)
        assert abs(alpha - spec['alpha']) < 1e-12 * alpha


INT_STATS = ('tree_depth', 'tree_size', 'diverging')
FLT_STATS = ('logp', 'energy', 'mean_tree_accept', 'step_size', 'step_size_bar', 'energy_change',
             'max_energy_change')


# HMC/NUTS with step-size and metric adaptation amplifies rounding differences (here only the
# summation order of BLAS ddot vs a plain loop) by ~1.25x per warm-up iteration (measured: 1e-15 ->
# 1e-6 over 40 warm-up iterations of the 2-D case), so floats are held to 1e-10 over the first
# EARLY iterations and to LATE_TOL afterwards; integer outcomes and draw counts must be identical throughout.
EARLY, EARLY_TOL, LATE_TOL = 8, 1e-10, 2e-4


def _flt(a, b, tag, early=EARLY):
    a, b = np.asarray(a, float), np.asarray(b, float)
    assert a.shape == b.shape, tag
    assert np.allclose(a[:, :early], b[:, :early], rtol=EARLY_TOL, atol=EARLY_TOL, equal_nan=True), tag
    assert np.allclose(a, b, rtol=LATE_TOL, atol=LATE_TOL, equal_nan=True), tag


@pytest.mark.parametrize('golden', ['sampler.npz', 'sampler_dense.npz', 'sampler_d26.npz'])
def test_sampler_cases(oracle, golden):
    """sampler_dense.npz: the dense mass matrix (metrics.py:94-132, 240-330); var0 / final_var are covariances"""
    g = gio.load(golden)
    for c in g['cases']:
        r = c['result']
        od = oracle.OracleDensity(c['spec'])
        cfg = {k: (int(v) if float(v) == int(v) and k not in ('max_change', 'step_size') else float(v))
               for k, v in c['trace_kw'].items()}
        cfg.pop('step_size', None)
        cfg['dense_metric'] = int(np.ndim(r['var0']) == 2)
        out = od.run(c['sampler'], cfg, c['x0'], float(r['step0']), r['var0'], draws_u=r['draws_u'],
                     draws_z=r['draws_z'])
        assert np.all(out['status'] == 0), c['name']
        assert np.array_equal(out['n_draws'], r['n_draws']), c['name']
        if c['sampler'] == 'NUTS':
            for k in INT_STATS:
                assert np.array_equal(out[k], r[k].astype(np.int32)), (c['name'], k)
            for k in FLT_STATS:
                _flt(out[k], r[k], (c['name'], k))
        else:
            assert np.array_equal(out['tree_depth'], r['accepted'].astype(np.int32)), c['name']
            assert np.array_equal(out['diverging'], r['diverging'].astype(np.int32)), c['name']
            for k, k2 in (('logp', 'logp'), ('energy', 'energy'), ('mean_tree_accept', 'accept_stat'),
                          ('step_size', 'step_size'), ('step_size_bar', 'step_size_bar'),
                          ('energy_change', 'energy_change')):
                _flt(out[k], r[k2], (c['name'], k))
        _flt(out['samples'], r['samples'], c['name'])
        assert np.allclose(out['final_step'], r['final_step'], rtol=LATE_TOL), c['name']
        assert np.allclose(out['final_var'], r['final_var'], rtol=LATE_TOL), c['name']


def _check_tempered(out, c, tag, early=EARLY):
    """shared with tests/test_gpu_tempered.py: integer outcomes and draw counts identical, floats by the two windows"""
    r = c['result']
    assert np.all(out['status'] == 0), tag
    assert np.array_equal(out['n_draws'], r['n_draws']), tag
    if c['sampler'] == 'TNUTS':
        for k in INT_STATS:
            assert np.array_equal(out[k], r[k].astype(np.int32)), (tag, k)
        for k in FLT_STATS + ('u', 'weight'):
            _flt(out[k], r[k], (tag, k), early)
    else:
        assert np.array_equal(out['tree_depth'], r['accepted'].astype(np.int32)), tag
        assert np.array_equal(out['diverging'], r['diverging'].astype(np.int32)), tag
        for k, k2 in (('logp', 'logp'), ('energy', 'energy'), ('mean_tree_accept', 'accept_stat'), ('step_size', 'step_size'),
                      ('step_size_bar', 'step_size_bar'), ('energy_change', 'energy_change'), ('u', 'u'), ('weight', 'weight')):
            _flt(out[k], r[k2], (tag, k), early)
    _flt(out['samples'], r['samples'], tag, early)


def test_tempered_sampler_cases(oracle):
    """TNUTS / THMC (samplers/tnuts.py, thmc.py, hmc_utils/base_hmc.py:220-262, integration.py:98-222) against runs of the real
    reference: target density + quadratic base density, log xi, stats 'u' and 'weight'"""
    for c in gio.load('sampler_tempered.npz')['cases']:
        r = c['result']
        od, ob = oracle.OracleDensity(c['spec']), oracle.OracleDensity(c['base_spec'])
        cfg = {k: int(v) for k, v in c['trace_kw'].items()}
        out = od.run(c['sampler'], cfg, c['x0'], float(r['step0']), r['var0'], draws_u=r['draws_u'], draws_z=r['draws_z'],
                     base=ob, logxi=float(c['logxi']), u0=c['u0'])
        _check_tempered(out, c, c['name'])
        assert np.allclose(out['final_step'], r['final_step'], rtol=LATE_TOL), c['name']
        assert np.allclose(out['final_var'], r['final_var'], rtol=LATE_TOL), c['name']


def test_pipeline_cases(oracle):
    """surrogate + Gaussian-likelihood module (2-D donut of examples/2d-donut.ipynb = BASELINE configs[0]; multi-output with
    masked configs): Density.logp_and_grad and NUTS runs of the real reference"""
    g = gio.load('pipeline.npz')
    for c in g['cases']:
        od = oracle.OracleDensity(c['spec'])
        lp, gr = od.logp_and_grad_batch(c['X'])
        assert _close(lp, c['logp'], 1e-11), c['name']
        assert _close(gr, c['grad'], 1e-11), c['name']
        r = c['result']
        cfg = {k: int(v) for k, v in c['trace_kw'].items()}
        out = od.run('NUTS', cfg, c['x0'], float(r['step0']), r['var0'], draws_u=r['draws_u'], draws_z=r['draws_z'])
        assert np.all(out['status'] == 0), c['name']
        assert np.array_equal(out['n_draws'], r['n_draws']), c['name']
        for k in INT_STATS:
            assert np.array_equal(out[k], r[k].astype(np.int32)), (c['name'], k)
        # the donut's first trees are 6-7 doublings deep: rounding differences reach 2e-10 by iteration 8 (2e-7 by the end),
        # so the 1e-10 window is the first 4 iterations here
        for k in FLT_STATS:
            _flt(out[k], r[k], (c['name'], k), early=4)
        _flt(out['samples'], r['samples'], c['name'], early=4)


def test_pipeline_extended_case(oracle):
    """multi-output pipeline with radial bound (far points take _fj_bound for every output), module rescale, variable transform
    with hard bounds and decay, cubic-2 + quadratic + linear configs: logp_and_grad and a NUTS run of the real reference"""
    for c in gio.load('pipeline_ext.npz')['cases']:
        assert c['spec']['use_bound'] and c['spec']['use_decay'] and c['spec']['transform_ranges'] is not None
        od = oracle.OracleDensity(c['spec'])
        lp, gr = od.logp_and_grad_batch(c['X'])
        assert _close(lp, c['logp'], 1e-11), c['name']
        assert _close(gr, c['grad'], 1e-11), c['name']
        r = c['result']
        # the reference ran on the oracle's Philox streams of (seed, chain): regenerated here, pinned by their digest
        nmax = int(np.max(r['n_draws'])) + 4
        U, Z = map(np.array, zip(*[oracle.rng_fill(c['seed'], i, 0, nmax) for i in range(len(r['n_draws']))]))
        assert gio.draws_digest(U, Z) == r['draws_sha256'], c['name']
        out = od.run('NUTS', {k: int(v) for k, v in c['trace_kw'].items()}, c['x0'], float(r['step0']), r['var0'],
                     draws_u=U, draws_z=Z)
        assert np.all(out['status'] == 0) and np.array_equal(out['n_draws'], r['n_draws'])
        for k in INT_STATS:
            assert np.array_equal(out[k], r[k].astype(np.int32)), (c['name'], k)
        _flt(out['samples'], r['samples'], c['name'], early=4)


def test_poly_eval_c3n64(oracle):
    """BASELINE configs[3] at its named size: 64-D cubic-3 stack (P = 47905), real-reference values inside and far outside
    the radial bound"""
    from _specs import c3n64_spec
    g = gio.load('poly_eval_c3n64.npz')
    F, J = oracle.OracleDensity(c3n64_spec(g)).poly_eval_batch(g['X'])
    assert np.allclose(F, g['raw_f'], rtol=1e-11, atol=1e-11 * np.abs(g['raw_f']).max())
    assert np.allclose(J, g['raw_j'], rtol=1e-11, atol=1e-11 * np.abs(g['raw_j']).max())


def test_pipeline_des_shaped_case(oracle):
    """the DES-Y1 example's three-module density (examples/des-y1-w-cosmosis.ipynb cells 12-18): surrogate with a linear config
    and a quadratic config on one shared 9-D mask -> chi2 module -> posterior module adding a Gaussian prior on 13 inputs;
    module input_scales, Density input_scales with hard_bounds=True on all 27 inputs, radial bound on.  logp_and_grad and a NUTS
    run (4 divergences) of the real reference."""
    for c in gio.load('pipeline_des.npz')['cases']:
        sp = c['spec']
        assert sp['use_bound'] and sp['transform_ranges'] is not None and sp['prior'] is not None and int(sp['n']) == 27
        od = oracle.OracleDensity(sp)
        lp, gr = od.logp_and_grad_batch(c['X'])
        assert _close(lp, c['logp'], 1e-11), c['name']
        assert _close(gr, c['grad'], 1e-11), c['name']
        r = c['result']
        out = od.run('NUTS', {k: int(v) for k, v in c['trace_kw'].items()}, c['x0'], float(r['step0']), r['var0'],
                     draws_u=r['draws_u'], draws_z=r['draws_z'])
        assert np.all(out['status'] == 0) and np.array_equal(out['n_draws'], r['n_draws'])
        for k in INT_STATS:
            assert np.array_equal(out[k], r[k].astype(np.int32)), (c['name'], k)
        assert int(r['diverging'].sum()) >= 1
        _flt(out['samples'], r['samples'], c['name'], early=4)


def test_post_step_restatements(oracle):
    """SystematicResampler.run (utils/misc.py:62-108) and PostStep's weights (recipe.py:1286-1297) against the real reference"""
    g = gio.load('post.npz')
    for c in g['cases']:
        idx, _ = oracle.systematic_resample(c['a'], int(c['n']), c['nodes'], c['weights'])
        assert np.array_equal(idx, c['idx']), c['name']
    w, wt = oracle.importance_weights(g['logp'], g['logq'], float(g['k_trunc']))
    assert np.array_equal(w, g['weights']) and np.array_equal(wt, g['weights_trunc'])
