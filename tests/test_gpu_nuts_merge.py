"""The one-warp tensor-core NUTS kernel (nuts_dmma_kernel, bfb_sampler_dmma.cu) against fixed references, bit for bit.

Where the warp-pair kernel (BFB200_SAMPLER=pair) runs the model, it is the reference: it computes every output of
nuts_dmma_kernel bit-identically with code of its own, so samples, all ten statistics, n_draws and the final chain state
must match exactly.  Model variants the pair kernel does not run (cubic-3 surrogates, the likelihood pipeline) are compared
with integer outcomes recorded in tests/golden/nuts_merge.npz; `python tests/test_gpu_nuts_merge.py OUT.npz` records them
with the library that bayesfast_b200 loads (BFB200_LIB selects another build)."""
import os
import sys

import numpy as np
import pytest

for _p in (os.path.dirname(os.path.abspath(__file__)), os.path.dirname(os.path.dirname(os.path.abspath(__file__)))):
    if _p not in sys.path:
        sys.path.insert(0, _p)
from _specs import to_device_spec, synthetic_spec  # noqa: E402

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'nuts_merge.npz')
INT_STATS = ('tree_depth', 'tree_size', 'diverging')


def nuts_cfg(n_warmup, seed, **kw):
    d = dict(n_warmup=n_warmup, max_treedepth=10, n_int_step=0, max_change=1000., adapt_step_size=1,
             target_accept=0.8, gamma=0.05, k=0.75, t0=10., adapt_metric=1, initial_weight=10., adapt_window=60,
             update_window=1, doubling=1, seed=seed, chain0=0)
    d.update(kw)
    return d


@pytest.fixture(scope='module')
def handle():
    from bayesfast_b200 import _cabi
    h = _cabi.Handle(0)
    yield h
    h.close()


def run(handle, family, cfg, x0, step0, launches):
    """NUTS over sum(launches) iterations in len(launches) launches; the outputs concatenated, plus the final chain state"""
    os.environ['BFB200_SAMPLER'] = family
    try:
        n = x0.shape[1]
        handle.sampler_init(cfg, x0, step0, np.ones(n), x0)
        parts = [handle.sampler_run('NUTS', k) for k in launches]
        assert handle.sampler_last_path() == family
    finally:
        del os.environ['BFB200_SAMPLER']
    out = {k: np.concatenate([p[k] for p in parts], axis=1) for k in parts[0] if k not in ('iters', 'total_tree_size')}
    out['total_tree_size'] = sum(p['total_tree_size'] for p in parts)
    for k, v in handle.sampler_state().items():
        out['state_' + k] = v
    return out


def assert_identical(a, b):
    assert a.keys() == b.keys()
    assert len([k for k in a if k not in ('samples', 'total_tree_size') and not k.startswith('state_')]) == 10
    for k in a:
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k]), equal_nan=True), k
        if isinstance(a[k], np.ndarray):
            assert a[k].dtype == b[k].dtype and a[k].tobytes() == b[k].tobytes(), k


def des_handle(n, C):
    from bayesfast_b200 import synthetic
    import bayesfast_b200 as bfb
    prob = synthetic.des_shaped(n, seed=1, n_chain=C)
    sur = bfb.PolyModel('cubic-2', input_size=n, output_size=1)
    sur.fit(prob['x_fit'], prob['y_fit'], logp=prob['y_fit'][:, 0])
    return bfb.Density(sur)._sync(False), prob['x_0']


@pytest.mark.parametrize('n,C,launches', [(26, 1000, (120,)),          # the headline shape (NR = 7, cubic-2)
                                          (26, 1000, (40, 80)),        # resumed: two launches against the pair kernel's one
                                          (16, 203, (90,))])           # NR = 4
def test_headline_shapes_match_pair_kernel(n, C, launches):
    h, x0 = des_handle(n, C)
    cfg = nuts_cfg(sum(launches) // 2, 1)
    new = run(h, 'dmma', cfg, x0, 1. / n**0.25, launches)
    ref = run(h, 'pair', cfg, x0, 1. / n**0.25, (sum(launches),))
    assert_identical(new, ref)


@pytest.mark.parametrize('levels_smem', ['0', '1'])
def test_deep_and_divergent_trees_match_pair_kernel(handle, monkeypatch, levels_smem):
    """max_treedepth = 10 with no or one shared-memory stack level above the current subtree: merges above it read the
    L2-resident levels; every other chain takes huge steps and diverges"""
    monkeypatch.setenv('BFB200_STACK_LEVELS_SMEM', levels_smem)
    n, C, n_iter = 26, 40, 6
    spec, cov = synthetic_spec(n, 'cubic-2', seed=5)
    handle.set_model(to_device_spec(spec))
    x0 = (np.linalg.cholesky(cov) @ np.random.default_rng(11).normal(size=(n, C))).T
    step0 = np.where(np.arange(C) % 2 == 0, 0.0035, 2.5)
    cfg = nuts_cfg(0, 55, adapt_step_size=0, adapt_metric=0, max_change=50.)
    new = run(handle, 'dmma', cfg, x0, step0, (n_iter,))
    ref = run(handle, 'pair', cfg, x0, step0, (n_iter,))
    assert new['tree_depth'].max() == 10 and new['diverging'][1::2].sum() > 0
    assert_identical(new, ref)


# ---- model variants without a pair kernel: integer outcomes of the kernel before its merges were folded into one loop ----
def golden_cases(handle):
    """name -> (cfg, x0, step0, n_iter) after loading the case's model into handle"""
    from bayesfast_b200.density import whiten_spec, GaussianLikelihood
    from test_gpu_pipeline import _lik_spec
    for n, C in ((26, 50), (10, 33)):
        spec, cov = synthetic_spec(n, 'cubic-3', seed=60 + n, cubic_scale=0.05)
        spec['alpha'] = spec['alpha'] / 1.6
        handle.set_model(to_device_spec(spec))
        x0 = (np.linalg.cholesky(cov) @ np.random.default_rng(9).normal(size=(n, C))).T
        yield 'cubic3_n%d' % n, nuts_cfg(15, 909), x0, 0.6 / n**0.25, 30
    n, m, C = 26, 30, 40
    rng = np.random.default_rng(300 + n + m)
    spec = _lik_spec(rng, n, m)
    ep = spec['epilogue']
    handle.set_model(whiten_spec(to_device_spec(spec), GaussianLikelihood(ep['d'], ep['cinv'], ep['c0'])))
    yield 'likelihood_n26_m30', nuts_cfg(15, 909), rng.normal(size=(C, n)) * 0.3, 1. / n**0.25, 30


def golden_outcomes(out):
    res = {k: out[k] for k in INT_STATS}
    res['n_draws'] = out['state_n_draws']
    res['total_tree_size'] = np.array(out['total_tree_size'])
    return res


def test_variants_without_pair_kernel_match_golden(handle):
    ref = np.load(GOLDEN)
    names = []
    for name, cfg, x0, step0, n_iter in golden_cases(handle):
        got = golden_outcomes(run(handle, 'dmma', cfg, x0, step0, (n_iter,)))
        for k, v in got.items():
            assert np.array_equal(v, ref[name + '/' + k]), (name, k)
        names.append(name)
    assert sorted(names) == sorted({k.split('/')[0] for k in ref.files})


if __name__ == '__main__':
    from bayesfast_b200 import _cabi
    h = _cabi.Handle(0)
    rec = {}
    for name, cfg, x0, step0, n_iter in golden_cases(h):
        for k, v in golden_outcomes(run(h, 'dmma', cfg, x0, step0, (n_iter,))).items():
            rec[name + '/' + k] = v
    np.savez_compressed(sys.argv[1], **rec)
    print('wrote', sys.argv[1], sorted(rec))
