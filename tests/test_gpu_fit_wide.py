"""PolyModel.fit, the bound ellipsoid and the decay ellipsoid at 64 < input_size <= 128 and up to P = 16384 parameters per output:
the Gram, moment and radius kernels above 48 KB of shared memory, the moments in slabs of 4096 pairs, and the in-place triangular
solve above P = 4096 (one P-vector of shared memory, 512 threads above P = 8192)."""
import os

import numpy as np
import pytest

from test_gpu_fit import COEF_TOL, VAL_TOL, block_err, ROOT

pytestmark = pytest.mark.gpu
# known-answer fits: noise-free y from random coefficients, recovered to this error relative to each coefficient block.  Measured
# on a B200, largest block error: cubic-2 n = 60 2.1e-12, quadratic n = 128 1.8e-12, cubic-2 n = 104 1.1e-11, masked n = 100 8.0e-13
KAT_TOL = 1e-9


def _dense_truth(oracle, configs, rng):
    """random coefficients per config in the reference's dense layout, (output_size, ...)"""
    out = []
    for c in configs:
        ni, k = len(c.input_mask), oracle.n_coef(c.order, len(c.input_mask))
        out.append(np.stack([oracle.unpack_coef(c.order, rng.normal(size=k), ni) for _ in c.output_mask]))
    return out


def _y_of(configs, dense, x, m):
    """the model's outputs at x: linear c0 + c.x, quadratic sum_{k<=l} c_kl x_k x_l, cubic-2 sum_kl c_kl x_k^2 x_l"""
    y = np.zeros((x.shape[0], m))
    for c, C in zip(configs, dense):
        xm = x[:, np.asarray(c.input_mask)]
        for q, o in enumerate(c.output_mask):
            if c.order == 'linear':
                y[:, o] += C[q][0] + xm @ C[q][1:]
            elif c.order == 'quadratic':
                y[:, o] += np.sum((xm @ C[q]) * xm, axis=1)
            else:
                y[:, o] += np.sum(((xm * xm) @ C[q]) * xm, axis=1)
    return y


def _check_bound(s, x, oracle):
    mu, hess, alpha = oracle.bound_from_points(x)             # np.mean, np.linalg.inv(np.cov), the largest radius
    assert np.allclose(s._mu, mu, rtol=1e-12, atol=1e-13)
    assert block_err(s._hess, hess) < 1e-10 and abs(s._alpha - alpha) < 1e-11 * alpha


def test_fit_vs_lstsq_quadratic_n72(oracle):
    """test_fit_vs_lstsq's problem with a quadratic model at n = 72 (P = 2701, N = 3 P) against scipy.linalg.lstsq"""
    import bayesfast_b200 as bfb
    n = 72
    rng = np.random.default_rng(n)
    A = rng.normal(size=(n, n))
    Pm = A @ A.T / n + np.eye(n)
    s = bfb.PolyModel('quadratic', input_size=n, output_size=1)
    N = 3 * s.n_param
    x = rng.normal(size=(N, n))
    y = (-0.5 * np.einsum('ij,jk,ik->i', x, Pm, x) - 0.02 * np.sum(x**3 * np.exp(-0.1 * x**2), axis=1))[:, None]
    s.fit(x, y, logp=y[:, 0])
    cfgs = [dict(order=c.order, input_mask=c.input_mask, output_mask=c.output_mask) for c in s.configs]
    ref = oracle.fit(cfgs, n, 1, x, y)
    errs = [block_err(conf._coef, r) for conf, r in zip(s.configs, ref)]
    F, _ = s.eval_batch(x[:512])
    spec = s.to_spec(with_bound=False)
    for cf, r in zip(spec['configs'], ref):
        cf['coef'] = r
    Fo, _ = oracle.OracleDensity(spec).poly_eval_batch(x[:512])
    verr = np.max(np.abs(F - Fo) / np.maximum(np.abs(Fo), 1e-3 * np.max(np.abs(Fo))))
    print('P', s.n_param, 'coef errs', errs, 'value err', verr, 'resid', s._fit_rel_resid)
    assert max(errs) < COEF_TOL and verr < VAL_TOL
    _check_bound(s, x, oracle)


def _masked_n100():
    import bayesfast_b200 as bfb
    # output 0: linear + quadratic (P = 5151); output 1: quadratic + cubic-2 on 80 inputs (P = 11450); output 2: linear (P = 101)
    return bfb.PolyModel([bfb.PolyConfig('linear', np.arange(100), [0, 2]), bfb.PolyConfig('quadratic', np.arange(100), [0, 1]),
                          bfb.PolyConfig('cubic-2', np.arange(10, 90), [1])], input_size=100, output_size=3)


@pytest.mark.parametrize('case', ['cubic-2-n60', 'quadratic-n128', 'cubic-2-n104', 'masked-n100'])
def test_known_answer_fit(oracle, case):
    """noise-free y from random coefficients, N = 2 P rows: the fit recovers the coefficients.  cubic-2 at n = 60 (P = 5491) is
    inside the 54 <= n <= 64 range whose Gram launch needed more than 48 KB; cubic-2 at n = 104 is P = 16381, at the cap."""
    import bayesfast_b200 as bfb
    if case == 'masked-n100':
        s = _masked_n100()
    else:
        order, n = case.rsplit('-n', 1)
        s = bfb.PolyModel(order, input_size=int(n), output_size=1)
    n, m = s.input_size, s.output_size
    rng = np.random.default_rng(7)
    N = 2 * s.n_param
    x = rng.normal(size=(N, n))
    truth = _dense_truth(oracle, s.configs, rng)
    y = _y_of(s.configs, truth, x, m)
    s.fit(x, y, logp=y[:, 0])
    errs = [block_err(conf._coef, t) for conf, t in zip(s.configs, truth)]
    print(case, 'P', s.n_param, 'N', N, 'coef errs', errs, 'resid', s._fit_rel_resid)
    assert max(errs) < KAT_TOL
    _check_bound(s, x, oracle)


def test_density_fit_and_sample_n96():
    """Recipe-shaped flow at n = 96: fit a quadratic surrogate with the decay ellipsoid from host rows, sample 1024 chains on the
    device; the posterior means are within 5 sd / sqrt(ESS) of the truth with the ESS the device measured.  The surrogate's bound
    is off: beyond the largest radius of the fit points it continues the polynomial linearly along the ray (poly.py:262-292),
    which at n = 96 puts a shell of mass outside the fit points, so the sampled density would not be the Gaussian.  The same
    fit, bound included, from CUDA-tensor rows is bit-identical to the fit from host rows."""
    import torch
    import bayesfast_b200 as bfb
    n = 96
    rng = np.random.default_rng(96)
    A = rng.normal(size=(n, n))
    cov = A @ A.T / n + np.eye(n)
    Pm = np.linalg.inv(cov)
    sur = bfb.PolyModel('quadratic', input_size=n, output_size=1, bound_options=dict(use_bound=False))
    xf = (np.linalg.cholesky(cov) @ rng.normal(size=(n, 2 * sur.n_param))).T
    logp = -0.5 * np.einsum('ij,jk,ik->i', xf, Pm, xf)
    den = bfb.Density(sur, decay_options=dict(use_decay=True))
    den.fit(xf, logp)
    lp, g = den.logp_and_grad(xf[:5], original_space=False)
    assert np.allclose(lp, logp[:5], rtol=1e-9, atol=1e-9) and np.allclose(g, -xf[:5] @ Pm, rtol=1e-8, atol=1e-8)
    C = 1024
    tt = bfb.sample(den, dict(n_chain=C, n_iter=600, n_warmup=300, x_0=xf[:C], random_generator=5), verbose=False,
                    keep='post_warmup', diagnostics=True)
    post = tt.get()
    assert post.shape == (C * 300, n)
    ess = tt.diagnostics['ess']
    sd = np.sqrt(np.diag(cov))
    z = np.abs(post.mean(axis=0)) / (sd / np.sqrt(ess))
    print('ESS min / median', ess.min(), np.median(ess), 'R-hat max', tt.diagnostics['rhat'].max(), 'largest |mean| / (sd / sqrt(ESS))',
          z.max(), 'variance / truth', (post.var(axis=0) / np.diag(cov))[[0, -1]])
    assert np.all(z < 5.)
    a = bfb.PolyModel('quadratic', input_size=n, output_size=1)
    a.fit(xf, logp[:, None], logp=logp)
    b = bfb.PolyModel('quadratic', input_size=n, output_size=1)
    xd, yd = torch.from_numpy(xf).cuda(), torch.from_numpy(logp[:, None]).cuda()
    b.fit(xd, yd, logp=yd[:, 0].contiguous())
    for cs, ca, cb in zip(sur.configs, a.configs, b.configs):
        assert np.array_equal(np.asarray(ca._coef), np.asarray(cb._coef))
        assert np.array_equal(np.asarray(cs._coef), np.asarray(cb._coef))
    assert np.array_equal(a._mu, b._mu) and np.array_equal(a._hess, b._hess) and a._alpha == b._alpha
    assert np.array_equal(a._f_mu, b._f_mu)


def _sharded_problem_n80():
    rng = np.random.default_rng(80)
    n, N = 80, 10000
    x = rng.normal(size=(N, n)) * 0.8 + 0.1
    y = (-0.5 * np.sum(x**2, axis=1) + x @ rng.normal(size=n) + 0.1 * x[:, 0] * x[:, 1] + 0.01 * rng.normal(size=N))[:, None]
    return x, y


def _sharded_worker_n80(rank, world, port, q):
    import sys
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ['MASTER_ADDR'], os.environ['MASTER_PORT'] = '127.0.0.1', str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)        # two ranks share cuda:0: the exchange is host-staged
    import bayesfast_b200 as bfb
    from bayesfast_b200.runtime import shard_bounds
    x, y = _sharded_problem_n80()
    lo, hi = shard_bounds(x.shape[0], rank, world)
    if rank == 1:
        lo = lo + 37                  # uneven shards
    else:
        hi = hi + 37
    sur = bfb.PolyModel('quadratic', input_size=x.shape[1], output_size=1)
    den = bfb.Density(sur, decay_options=dict(use_decay=True))
    den.fit(x[lo:hi], y[lo:hi], comm=True)
    q.put((rank, [np.array(c._coef) for c in sur.configs], sur._mu, sur._hess, sur._alpha, sur._f_mu, den._mu, den._hess,
           den._alpha))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_fit_n80_two_ranks():
    """Density.fit(..., comm=True) of two ranks (gloo, both on cuda:0) at n = 80: both ranks hold the same model, and it agrees with
    the single-process fit"""
    import torch.multiprocessing as mp
    import bayesfast_b200 as bfb
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 27700 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_sharded_worker_n80, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=600) for _ in procs], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for k in range(1, 9):
        a, b = res[0][k], res[1][k]
        assert all(np.array_equal(u, v) for u, v in zip(a, b)) if isinstance(a, list) else np.array_equal(a, b)
    x, y = _sharded_problem_n80()
    sur = bfb.PolyModel('quadratic', input_size=x.shape[1], output_size=1)
    den = bfb.Density(sur, decay_options=dict(use_decay=True))
    den.fit(x, y)
    r = res[0]
    for a, b in zip(r[1], [np.array(c._coef) for c in sur.configs]):
        assert block_err(a, b) < 1e-9
    assert np.allclose(r[2], sur._mu, rtol=1e-9, atol=1e-12) and block_err(r[3], sur._hess) < 1e-9
    assert np.isclose(r[4], sur._alpha, rtol=1e-9) and np.allclose(r[5], sur._f_mu, rtol=1e-9)
    assert np.allclose(r[6], den._mu, rtol=1e-9, atol=1e-12) and block_err(r[7], den._hess) < 1e-9
    assert np.isclose(r[8], den._alpha, rtol=1e-9)


def test_fit_above_the_parameter_cap():
    """cubic-2 at n = 105 is P = 16696 > 16384: refused, and the message names the cap"""
    import bayesfast_b200 as bfb
    from bayesfast_b200 import _cabi
    s = bfb.PolyModel('cubic-2', input_size=105, output_size=1)
    assert s.n_param == 16696
    x = np.random.default_rng(0).normal(size=(s.n_param + 10, 105))
    with pytest.raises(_cabi.BfbError, match='16384'):
        s.fit(x, x[:, :1])
