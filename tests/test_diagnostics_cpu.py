"""Split-R-hat and ESS without a GPU: the oracle's restatement of the definitions on chains whose answer is known, its edge cases,
the host finishing step of bayesfast_b200.diag (fed partials computed here with numpy) against the oracle, the pairwise merge of
uneven chain shards, and a world_size-2 `gloo` run whose ranks must agree.  The reference is tests/_diag_oracle.py."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ar1(rng, M, N, phi, n=1):
    """AR(1) chains with unit stationary variance, started in the stationary distribution; phi scalar or [n]"""
    phi = np.broadcast_to(np.asarray(phi, dtype=np.float64), (n,))
    x = np.empty((M, N, n))
    x[:, 0] = rng.normal(size=(M, n))
    s = np.sqrt(1. - phi**2)
    for t in range(1, N):
        x[:, t] = phi * x[:, t - 1] + s * rng.normal(size=(M, n))
    return x


def _partials(x):
    """the partials of bfb_chain_diagnostics in numpy: [n, L + 3] = M' | mean of the half-chain means | their M2 | S(0 .. L-1)"""
    x = np.asarray(x, dtype=np.float64)
    if x.ndim == 2:
        x = x[:, :, None]
    M, N, n = x.shape
    L = N // 2
    h = np.concatenate([x[:, :L], x[:, N - L:]], axis=0)
    m = h.mean(axis=1)                                                   # [M', n]
    y = h - m[:, None]
    P = np.empty((n, L + 3))
    P[:, 0] = 2 * M
    P[:, 1] = m.mean(axis=0)
    P[:, 2] = ((m - P[:, 1])**2).sum(axis=0)
    for k in range(L):
        P[:, 3 + k] = (y[:, :L - k] * y[:, k:]).sum(axis=(0, 1))
    return P


def test_oracle_ar1_ess_and_iid_rhat():
    import _diag_oracle as o
    rng = np.random.default_rng(11)
    x = _ar1(rng, 64, 4000, 0.5)                     # tau = (1 + phi) / (1 - phi) = 3
    rhat, ess = o.split_rhat_ess(x)
    assert abs(ess[0] / (64 * 4000) - 1. / 3.) < 0.1 / 3.
    assert abs(rhat[0] - 1.) < 0.01
    iid = rng.normal(size=(64, 4000, 2))
    rhat, ess = o.split_rhat_ess(iid)
    assert np.all(np.abs(rhat - 1.) < 0.01)
    assert np.all(np.abs(ess / (64 * 4000) - 1.) < 0.1)
    four = np.random.default_rng(5).normal(size=(4, 1000))
    four[3] += 2.                                    # one chain 2 sd away
    rhat, _ = o.split_rhat_ess(four)
    assert rhat[0] > 1.2


def test_oracle_edge_cases():
    import _diag_oracle as o
    rng = np.random.default_rng(2)
    x = rng.normal(size=(5, 101, 3))
    r_odd, e_odd = o.split_rhat_ess(x)               # odd N: the middle draw is dropped
    r_cut, e_cut = o.split_rhat_ess(np.concatenate([x[:, :50], x[:, 51:]], axis=1))
    assert np.array_equal(r_odd, r_cut) and np.array_equal(e_odd, e_cut)
    with pytest.raises(ValueError):
        o.split_rhat_ess(x[:, :3])
    c = x.copy()
    c[:, :, 1] = 2.5                                 # constant coordinate
    c[2, 7, 2] = np.nan                              # a draw that is not finite
    r, e = o.split_rhat_ess(c)
    assert np.isfinite(r[0]) and np.isfinite(e[0]) and np.all(np.isnan(r[1:])) and np.all(np.isnan(e[1:]))
    r1, e1 = o.split_rhat_ess(x[:1])                 # M = 1: two half-chains
    assert np.all(np.isfinite(r1)) and np.all(e1 > 0)


@pytest.mark.parametrize('M,N,n', [(1, 9, 1), (1, 4, 2), (3, 101, 5), (7, 64, 3), (64, 400, 4)])
def test_finish_matches_oracle(M, N, n):
    import _diag_oracle as o
    from bayesfast_b200 import diag
    rng = np.random.default_rng(M * 1000 + N)
    x = _ar1(rng, M, N, np.linspace(0.1, 0.9, n), n) + np.linspace(-1., 1., M)[:, None, None] * 0.1
    ref_r, ref_e = o.split_rhat_ess(x)
    got = diag.finish(_partials(x))
    assert np.allclose(got['rhat'], ref_r, rtol=1e-12, atol=0)
    assert np.allclose(got['ess'], ref_e, rtol=1e-12, atol=0)


def test_finish_degenerate_coordinates():
    from bayesfast_b200 import diag
    x = np.random.default_rng(4).normal(size=(6, 40, 3))
    x[:, :, 0] = -1.
    x[4, 3, 2] = np.inf
    got = diag.finish(_partials(x))
    assert np.isnan(got['rhat'][0]) and np.isnan(got['ess'][0]) and np.isnan(got['rhat'][2]) and np.isnan(got['ess'][2])
    assert np.isfinite(got['rhat'][1]) and np.isfinite(got['ess'][1])


def test_short_chains_raise_before_any_device_work():
    from bayesfast_b200 import diag
    with pytest.raises(ValueError):
        diag.diagnostics(np.zeros((4, 3, 2)))
    with pytest.raises(ValueError):
        diag.diagnostics(np.zeros((4, 3, 2, 1)))


def test_chan_merge_of_uneven_shards():
    import _diag_oracle as o
    from bayesfast_b200 import diag
    rng = np.random.default_rng(8)
    x = _ar1(rng, 13, 250, [0.3, 0.7, 0.95], 3) + rng.normal(size=(13, 1, 3)) * 0.2 + 5.
    merged = diag._merge([_partials(x[:3]), _partials(x[3:])])
    whole = _partials(x)
    assert merged[:, 0].tolist() == whole[:, 0].tolist()
    assert np.allclose(merged[:, 1:], whole[:, 1:], rtol=1e-12, atol=1e-12 * np.abs(whole[:, 3:4]))
    ref_r, ref_e = o.split_rhat_ess(x)
    got = diag.finish(merged)
    assert np.allclose(got['rhat'], ref_r, rtol=1e-12, atol=0) and np.allclose(got['ess'], ref_e, rtol=1e-12, atol=0)


def _chains():
    return _ar1(np.random.default_rng(21), 9, 120, [0.2, 0.6], 2)


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    import torch.distributed as dist
    from bayesfast_b200 import diag
    from bayesfast_b200.runtime import shard_bounds
    from test_diagnostics_cpu import _chains, _partials
    os.environ['MASTER_ADDR'], os.environ['MASTER_PORT'] = '127.0.0.1', str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    x = _chains()
    lo, hi = shard_bounds(x.shape[0], rank, world)
    diag.check_same_length(x.shape[1], True, 0)
    res = diag.finish(diag.combine(_partials(x[lo:hi]), True, 0))
    try:                                               # ranks that hold different chain lengths are refused on every rank
        diag.check_same_length(x.shape[1] + rank, True, 0)
        refused = False
    except ValueError:
        refused = True
    q.put((rank, res['rhat'], res['ess'], refused))
    dist.barrier()
    dist.destroy_process_group()


def test_two_ranks_gloo_agree():
    import torch.multiprocessing as mp
    import _diag_oracle as o
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 31500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=180) for _ in procs], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert np.array_equal(res[0][1], res[1][1]) and np.array_equal(res[0][2], res[1][2])
    assert res[0][3] and res[1][3]
    ref_r, ref_e = o.split_rhat_ess(_chains())
    assert np.allclose(res[0][1], ref_r, rtol=1e-12, atol=0) and np.allclose(res[0][2], ref_e, rtol=1e-12, atol=0)
