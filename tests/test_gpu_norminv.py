"""The tensor-core samplers draw their momenta with a restatement of Phi^-1 (bfb_norminv_small, bfb_nuts_dmma_common.cuh) that
is smaller code than bfb_norminv of bfb_rng.h.  It must be the same function bit for bit on every uniform the stream can
produce: U = (k + 0.5) 2^-52, k = 0 .. 2^52 - 1."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

K_MAX = 1 << 52


def draws(k):
    k = np.asarray(k, dtype=np.int64)
    k = k[(k >= 0) & (k < K_MAX)]
    return (k.astype(np.float64) + 0.5) * 2.0 ** -52       # exact: the uniforms of bfb_u64_to_uniform


def around(p, half_width):
    """the half_width draws on either side of probability p (and of 1 - p)"""
    k0 = int(p * K_MAX)
    k = np.arange(k0 - half_width, k0 + half_width, dtype=np.int64)
    return np.concatenate([k, K_MAX - 1 - k])


@pytest.fixture(scope='module')
def handle():
    from bayesfast_b200 import _cabi
    h = _cabi.Handle(0)
    yield h
    h.close()


def assert_bit_identical(handle, p):
    z, z_ref = handle.norminv_fill(p)
    assert np.all(np.isfinite(z_ref))
    diff = np.flatnonzero(z.view(np.uint64) != z_ref.view(np.uint64))
    assert diff.size == 0, 'p = %r: %r != %r' % (p[diff[0]], z[diff[0]], z_ref[diff[0]])


def test_dense_grid(handle):
    k = np.arange(1 << 22, dtype=np.int64) * (K_MAX >> 22) + (np.arange(1 << 22) % 977)    # 4M draws over (0, 1)
    rng = np.random.default_rng(0)
    assert_bit_identical(handle, draws(np.concatenate([k, rng.integers(0, K_MAX, 1 << 20)])))


def test_tails(handle):
    # the extreme draws and every power of two (and its neighbours) in k, on both sides: down to the smallest draw 2^-53
    k = np.arange(1 << 16, dtype=np.int64)
    pw = (1 << np.arange(52, dtype=np.int64))[:, None] + np.arange(-3, 4)[None, :]
    k = np.concatenate([k, pw.ravel()])
    p = draws(np.concatenate([k, K_MAX - 1 - k]))
    assert p.min() == 2.0 ** -53 and p.max() == 1. - 2.0 ** -53
    assert_bit_identical(handle, p)


def test_branch_switches(handle):
    # |p - 0.5| = 0.425 (central branch / tails) and r = sqrt(-log p) = 5 (the two tail polynomials)
    p = draws(np.concatenate([around(0.075, 1 << 16), around(np.exp(-25.), 1 << 12)]))
    q = p - 0.5
    assert (np.abs(q) <= 0.425).any() and (np.abs(q) > 0.425).any()
    r = np.sqrt(-np.log(np.where(q < 0, p, 1. - p)))
    assert (r <= 5.).any() and (r > 5.).any()
    assert_bit_identical(handle, p)
