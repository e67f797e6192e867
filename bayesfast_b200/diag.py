"""
Convergence diagnostics of sampled chains: split-R-hat and effective sample size (the non-rank-normalised ones of Stan and of
ArviZ's ess(method='mean')), computed where the draws live.

Everything the estimators need before Geyer's truncation is a sum over chains -- per coordinate the number of half-chains, the mean
and the sum of squared deviations of their means, and the lag sums S(k) of the centred half-chains (csrc/bfb_diag.cu, the lag sums on
the FP64 tensor cores) -- so chains sharded over GPUs combine with one all-gather of an n x (L + 3) buffer per rank, and every rank
then finishes the same global result on the host in O(n L).
"""
import numpy as np

from . import _cabi

__all__ = ['diagnostics']


def _is_cuda(t):
    return hasattr(t, 'is_cuda') and t.is_cuda


def _handle(device=None, handle=None):
    if handle is not None:
        return handle
    from .runtime import default_device
    return _cabi.Handle(default_device() if device is None else device)


def _merge(parts):
    """partials of disjoint sets of chains ([n, L + 3] each, the same L), combined in the order given: count, mean and M2 of the
    half-chain means with the pairwise update of Chan et al., the lag sums added"""
    out = np.array(parts[0], dtype=np.float64, copy=True)
    for p in parts[1:]:
        na, nb = out[:, 0], p[:, 0]
        nab = na + nb
        delta = p[:, 1] - out[:, 1]
        out[:, 1] = out[:, 1] + delta * (nb / nab)
        out[:, 2] = out[:, 2] + p[:, 2] + delta * delta * (na * nb / nab)
        out[:, 0] = nab
        out[:, 3:] += p[:, 3:]
    return out


def _tau(rho, L):
    """integrated autocorrelation time from rho_0 .. rho_{L-1}: Geyer's initial positive sequence, then the monotone sequence"""
    r = np.zeros(L)
    r[0], r[1] = 1., rho[1]
    even, odd = 1., rho[1]
    t = 1
    while t < L - 3 and even + odd > 0:
        even, odd = rho[t + 1], rho[t + 2]
        if even + odd >= 0:
            r[t + 1], r[t + 2] = even, odd
        t += 2
    max_t = t - 2
    if even > 0:
        r[max_t + 1] = even
    t = 1
    while t <= max_t - 2:
        if r[t + 1] + r[t + 2] > r[t - 1] + r[t]:
            r[t + 1] = r[t + 2] = (r[t - 1] + r[t]) / 2.
        t += 2
    return -1. + 2. * r[:max_t + 1].sum() + r[max_t + 1]


def finish(partials):
    """dict(rhat=(n,), ess=(n,)) from the global partials [n, L + 3] (bfb_chain_diagnostics); nan where W is 0 or a partial is not
    finite (a draw that is not finite)"""
    P = np.asarray(partials, dtype=np.float64)
    n, L = P.shape[0], P.shape[1] - 3
    rhat, ess = np.full(n, np.nan), np.full(n, np.nan)
    for j in range(n):
        Mp, m2, S = P[j, 0], P[j, 2], P[j, 3:]
        W = S[0] / (Mp * (L - 1))
        if not (np.all(np.isfinite(P[j])) and W > 0.):
            continue
        var_plus = (L - 1) / L * W + m2 / (Mp - 1)
        rhat[j] = np.sqrt(var_plus / W)
        rho = 1. - (W - S / (Mp * L)) / var_plus
        tau = max(_tau(rho, L), 1. / np.log10(Mp * L))
        ess[j] = Mp * L / tau
    return dict(rhat=rhat, ess=ess)


def check_same_length(N, comm=None, device=None):
    """raise ValueError on every rank of `comm` unless all ranks hold N draws per chain (a collective: call it on all ranks)"""
    from .runtime import dist_info, allreduce_values, default_device
    rank, world, group = dist_info(comm)
    if world == 1:
        return
    hi, neg_lo = allreduce_values([N, -N], 'max', group, default_device() if device is None else device, 'int64')
    if int(hi) != N or int(-neg_lo) != N:
        raise ValueError('the diagnostics need the same number of draws per chain on every rank: this rank has {}, the ranks '
                         'have {} to {}.'.format(N, int(-neg_lo), int(hi)))


def combine(partials, comm=None, device=None):
    """the global partials from this rank's partials under `comm` (torch.distributed group, or True): all ranks' buffers are
    gathered and merged in rank order, so every rank gets the same bits.  All ranks must have the same L (check_same_length)."""
    from .runtime import dist_info, allgather_vector, default_device
    rank, world, group = dist_info(comm)
    if world == 1:
        return partials
    allp = allgather_vector(np.ascontiguousarray(partials).ravel(), group, default_device() if device is None else device)
    return _merge([a.reshape(partials.shape) for a in allp])


def diagnostics(samples, comm=None, handle=None):
    """
    Split-R-hat and effective sample size of every coordinate of `samples`, [C, N, n] or [C, N] (C chains of N draws), a numpy
    array or a CUDA torch tensor (read where it lives).  Each chain is split into two halves of N // 2 draws (the middle draw of an
    odd N is dropped); ESS uses Geyer's initial positive and monotone sequences.  A coordinate whose within-chain variance is 0 or
    that has a draw that is not finite gets nan.  Under `comm` (torch.distributed group, or True) `samples` are this rank's chains
    and every rank returns the result over all ranks' chains.

    Returns
    -------
    dict(rhat=(n,), ess=(n,)) of numpy arrays
    """
    if _is_cuda(samples):
        x = samples.detach()
        if x.dim() not in (2, 3):
            raise ValueError('samples should have shape (C, N, n) or (C, N), not {}.'.format(tuple(x.shape)))
        x = x.double().contiguous()
        Cc, N = int(x.shape[0]), int(x.shape[1])
        n = int(x.shape[2]) if x.dim() == 3 else 1
        h = _handle(x.device.index, handle)
        if h.device != x.device.index:
            raise ValueError('the samples live on cuda:{} but the handle on cuda:{}.'.format(x.device.index, h.device))
    else:
        x = np.asarray(samples, dtype=np.float64)
        if x.ndim not in (2, 3):
            raise ValueError('samples should have shape (C, N, n) or (C, N), not {}.'.format(x.shape))
        x = np.ascontiguousarray(x)
        Cc, N = x.shape[0], x.shape[1]
        n = x.shape[2] if x.ndim == 3 else 1
        h = None
    check_same_length(N, comm, None if h is None else h.device)
    if N < 4:
        raise ValueError('the diagnostics need at least 4 draws per chain, got {}.'.format(N))
    if Cc < 1 or n < 1:
        raise ValueError('samples should hold at least one chain and one coordinate.')
    if h is None:
        h = _handle(None, handle)
        P = h.chain_diagnostics(x, Cc, N, 0, N, n, _cabi.BFB_HOST)
    else:
        import torch
        torch.cuda.current_stream(x.device).synchronize()
        P = h.chain_diagnostics(x.data_ptr(), Cc, N, 0, N, n, _cabi.BFB_DEVICE)
    return finish(combine(P, comm, h.device))
