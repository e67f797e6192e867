"""Independent numpy restatement of split-R-hat and ESS, the reference the device diagnostics (bayesfast_b200.diag,
csrc/bfb_diag.cu) are tested against.  It follows the definitions directly -- per half-chain autocovariances from np.correlate,
Geyer's truncation on their chain average -- and shares no code with the product's partial sums or host finishing step."""
import numpy as np


def split_rhat_ess(x):
    """Split-R-hat and ESS (the non-rank-normalised ones of Stan / ArviZ ess(method='mean')) of draws x [M, N, n] or [M, N], restated
    directly: every half-chain's autocovariance comes from np.correlate; Geyer's initial positive and monotone sequences truncate
    the autocorrelations.  Returns (rhat [n], ess [n]); nan for a coordinate with a non-finite draw or zero within-chain variance."""
    x = np.asarray(x, dtype=np.float64)
    if x.ndim == 2:
        x = x[:, :, None]
    M, N, n = x.shape
    if N < 4:
        raise ValueError('need at least 4 draws per chain')
    L = N // 2
    halves = np.concatenate([x[:, :L], x[:, N - L:]], axis=0)           # [2M, L, n]
    Mp = halves.shape[0]
    rhat, ess = np.full(n, np.nan), np.full(n, np.nan)
    for j in range(n):
        h = halves[:, :, j]
        if not np.all(np.isfinite(h)):
            continue
        means = h.mean(axis=1)
        acov = np.empty((Mp, L))
        for c in range(Mp):
            y = h[c] - means[c]
            acov[c] = np.correlate(y, y, mode='full')[L - 1:] / L        # biased autocovariance of lags 0 .. L-1
        chain_var = acov[:, 0] * L / (L - 1.)
        W = chain_var.mean()
        if not W > 0:
            continue
        B_over_n = means.var(ddof=1)
        var_plus = (L - 1.) / L * W + B_over_n
        rhat[j] = np.sqrt(var_plus / W)
        rho = 1. - (W - acov.mean(axis=0)) / var_plus
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
        tau = -1. + 2. * np.sum(r[:max_t + 1]) + np.sum(r[max_t + 1:max_t + 2])
        tau = max(tau, 1. / np.log10(Mp * L))
        ess[j] = Mp * L / tau
    return rhat, ess
