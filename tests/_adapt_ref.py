"""Independent numpy restatement of the warm-up adaptation of the NUTS / HMC samplers, the reference the adaptation state of the
device kernels and of the oracle is tested against.  It is written from the definitions of the reference's hmc_utils --
Nesterov dual averaging of the step size (step_size.py:10-51) and the windowed, weighted Welford estimate of the mass matrix
(metrics.py:135-237, 240-330, 333-417) -- and shares no code with the product or with the oracle.

Everything here is a function of what a run records: the accept statistics of the warm-up iterations fix the step size, the
warm-up samples fix the metric."""
import numpy as np


def dual_average(accept, step0, target_accept=0.8, gamma=0.05, k=0.75, t0=10.):
    """Step-size adaptation over the accept statistics `accept` of one chain's warm-up iterations, started from `step0`.

    After iteration i the error average is hbar_i = (1 - w) hbar_{i-1} + w (target_accept - accept_i), w = 1 / (i + t0)
    (i = 1, 2, ...), the step log_step_i = log(10 step0) - hbar_i sqrt(i) / gamma and its average
    log_bar_i = i^-k log_step_i + (1 - i^-k) log_bar_{i-1}, log_bar_0 = log(step0).

    Returns (step_size [N], step_size_bar [N], final): exp(log_step_i), exp(log_bar_i) after every iteration -- the recorded
    `step_size` / `step_size_bar` -- and final = (log_step, log_bar, hbar, count) after the last one, count = N + 1 (the layout
    of the sampler's final step-size state)."""
    accept = np.asarray(accept, dtype=np.float64)
    log_step = log_bar = float(np.log(step0))
    mu = float(np.log(10. * step0))
    hbar = 0.
    steps, bars = np.empty(accept.size), np.empty(accept.size)
    for i, a in enumerate(accept, start=1):
        w = 1. / (i + t0)
        hbar = (1. - w) * hbar + w * (target_accept - a)
        log_step = mu - hbar * np.sqrt(i) / gamma
        eta = float(i) ** -k
        log_bar = eta * log_step + (1. - eta) * log_bar
        steps[i - 1], bars[i - 1] = np.exp(log_step), np.exp(log_bar)
    return steps, bars, np.array([log_step, log_bar, hbar, accept.size + 1.])


class _Moments:
    """Weighted running mean and (co)variance: `weight` pseudo-samples at `mean` with (co)variance `cov`, then one sample at a
    time.  The raw second moment gains (x - mean_new) (x - mean_old)^T per sample; the estimate is raw / weight."""

    def __init__(self, mean, cov, weight):
        self.weight = float(weight)
        self.mean = np.array(mean, dtype=np.float64)
        self.raw = np.array(cov, dtype=np.float64) * self.weight

    def add(self, x):
        self.weight += 1.
        before = x - self.mean
        self.mean = self.mean + before / self.weight
        after = x - self.mean
        self.raw = self.raw + (np.outer(after, before) if self.raw.ndim == 2 else before * after)

    def estimate(self):
        return self.raw / self.weight


def windowed_metric(samples, mean0, var0, initial_weight=10., adapt_window=60, update_window=1, doubling=True):
    """Mass-matrix adaptation over one chain's warm-up `samples` [N, n].  var0 [n] is a diagonal metric, var0 [n, n] a dense one.

    Two estimates see every sample: the foreground, started at (mean0, var0) with weight initial_weight, and the background,
    started empty with weight 10 (zero mean; zero variance for a diagonal metric, the identity for a dense one).  Sample i
    (0-based) is `delta = i - start` samples into the current window.  It is added to both; then the metric becomes the
    foreground's estimate if (delta + 1) is a multiple of update_window; then, if delta >= the window length, the window
    closes: the background becomes the foreground, a fresh background starts, start = i, and with doubling the window length
    doubles.

    Returns (metric after every sample [N, ...], final metric, indices of the samples that closed a window)."""
    samples = np.asarray(samples, dtype=np.float64)
    var0 = np.asarray(var0, dtype=np.float64)
    n = samples.shape[1]
    dense = var0.ndim == 2

    def empty():
        return _Moments(np.zeros(n), np.eye(n) if dense else np.zeros(n), 10.)

    fg, bg = _Moments(mean0, var0, initial_weight), empty()
    metric = var0.copy()
    start, window = 0, int(adapt_window)
    history, closed = np.empty((len(samples),) + var0.shape), []
    for i, x in enumerate(samples):
        delta = i - start
        fg.add(x)
        bg.add(x)
        if (delta + 1) % update_window == 0:
            metric = fg.estimate()
        if delta >= window:
            fg, bg = bg, empty()
            start = i
            closed.append(i)
            if doubling:
                window *= 2
        history[i] = metric
    return history, metric, closed


def adaptation(rec, n_warmup, step0, var0, mean0, cfg):
    """Adaptation state of every chain of a run, restated from its records.

    rec: dict with 'mean_tree_accept' [C, T] and 'samples' [C, T, n] (T >= n_warmup); step0 [C], var0 [C, n] or [C, n, n],
    mean0 [C, n]; cfg: the sampler settings (target_accept, gamma, k, t0, adapt_step_size, initial_weight, adapt_window,
    update_window, doubling, adapt_metric).  Returns dict(step_size [C, T], step_size_bar [C, T], final_step [C, 4],
    final_var [C, n(, n)]): the records and the final state the sampler must report.  After the warm-up neither changes."""
    acc = np.asarray(rec['mean_tree_accept'])
    C, T = acc.shape
    n_warmup = min(int(n_warmup), T)
    step0 = np.broadcast_to(np.asarray(step0, dtype=np.float64), (C,))
    out = dict(step_size=np.empty((C, T)), step_size_bar=np.empty((C, T)), final_step=np.empty((C, 4)),
               final_var=np.empty(np.shape(var0)))
    for c in range(C):
        if cfg.get('adapt_step_size', 1):
            s, b, f = dual_average(acc[c, :n_warmup], step0[c], cfg['target_accept'], cfg['gamma'], cfg['k'], cfg['t0'])
        else:
            ls = np.log(step0[c])
            s, b, f = np.full(n_warmup, step0[c]), np.full(n_warmup, step0[c]), np.array([ls, ls, 0., 1.])
        out['step_size'][c, :n_warmup], out['step_size_bar'][c, :n_warmup] = s, b
        out['step_size'][c, n_warmup:], out['step_size_bar'][c, n_warmup:] = np.exp(f[0]), np.exp(f[1])
        out['final_step'][c] = f
        if cfg.get('adapt_metric', 1):
            out['final_var'][c] = windowed_metric(rec['samples'][c, :n_warmup], mean0[c], var0[c], cfg['initial_weight'],
                                                  cfg['adapt_window'], cfg['update_window'], cfg['doubling'])[1]
        else:
            out['final_var'][c] = var0[c]
    return out
