"""
sample(): the reference's chain pool (bayesfast/core/sample.py:26-220 + utils/parallel.py) replaced by one
lock-step launch on the GPU: all chains of this process run as warps of one CUDA kernel (csrc/bfb_sampler.cu).
Under torchrun (one process per GPU) pass comm=True: chains are sharded over the ranks, no collective is
needed while sampling.
"""
import time

import numpy as np

from . import _cabi, diag
from .density import Density
from .random import get_generator, new_seed
from .runtime import dist_info, shard_bounds
from .sample_trace import NTrace, HTrace, TNTrace, THTrace, TraceTuple, SampleTrace, DualAverageAdaptation, QuadMetricDiag, QuadMetricFull

__all__ = ['sample']

_ERR = {1: (ValueError, 'failed to get finite logp and/or grad at x_0.'),
        2: (RuntimeError, 'Bad initial energy, please check the Hamiltonian.'),
        3: (FloatingPointError, "logp can't be nan.")}


def _as_density(density):
    if isinstance(density, Density):
        return density
    if hasattr(density, '_surrogate_list'):            # a reference bayesfast.Density (duck-typed)
        return Density.from_reference(density)
    raise ValueError('density should be a bayesfast_b200.Density (or a fitted, surrogate-only bayesfast.Density); '
                     'arbitrary Python densities cannot run on the device and there is no CPU fallback.')


def _out_plan(trace, i_iter, n_run, keep, thin):
    """(skip, thin) for bfb_sampler_run_ex: keep='post_warmup' drops the records of the warm-up iterations still ahead"""
    if keep not in ('all', 'post_warmup'):
        raise ValueError("keep should be 'all' or 'post_warmup'.")
    thin = int(thin)
    if thin < 1:
        raise ValueError('thin should be a positive int.')
    skip = min(max(trace.n_warmup - i_iter, 0), n_run) if keep == 'post_warmup' else 0
    return skip, thin



def _diag_from(trace, i_iter, n_run, diagnostics):
    """first iteration of this call after the warm-up, where the diagnostics start (None: no diagnostics)"""
    if not diagnostics:
        return None
    d = min(max(trace.n_warmup - i_iter, 0), n_run)
    if n_run - d < 4:
        raise ValueError('diagnostics=True needs at least 4 post-warm-up iterations in this call, there are {}.'.format(n_run - d))
    return d


def _diagnostics(res, comm, device):
    """this call's diagnostics over all ranks' chains from the partials bfb_sampler_run_ex left in res"""
    P = res.pop('diag_partials', None)
    if P is None:
        return None
    return diag.finish(diag.combine(P, comm, device))


def sobol_multivariate_normal(dim, size, skip=1):
    """bayesfast.utils.sobol.multivariate_normal(zeros(dim), eye(dim), size) (utils/sobol.py:48-60, utils/_sobol.pyx): the first
    `size` points after `skip` of the Joe-Kuo Sobol sequence (Gray-code order, direction numbers new-joe-kuo-6.21201), mapped through
    the normal quantile function.  scipy's unscrambled qmc.Sobol uses the same direction numbers and order: identical to the
    reference's Cython generator bit for bit (tests/golden/sobol_x0.npz)."""
    from scipy.stats import qmc, norm
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')                # scipy warns when size + skip is not a power of two
        pts = qmc.Sobol(int(dim), scramble=False).random(int(size) + int(skip))[int(skip):]
    a, w = np.linalg.eigh(np.eye(int(dim)))            # the reference's eigen-decomposition of the (identity) covariance
    return (norm.ppf(pts) * a**0.5) @ w.T


def sample(density, sample_trace=None, sampler='NUTS', n_run=None, parallel_backend='b200', verbose=True,
           comm=None, fields=None, keep='all', thin=1, summaries=False, diagnostics=False):
    """
    Sampling a surrogate density with lock-step NUTS / HMC on the GPU.

    Parameters follow bayesfast.core.sample.sample (sample.py:26-60).  `parallel_backend` is accepted for
    signature compatibility and must be 'b200' / None.  `comm`: torch.distributed group (or True) to shard
    the chains over ranks; the returned TraceTuple then holds this rank's chains (global chain ids).
    `fields`: optional subset of outputs to bring back to the host (default: everything).
    `keep='post_warmup'`: the records of the warm-up iterations are never written or copied (SampleTrace.get drops them
    anyway, sample_trace.py:762-787); `thin=k`: of the iterations kept only every k-th record comes back; `summaries=True`:
    mean and covariance (np.cov) of ALL samples after the dropped iterations, over this rank's chains, accumulated on the
    device (tt.summaries).  `diagnostics=True`: split-R-hat and effective sample size (bayesfast_b200.diagnostics) of the samples of
    this call's post-warm-up iterations over all ranks' chains, whatever `fields`, `keep` and `thin` bring back, computed on the
    device (tt.diagnostics = dict(rhat, ess)).  A 4096-chain, 1500-iteration run at n = 26 brings back 1.7 GB per GPU with the defaults,
    1.1 GB with keep='post_warmup', 0.11 GB with thin=10 on top.

    Returns
    -------
    tt : TraceTuple
    """
    if parallel_backend not in (None, 'b200'):
        raise ValueError("bayesfast_b200.sample runs on the GPU only: parallel_backend should be 'b200' or None.")
    den = _as_density(density)
    resume = None
    if isinstance(sample_trace, TraceTuple):
        resume = sample_trace
        sampler = resume.sampler
        trace = resume._template
    elif isinstance(sample_trace, TNTrace):            # before NTrace: the reference tests NTrace first (core/sample.py:64-70)
        sampler, trace = 'TNUTS', sample_trace         # and so runs plain NUTS on a TNTrace; TNUTS is what the trace asks for
    elif isinstance(sample_trace, THTrace):
        sampler, trace = 'THMC', sample_trace
    elif isinstance(sample_trace, NTrace):
        sampler, trace = 'NUTS', sample_trace
    elif isinstance(sample_trace, HTrace):
        sampler, trace = 'HMC', sample_trace
    elif sample_trace is None or isinstance(sample_trace, dict):
        kw = {} if sample_trace is None else sample_trace
        if sampler == 'NUTS':
            trace = NTrace(**kw)
        elif sampler == 'HMC':
            trace = HTrace(**kw)
        elif sampler == 'TNUTS':                       # density_base is a required argument of the trace
            trace = TNTrace(**kw)
        elif sampler == 'THMC':
            trace = THTrace(**kw)
        elif sampler == 'Ensemble':
            raise NotImplementedError('{} is not available on the device.'.format(sampler))
        else:
            raise ValueError('unexpected value for sampler.')
    else:
        raise ValueError('unexpected value for sample_trace.')

    n = den.input_size
    rank, world, _ = dist_info(comm)
    if resume is not None:
        return _continue(den, resume, n_run, verbose, comm)

    if trace.random_generator is None:
        trace.random_generator = new_seed()
        get_generator().normal()                       # sample.py:101
    seed = trace.random_generator
    hostrng = np.random.default_rng(seed)
    C = trace.n_chain
    if trace.x_0 is None:
        x0 = sobol_multivariate_normal(n, C)           # sample.py:107-112: Sobol points through Phi^-1, identity covariance
        trace._x_0_transformed = True
    else:
        x0 = np.asarray(trace.x_0, dtype=np.float64).reshape((-1, trace.x_0.shape[-1]))
        if x0.shape[-1] != n:
            raise ValueError('x_0 should have {} columns.'.format(n))
        if not trace.x_0_transformed:
            x0 = den.from_original(x0)                 # sample.py:113-116
        if x0.shape[0] != C:                           # sample_trace.py:201-205
            x0 = x0[hostrng.integers(0, x0.shape[0], size=C)]
    lo, hi = shard_bounds(C, rank, world)
    x0 = np.ascontiguousarray(x0[lo:hi])
    Cl = hi - lo
    if Cl == 0:
        raise ValueError('rank {} received no chain: n_chain={} < world_size={}.'.format(rank, C, world))

    # sample_trace.py:365-373 and :417-455
    if isinstance(trace._step_size, DualAverageAdaptation):
        step0 = np.full(Cl, np.exp(trace._step_size._log_step))
    else:
        step0 = np.full(Cl, (1. if trace._step_size is None else trace._step_size) / n**0.25)
    m = trace._metric
    dense = False
    if isinstance(m, QuadMetricFull):
        m, dense = m._cov, True
    elif isinstance(m, QuadMetricDiag):
        m = m._var
    elif isinstance(m, str):
        m, dense = (np.eye(n), True) if m == 'full' else (np.ones(n), False)       # sample_trace.py:428-431
    else:
        dense = m.ndim == 2
    if m.shape != ((n, n) if dense else (n,)):
        raise ValueError('metric should have shape ({0},) or ({0}, {0}).'.format(n))
    var0 = np.broadcast_to(m, (Cl, n, n) if dense else (Cl, n))
    mean0 = x0 if trace._initial_mean is None else np.broadcast_to(trace._initial_mean, (Cl, n))

    if sampler in ('TNUTS', 'THMC'):
        if diagnostics:
            raise NotImplementedError('diagnostics are not available for the tempered samplers.')
        return _sample_tempered(den, trace, sampler, n_run, verbose, fields, keep, thin, summaries, seed, lo, x0, step0,
                                dense, var0, mean0)
    h = den._sync(False)
    # a dense mass matrix (metric='full' / a covariance: QuadMetricFull(Adapt), metrics.py:94-132, 240-330) runs on the
    # generic warp-per-chain kernel; the diagonal default takes the tensor-core path
    h.sampler_init(trace._cfg_dict(seed, lo), x0, step0, np.ascontiguousarray(var0), np.ascontiguousarray(mean0), dense=dense)
    n_run = trace.n_iter if n_run is None else int(n_run)
    if n_run <= 0:
        raise ValueError('invalid value for n_run.')
    if n_run > trace.n_iter:
        trace._n_iter = n_run
    t0 = time.time()
    skip, thin = _out_plan(trace, 0, n_run, keep, thin)
    dfrom = _diag_from(trace, 0, n_run, diagnostics)
    res = h.sampler_run(sampler, n_run, fields=fields, skip=skip, thin=thin, summaries=summaries, diag_from=dfrom)
    final = h.sampler_state()
    _raise_status(final['status'], lo)
    dg = _diagnostics(res, comm, h.device)
    final['step0'], final['x_0'] = step0, x0
    arrays = _finish_arrays(den, res)
    tt = TraceTuple(trace, arrays, final, chain0=lo, device_state=h, iters=res['iters'], i_iter=n_run,
                    out_opts=dict(fields=fields, keep=keep, thin=thin, summaries=summaries, diagnostics=bool(diagnostics)),
                    generation=h.generation)
    tt.summaries = {k: res[k] for k in ('mean', 'cov') if k in res}
    tt.diagnostics = dg
    tt.total_tree_size = res['total_tree_size']
    tt.kernel_ms = h.last_kernel_ms()
    if verbose:
        print(' B200 : sampling finished [ {} / {} ], {} chains, {} leapfrog steps in {:.2f} seconds '
              '(kernel {:.1f} ms).'.format(n_run, trace.n_iter, Cl, res['total_tree_size'], time.time() - t0,
                                           tt.kernel_ms))
    return tt


def _sample_tempered(den, trace, sampler, n_run, verbose, fields, keep, thin, summaries, seed, lo, x0, step0, dense, var0, mean0):
    """TNUTS / THMC (samplers/tnuts.py, thmc.py, hmc_utils/base_hmc.py:220-262): the base density sits in a second device handle;
    one warp per chain (csrc/bfb_sampler_tempered.cu).  Full records only."""
    if dense:
        raise NotImplementedError('the tempered samplers run with the diagonal metric on the device.')
    if keep != 'all' or int(thin) != 1 or summaries:
        raise NotImplementedError('reduced outputs (keep / thin / summaries) are not available for the tempered samplers.')
    base = _as_density(trace.density_base)
    if base is den:
        raise ValueError('density_base should be a density object of its own.')
    if base.input_size != den.input_size:
        raise ValueError('density_base should have {} inputs.'.format(den.input_size))
    Cl = x0.shape[0]
    if trace.u_0 is None:
        u0 = np.array([np.random.normal(0, 1) for _ in range(trace.n_chain)])[lo:lo + Cl]     # base_hmc.py:242
    else:
        u0 = np.broadcast_to(trace.u_0, (trace.n_chain,))[lo:lo + Cl]
    h, hb = den._sync(False), base._sync(False)
    h.tsampler_init(hb, trace.logxi, trace._cfg_dict(seed, lo), x0, u0, step0, np.ascontiguousarray(var0),
                    np.ascontiguousarray(mean0))
    n_run = trace.n_iter if n_run is None else int(n_run)
    if n_run <= 0:
        raise ValueError('invalid value for n_run.')
    if n_run > trace.n_iter:
        trace._n_iter = n_run
    t0 = time.time()
    res = h.tsampler_run(sampler, n_run, fields=fields)
    final = h.sampler_state()
    _raise_status(final['status'], lo)
    final['step0'], final['x_0'] = step0, x0
    arrays = _finish_arrays(den, res)
    tt = TraceTuple(trace, arrays, final, chain0=lo, device_state=None, iters=res['iters'], i_iter=n_run,
                    out_opts=dict(fields=fields, keep='all', thin=1, summaries=False), generation=h.generation)
    tt.total_tree_size = res['total_tree_size']
    tt.kernel_ms = h.last_kernel_ms()
    if verbose:
        print(' B200 : {} finished [ {} / {} ], {} chains, {} leapfrog steps in {:.2f} seconds (kernel {:.1f} ms).'.format(
            sampler, n_run, trace.n_iter, Cl, res['total_tree_size'], time.time() - t0, tt.kernel_ms))
    return tt


def _raise_status(status, chain0):
    bad = np.flatnonzero(status)
    if bad.size:
        code = int(status[bad[0]])
        exc, msg = _ERR.get(code, (RuntimeError, 'sampler failed with status {}.'.format(code)))
        raise exc(' CHAIN #{} : {}'.format(chain0 + int(bad[0]), msg))


def _finish_arrays(den, res):
    """sample.py:175-177: samples / logp in the original space"""
    arrays = {k: v for k, v in res.items() if isinstance(v, np.ndarray) and k not in ('iters', 'mean', 'cov')}
    if 'samples' in arrays and 'logp' in arrays:
        if den.input_scales is None:
            arrays['samples_original'] = arrays['samples']
            arrays['logp_original'] = arrays['logp']
        else:
            arrays['samples_original'] = den.to_original(arrays['samples'])
            arrays['logp_original'] = den.to_original_density(arrays['logp'], x_trans=arrays['samples'])
    return arrays


def _continue(den, tt, n_run, verbose, comm=None):
    """in-memory resume (sample.py:91-98, base_hmc.py:101-111): the chains are still resident on the device"""
    h = tt._device_state
    if h is None or h is not den._sync(False) or getattr(h, 'generation', None) != tt._generation:
        raise RuntimeError('these chains are no longer resident on the device (the density changed, or other chains were '
                           'started on it since): cannot continue them.')
    trace = tt._template
    left = trace.n_iter - tt.i_iter
    n_run = left if n_run is None else int(n_run)
    if n_run <= 0:
        raise ValueError('invalid value for n_run.')
    if n_run > left:
        trace._n_iter = tt.i_iter + n_run
    oo = tt._out_opts
    skip, thin = _out_plan(trace, tt.i_iter, n_run, oo['keep'], oo['thin'])
    dfrom = _diag_from(trace, tt.i_iter, n_run, oo.get('diagnostics', False))
    res = h.sampler_run(tt.sampler, n_run, fields=oo['fields'], skip=skip, thin=thin, summaries=oo['summaries'], diag_from=dfrom)
    final = h.sampler_state()
    _raise_status(final['status'], tt._chain0)
    dg = _diagnostics(res, comm, h.device)
    final['step0'], final['x_0'] = tt._final['step0'], tt._final['x_0']
    new = _finish_arrays(den, res)
    arrays = {k: np.concatenate((tt._arrays[k], new[k]), axis=1) for k in new if k in tt._arrays}
    out = TraceTuple(trace, arrays, final, chain0=tt._chain0, device_state=h,
                     iters=np.concatenate((tt._iters, tt.i_iter + res['iters'])), i_iter=tt.i_iter + n_run, out_opts=oo,
                     generation=tt._generation)
    out.summaries = {k: res[k] for k in ('mean', 'cov') if k in res}       # of this call's iterations
    out.diagnostics = dg                                                      # of this call's post-warm-up iterations
    out.total_tree_size = tt.total_tree_size + res['total_tree_size']
    out.kernel_ms = h.last_kernel_ms()
    if verbose:
        print(' B200 : sampling continued [ {} / {} ].'.format(out.i_iter, trace.n_iter))
    return out
