"""
Sampler configuration + result containers with the interface of bayesfast.samplers.sample_trace
(reference: bayesfast/samplers/sample_trace.py:18-847, hmc_utils/stats.py, step_size.py, metrics.py).

A run on the device produces chain-major arrays [C, n_iter(, n)]; TraceTuple owns them and hands out per-chain
NTrace / HTrace objects that are VIEWS into those arrays (the reference keeps python lists of per-iteration
arrays; 4096 chains x 1500 iterations of list appends would dominate the run time).
"""
import warnings
from collections import OrderedDict, namedtuple

import numpy as np

__all__ = ['SampleTrace', 'NTrace', 'HTrace', 'TNTrace', 'THTrace', 'TNStats', 'THStats', 'TraceTuple', 'DualAverageAdaptation', 'QuadMetricDiag',
           'QuadMetricDiagAdapt', 'QuadMetricFull', 'QuadMetricFullAdapt', 'NStats', 'HStats', 'NStepStats', 'HStepStats', '_get_step_size', '_get_metric']

hstats_items = ('logp', 'energy', 'n_int_step', 'accept_stat', 'accepted', 'step_size', 'step_size_bar', 'warmup',
                'energy_change', 'diverging')
nstats_items = ('logp', 'energy', 'tree_depth', 'tree_size', 'mean_tree_accept', 'step_size', 'step_size_bar',
                'warmup', 'energy_change', 'max_energy_change', 'diverging')
# hmc_utils/stats.py:9-24: the tempered samplers put 'u' and 'weight' in front
thstats_items = ('u', 'weight') + hstats_items
tnstats_items = ('u', 'weight') + nstats_items
THStepStats = namedtuple('THStepStats', thstats_items)
TNStepStats = namedtuple('TNStepStats', tnstats_items)
HStepStats = namedtuple('HStepStats', hstats_items)
NStepStats = namedtuple('NStepStats', nstats_items)


class DualAverageAdaptation:
    """State holder + the two read-only methods of step_size.py:10-51 (the update runs on the device)."""

    def __init__(self, initial_step, target, gamma, k, t_0, adapt=True):
        self._log_step = np.log(initial_step)
        self._log_bar = self._log_step
        self._target, self._hbar, self._k, self._t_0 = target, 0., k, t_0
        self._count = 1
        self._mu = np.log(10. * initial_step)
        self._gamma, self._adapt = gamma, adapt

    def current(self, warmup):
        return np.exp(self._log_step) if warmup else np.exp(self._log_bar)

    def sizes(self):
        return {'step_size': np.exp(self._log_step), 'step_size_bar': np.exp(self._log_bar)}


class QuadMetricDiag:
    """metrics.py:51-91 (state only)"""

    def __init__(self, var):
        var = np.atleast_1d(var).astype(np.float64)
        if var.ndim != 1:
            raise ValueError('var should be a 1-d array.')
        if not np.all(var > 0):
            raise ValueError('the input diagonal covariance is not positive definite.')
        self._var = var.copy()
        self._std = var**0.5
        self._inv_std = 1. / self._std
        self._n = len(var)


class QuadMetricDiagAdapt(QuadMetricDiag):
    """metrics.py:135-237 (state only: the windowed Welford update runs on the device)"""


class QuadMetricFull:
    """metrics.py:94-132 (state only): dense mass matrix"""

    def __init__(self, cov):
        cov = np.atleast_2d(cov).astype(np.float64)
        if cov.ndim != 2 or cov.shape[0] != cov.shape[1]:
            raise ValueError('cov should be a 2-d array.')
        if not np.all(np.linalg.eigvalsh(cov) > 0):
            raise ValueError('the input covariance is not positive definite.')
        self._cov = cov.copy()
        self._chol = np.linalg.cholesky(cov)
        self._n = len(cov)


class QuadMetricFullAdapt(QuadMetricFull):
    """metrics.py:240-330 (state only: the windowed Welford covariance and its Cholesky factor live on the device)"""
    _chol_error = None

    def raise_ok(self, vmap=None):
        if self._chol_error is not None:
            raise ValueError('{0}'.format(self._chol_error))


class _Stats:
    def __init__(self, items):
        self._items = items
        for si in items:
            setattr(self, '_' + si, np.empty(0))

    stats_items = property(lambda self: self._items)

    def get(self, since_iter=None, include_warmup=False):
        if since_iter is None:
            since_iter = 0 if include_warmup else self.n_warmup
        since_iter = int(since_iter)
        return OrderedDict((si, getattr(self, '_' + si)[since_iter:]) for si in self._items)

    __call__ = get

    @property
    def n_iter(self):
        return len(self._logp)

    @property
    def n_warmup(self):
        w = np.asarray(self._warmup, dtype=bool)
        idx = np.flatnonzero(~w)
        if idx.size == 0:
            raise ValueError('False is not in list')
        return int(idx[0])


class NStats(_Stats):
    _step_stats = NStepStats

    def __init__(self):
        super().__init__(nstats_items)


class HStats(_Stats):
    _step_stats = HStepStats

    def __init__(self):
        super().__init__(hstats_items)


class TNStats(_Stats):
    """hmc_utils/stats.py:112-118"""
    _step_stats = TNStepStats

    def __init__(self):
        super().__init__(tnstats_items)

    u = property(lambda self: self._u)
    weight = property(lambda self: self._weight)


class THStats(_Stats):
    """hmc_utils/stats.py:103-109"""
    _step_stats = THStepStats

    def __init__(self):
        super().__init__(thstats_items)

    u = property(lambda self: self._u)
    weight = property(lambda self: self._weight)


def _pos_int(v, name, allow_zero=False):
    try:
        v = int(v)
        assert v > 0 or (allow_zero and v == 0)
    except Exception:
        raise ValueError('{} should be a positive int, instead of {}.'.format(name, v))
    return v


class SampleTrace:
    """sample_trace.py:18-154"""

    def __init__(self, n_chain=4, n_iter=1500, n_warmup=500, x_0=None, random_generator=None):
        self._chain_initialized = False
        self._n_chain = _pos_int(n_chain, 'n_chain')
        self._n_iter = _pos_int(n_iter, 'n_iter')
        n_warmup = _pos_int(n_warmup, 'n_warmup')
        if n_warmup >= self._n_iter:
            raise ValueError('n_iter is {}, so n_warmup should be smaller than this number.'.format(self._n_iter))
        self._n_warmup = n_warmup
        self.x_0 = x_0
        self.random_generator = random_generator
        self._x_0_transformed = False

    chain_initialized = property(lambda self: self._chain_initialized)
    n_chain = property(lambda self: self._n_chain)
    n_warmup = property(lambda self: self._n_warmup)
    x_0_transformed = property(lambda self: self._x_0_transformed)

    @property
    def n_iter(self):
        return self._n_iter

    @n_iter.setter
    def n_iter(self, n):
        n = _pos_int(n, 'n_iter')
        if n < self.i_iter:
            raise ValueError('you have already run {} iterations, so n_iter should not be smaller than this '
                             'number.'.format(self.i_iter))
        if n < self._n_warmup:
            raise ValueError('n_warmup is {}, so n_iter should not be smaller than this number.'.format(
                self._n_warmup))
        self._n_iter = n

    def add_iter(self, n):
        self.n_iter = self.n_iter + n

    @property
    def i_iter(self):
        return 0

    @property
    def x_0(self):
        return self._x_0

    @x_0.setter
    def x_0(self, x):
        if self._chain_initialized:
            raise RuntimeError('you should not change x_0 once the chain is initialized.')
        self._x_0 = None if x is None else np.atleast_1d(np.asarray(x, dtype=np.float64)).copy()

    @property
    def input_size(self):
        try:
            return self.x_0.shape[-1]
        except Exception:
            return None

    @property
    def random_generator(self):
        """the 64-bit seed of this trace's Philox streams (None: drawn from bayesfast_b200.random at sample())"""
        return self._random_generator

    @random_generator.setter
    def random_generator(self, generator):
        if generator is None or isinstance(generator, (int, np.integer)):
            self._random_generator = None if generator is None else int(generator)
        else:
            self._random_generator = int(np.random.default_rng(generator).integers(0, 2**63 - 1))


class _HTrace(SampleTrace):
    """sample_trace.py:157-456: options shared by HTrace and NTrace"""

    def __init__(self, n_chain=4, n_iter=1500, n_warmup=500, x_0=None, random_generator=None, step_size=None,
                 adapt_step_size=True, metric='diag', adapt_metric=True, max_change=1000., target_accept=0.8,
                 gamma=0.05, k=0.75, t_0=10., initial_mean=None, initial_weight=10., adapt_window=60,
                 update_window=1, doubling=True):
        super().__init__(n_chain, n_iter, n_warmup, x_0, random_generator)
        self._samples = np.empty((0, 0))
        self._chain_id = None
        try:
            max_change = float(max_change)
            assert max_change > 0
        except Exception:
            raise ValueError('max_change should be a positive float, instead of {}.'.format(max_change))
        self._max_change = max_change
        if isinstance(step_size, DualAverageAdaptation):
            self._step_size = step_size
        else:
            if step_size is not None:
                try:
                    step_size = float(step_size)
                    assert step_size > 0
                except Exception:
                    raise ValueError('invalid value for step_size.')
            self._step_size = step_size
        self._adapt_step_size = bool(adapt_step_size)
        try:
            target_accept = float(target_accept)
            assert 0 < target_accept < 1
        except Exception:
            raise ValueError('invalid value for target_accept.')
        try:
            gamma = float(gamma)
            assert gamma != 0
        except Exception:
            raise ValueError('invalid value for gamma.')
        try:
            k, t_0 = float(k), float(t_0)
            assert t_0 >= 0
        except Exception:
            raise ValueError('invalid value for k or t_0.')
        self._target_accept, self._gamma, self._k, self._t_0 = target_accept, gamma, k, t_0
        # sample_trace.py:375-390, 424-455: 'diag' | 'full' | variances (n,) | covariance (n, n) | a QuadMetric
        if isinstance(metric, (QuadMetricDiag, QuadMetricFull)):
            self._metric = metric
        elif isinstance(metric, str):
            if metric not in ('diag', 'full'):
                raise ValueError('invalid value for metric.')
            self._metric = metric
        else:
            try:
                metric = np.asarray(metric, dtype=np.float64)
                assert metric.ndim == 1 or (metric.ndim == 2 and metric.shape[0] == metric.shape[1])
            except Exception:
                raise ValueError('invalid value for metric.')
            self._metric = metric
        self._adapt_metric = bool(adapt_metric)
        self._initial_mean = None if initial_mean is None else np.atleast_1d(np.asarray(initial_mean, float))
        try:
            initial_weight = float(initial_weight)
            assert initial_weight > 0
        except Exception:
            raise ValueError('invalid value for initial_weight.')
        self._initial_weight = initial_weight
        self._adapt_window = _pos_int(adapt_window, 'adapt_window')
        self._update_window = _pos_int(update_window, 'update_window')
        self._doubling = bool(doubling)

    chain_id = property(lambda self: self._chain_id)
    step_size = property(lambda self: self._step_size)
    metric = property(lambda self: self._metric)
    max_change = property(lambda self: self._max_change)
    stats = property(lambda self: self._stats)

    @property
    def samples(self):
        return np.asarray(self._samples)

    @property
    def samples_original(self):
        return np.asarray(self._samples_original)

    @property
    def i_iter(self):
        try:
            return len(self._samples)
        except Exception:
            return 0

    @property
    def finished(self):
        return self.i_iter >= self.n_iter

    @property
    def logp(self):
        return np.asarray(self.stats._logp)

    @property
    def logp_original(self):
        return np.asarray(self._logp_original)

    _all_return = ['samples', 'logp']

    def get(self, since_iter=None, include_warmup=False, original_space=True, return_type='samples', flatten=True):
        """sample_trace.py:278-310"""
        if return_type == 'all':
            return [self.get(since_iter, include_warmup, original_space, _, flatten) for _ in self._all_return]
        if since_iter is None:
            since_iter = 0 if include_warmup else self.n_warmup
        since_iter = int(since_iter)
        if since_iter >= self.i_iter - 1:
            raise ValueError('since_iter is too large. Nothing to return.')
        if return_type == 'samples':
            return (self.samples_original if original_space else self.samples)[since_iter:]
        if return_type == 'logp':
            return (self.logp_original if original_space else self.logp)[since_iter:]
        raise ValueError('invalid value for return_type.')

    __call__ = get

    def _cfg_dict(self, seed, chain0):
        """the bfb_sampler_cfg fields (include/bfb200.h)"""
        return dict(n_warmup=self._n_warmup, max_treedepth=getattr(self, '_max_treedepth', 10),
                    n_int_step=getattr(self, '_n_int_step', 0), max_change=self._max_change,
                    adapt_step_size=int(self._adapt_step_size), target_accept=self._target_accept,
                    gamma=self._gamma, k=self._k, t0=self._t_0, adapt_metric=int(self._adapt_metric),
                    initial_weight=self._initial_weight, adapt_window=self._adapt_window,
                    update_window=self._update_window, doubling=int(self._doubling), seed=int(seed),
                    chain0=int(chain0))


class HTrace(_HTrace):
    """sample_trace.py:458-496"""

    def __init__(self, n_chain=4, n_iter=1500, n_warmup=500, n_int_step=32, x_0=None, random_generator=None,
                 step_size=1., **kwargs):
        super().__init__(n_chain, n_iter, n_warmup, x_0, random_generator, step_size, **kwargs)
        self._n_int_step = _pos_int(n_int_step, 'n_int_step')
        self._stats = HStats()

    n_int_step = property(lambda self: self._n_int_step)

    @property
    def n_call(self):
        return self.n_iter * (self.n_int_step + 1) + 1


class NTrace(_HTrace):
    """sample_trace.py:499-537"""

    def __init__(self, n_chain=4, n_iter=1500, n_warmup=500, x_0=None, random_generator=None, step_size=1.,
                 adapt_step_size=True, metric='diag', adapt_metric=True, max_change=1000., max_treedepth=10,
                 **kwargs):
        super().__init__(n_chain, n_iter, n_warmup, x_0, random_generator, step_size, adapt_step_size, metric,
                         adapt_metric, max_change, **kwargs)
        self._max_treedepth = _pos_int(max_treedepth, 'max_treedepth')
        self._stats = NStats()

    max_treedepth = property(lambda self: self._max_treedepth)

    @property
    def n_call(self):
        return int(np.sum(self._stats._tree_size[1:])) + self.n_iter + 1


class _TTrace:
    """sample_trace.py:540-588: the base density and log xi of the tempered samplers; get(return_type='weights')"""

    def _t_init(self, density_base, logxi, u_0):
        if not (hasattr(density_base, 'logp_and_grad') or hasattr(density_base, '_surrogate_list')):
            raise ValueError('invalid value for density_base.')
        self._density_base = density_base
        try:
            self._logxi = float(logxi)
        except Exception:
            raise ValueError('invalid value for logxi.')
        self._u_0 = None if u_0 is None else np.atleast_1d(np.asarray(u_0, dtype=np.float64))

    density_base = property(lambda self: self._density_base)
    logxi = property(lambda self: self._logxi)
    u_0 = property(lambda self: self._u_0)
    weights = property(lambda self: np.asarray(self.stats._weight))

    _all_return = ['samples', 'logp', 'weights']

    def get(self, since_iter=None, include_warmup=False, original_space=True, return_type='samples', flatten=True):
        if return_type == 'weights':                   # sample_trace.py:574-585
            if since_iter is None:
                since_iter = 0 if include_warmup else self.n_warmup
            if int(since_iter) >= self.i_iter - 1:
                raise ValueError('since_iter is too large. Nothing to return.')
            return self.weights[int(since_iter):]
        return _HTrace.get(self, since_iter, include_warmup, original_space, return_type, flatten)

    __call__ = get


class THTrace(_TTrace, HTrace):
    """Trace of the THMC sampler (sample_trace.py:590-604; the reference's own constructor raises -- it calls
    HTrace.__init__ without self -- so this follows what it evidently means).  u_0: tempering variable of the first iteration,
    one per chain (default: numpy's global generator, base_hmc.py:242)."""

    def __init__(self, density_base, logxi=0., n_chain=4, n_iter=1500, n_warmup=500, n_int_step=32, x_0=None,
                 random_generator=None, step_size=1., u_0=None, **kwargs):
        self._t_init(density_base, logxi, u_0)
        HTrace.__init__(self, n_chain, n_iter, n_warmup, n_int_step, x_0, random_generator, step_size, **kwargs)
        self._stats = THStats()


class TNTrace(_TTrace, NTrace):
    """Trace of the TNUTS sampler (sample_trace.py:607-622).  u_0 as in THTrace."""

    def __init__(self, density_base, logxi=0., n_chain=4, n_iter=1500, n_warmup=500, x_0=None, random_generator=None,
                 step_size=1., u_0=None, **kwargs):
        self._t_init(density_base, logxi, u_0)
        NTrace.__init__(self, n_chain, n_iter, n_warmup, x_0, random_generator, step_size, **kwargs)
        self._stats = TNStats()


class TraceTuple:
    """
    Results of all chains of one sample() call (sample_trace.py:631-801).  `arrays` maps names to chain-major
    numpy arrays: samples [C, n_iter, n], samples_original, logp_original and the stats fields [C, n_iter].
    """

    def __init__(self, template, arrays, final_state, chain0=0, device_state=None, iters=None, i_iter=None, out_opts=None,
                 generation=None):
        self._template = template
        self._sampler = ('TNUTS' if isinstance(template, TNTrace) else 'THMC' if isinstance(template, THTrace) else
                         'NUTS' if isinstance(template, NTrace) else 'HMC')
        self._arrays = arrays
        self._final = final_state
        self._chain0 = int(chain0)
        self._device_state = device_state       # live device handle: lets sample() continue these chains
        self._generation = generation           # ... as long as nothing else was started on it since (Handle.generation)
        self._out_opts = out_opts or dict(fields=None, keep='all', thin=1, summaries=False)
        n_rec = next(iter(arrays.values())).shape[1] if arrays else 0
        # iteration index of every stored record (sample(keep='post_warmup', thin=k) stores a subset) and iterations done
        self._iters = np.arange(n_rec) if iters is None else np.asarray(iters)
        self._i_iter = n_rec if i_iter is None else int(i_iter)
        self.total_tree_size = 0
        self.summaries = {}
        self.diagnostics = None                 # sample(diagnostics=True): dict(rhat, ess) of the call's post-warm-up iterations
        self._cache = {}

    def _arr(self, name):
        try:
            return self._arrays[name]
        except KeyError:
            raise KeyError("'{}' was not brought back to the host (sample(fields=...)).".format(name)) from None

    sampler = property(lambda self: self._sampler)
    n_chain = property(lambda self: next(iter(self._arrays.values())).shape[0])
    n_iter = property(lambda self: self._template.n_iter)
    n_warmup = property(lambda self: self._template.n_warmup)
    i_iter = property(lambda self: self._i_iter)
    iters = property(lambda self: self._iters)
    input_size = property(lambda self: self._arr('samples').shape[-1])
    samples = property(lambda self: self._arr('samples'))
    samples_original = property(lambda self: self._arr('samples_original'))
    logp = property(lambda self: self._arr('logp'))
    logp_original = property(lambda self: self._arr('logp_original'))
    finished = property(lambda self: self.i_iter >= self.n_iter)
    arrays = property(lambda self: self._arrays)

    @property
    def n_call(self):
        if self._sampler in ('NUTS', 'TNUTS'):
            if len(self._iters) == self._i_iter and 'tree_size' in self._arrays:
                return int(np.sum(self._arrays['tree_size'][:, 1:])) + self.n_chain * (self.n_iter + 1)
            return int(self.total_tree_size) + self.n_chain * (self.n_iter + 1)      # reduced records: all iterations counted
        return self.n_chain * (self.n_iter * (self._template.n_int_step + 1) + 1)

    def _make(self, i):
        import copy
        t = copy.copy(self._template)
        t._chain_id = self._chain0 + i
        t._chain_initialized = True
        A = self._arrays
        for name in ('samples', 'samples_original', 'logp_original'):
            setattr(t, '_' + name, A[name][i] if name in A else None)
        t._x_0 = None if self._final.get('x_0') is None else self._final['x_0'][i]
        st = {'NUTS': NStats, 'HMC': HStats, 'TNUTS': TNStats, 'THMC': THStats}[self._sampler]()
        warm = self._iters < t._n_warmup
        alias = {'diverging': ('diverging', bool), 'n_int_step': ('tree_size', None), 'accepted': ('tree_depth', bool),
                 'accept_stat': ('mean_tree_accept', None)}
        for si in st.stats_items:
            if si == 'warmup':
                v = warm
            else:
                key, cast = alias.get(si, (si, None))
                if key not in A:                      # sample(fields=...) left this statistic on the device
                    continue
                v = A[key][i].astype(cast) if cast else A[key][i]
            setattr(st, '_' + si, v)
        t._stats = st
        fs = self._final['final_step'][i]
        da = DualAverageAdaptation(float(self._final['step0'][i]), t._target_accept, t._gamma, t._k, t._t_0,
                                   t._adapt_step_size)
        da._log_step, da._log_bar, da._hbar, da._count = float(fs[0]), float(fs[1]), float(fs[2]), int(fs[3])
        t._step_size = da
        fv = self._final['final_var'][i]
        if fv.ndim == 2:
            t._metric = (QuadMetricFullAdapt if t._adapt_metric else QuadMetricFull)(fv)
            if 'chol_error' in self._final and self._final['chol_error'][i]:
                t._metric._chol_error = 'a Cholesky factorisation of the adapted covariance failed (metrics.py:284-287).'
        else:
            t._metric = (QuadMetricDiagAdapt if t._adapt_metric else QuadMetricDiag)(fv)
        return t

    @property
    def sample_traces(self):
        return tuple(self[i] for i in range(self.n_chain))

    def __getitem__(self, key):
        if isinstance(key, slice):
            return tuple(self[i] for i in range(*key.indices(self.n_chain)))
        key = int(key)
        if key < 0:
            key += self.n_chain
        if not 0 <= key < self.n_chain:
            raise IndexError('chain index out of range.')
        if key not in self._cache:
            self._cache[key] = self._make(key)
        return self._cache[key]

    def __len__(self):
        return self.n_chain

    def __iter__(self):
        return (self[i] for i in range(self.n_chain))

    @property
    def stats(self):
        return [t.stats for t in self]

    def get(self, since_iter=None, include_warmup=False, original_space=True, return_type='samples', flatten=True):
        """sample_trace.py:762-787, without materialising the per-chain objects"""
        if return_type == 'all':
            return [self.get(since_iter, include_warmup, original_space, _, flatten) for _ in ('samples', 'logp')]
        if since_iter is None:
            since_iter = 0 if include_warmup else self.n_warmup
        since_iter = int(since_iter)
        if since_iter >= self.i_iter - 1:
            raise ValueError('since_iter is too large. Nothing to return.')
        first = int(np.searchsorted(self._iters, since_iter))         # stored records may be a subset of the iterations
        if return_type == 'samples':
            s = (self.samples_original if original_space else self.samples)[:, first:]
            return s.reshape((-1, self.input_size)) if flatten else s
        if return_type == 'logp':
            l = (self.logp_original if original_space else self.logp)[:, first:]
            return l.flatten() if flatten else l
        raise ValueError('invalid value for return_type.')

    __call__ = get


def _get_step_size(sample_trace):
    """sample_trace.py:804-817"""
    if isinstance(sample_trace, TraceTuple):
        fs = sample_trace._final['final_step']
        return float(np.mean(np.exp(fs[:, 1]))) * sample_trace.input_size**0.25
    if isinstance(sample_trace, _HTrace):
        return sample_trace.step_size.current(False) * sample_trace.input_size**0.25
    raise ValueError('invalid value for sample_trace.')


def _get_metric(sample_trace, target, from_samples=True):
    """sample_trace.py:820-847"""
    if from_samples:
        cov = np.cov(sample_trace.get(original_space=False, flatten=True), rowvar=False)
    elif isinstance(sample_trace, TraceTuple):
        fv = np.mean(sample_trace._final['final_var'], axis=0)
        cov = fv if fv.ndim == 2 else np.diag(fv)
    elif isinstance(sample_trace, _HTrace):
        m = sample_trace.metric
        cov = np.copy(m._cov) if isinstance(m, QuadMetricFull) else np.diag(m._var)
    else:
        raise ValueError('invalid value for sample_trace.')
    if target == 'diag':
        return np.diag(cov)
    if target == 'full':
        return cov
    raise ValueError('unexpected value for target.')


def _warn(msg):
    warnings.warn(msg, RuntimeWarning)
