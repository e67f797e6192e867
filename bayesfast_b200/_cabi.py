"""
ctypes binding of libbfb200.so (include/bfb200.h).  There is no CPU fallback: importing is cheap, but
the first call that needs the device raises if the library or a CUDA device is missing.
"""
import ctypes as C
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('BFB200_LIB', os.path.join(_HERE, 'libbfb200.so'))     # BFB200_LIB: experiment builds

BFB_HOST, BFB_DEVICE = 0, 1
ORDER_CODE = {'linear': 1, 'quadratic': 2, 'cubic-2': 3, 'cubic-3': 4}
SAMPLER_CODE = {'NUTS': 0, 'HMC': 1}

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)
_lp = C.POINTER(C.c_int64)
_bp = C.POINTER(C.c_uint8)


class ModelDesc(C.Structure):
    _fields_ = [('n', C.c_int32), ('m', C.c_int32), ('n_config', C.c_int32),
                ('cfg_order', _ip), ('cfg_n_in', _ip), ('cfg_n_out', _ip),
                ('cfg_in_mask', _lp), ('cfg_out_mask', _lp), ('cfg_coef', _dp),
                ('use_bound', C.c_int32), ('mu', _dp), ('hess', _dp), ('alpha', C.c_double), ('f_mu', _dp),
                ('use_scales', C.c_int32), ('s0', _dp), ('sdiff', _dp),
                ('use_decay', C.c_int32), ('d_mu', _dp), ('d_hess', _dp), ('d_alpha2', C.c_double),
                ('d_gamma', C.c_double),
                ('use_transform', C.c_int32), ('ranges', _dp), ('hard_bounds', _bp)]


class SamplerCfg(C.Structure):
    _fields_ = [('n_warmup', C.c_int32), ('max_treedepth', C.c_int32), ('n_int_step', C.c_int32),
                ('max_change', C.c_double), ('adapt_step_size', C.c_int32), ('target_accept', C.c_double),
                ('gamma', C.c_double), ('k', C.c_double), ('t0', C.c_double), ('adapt_metric', C.c_int32),
                ('initial_weight', C.c_double), ('adapt_window', C.c_int32), ('update_window', C.c_int32),
                ('doubling', C.c_int32), ('seed', C.c_uint64), ('chain0', C.c_int64)]


class RunOut(C.Structure):
    _fields_ = [('samples', C.c_void_p), ('logp', C.c_void_p), ('energy', C.c_void_p),
                ('mean_tree_accept', C.c_void_p), ('step_size', C.c_void_p), ('step_size_bar', C.c_void_p),
                ('energy_change', C.c_void_p), ('max_energy_change', C.c_void_p),
                ('tree_depth', C.c_void_p), ('tree_size', C.c_void_p), ('diverging', C.c_void_p)]


class RunOpts(C.Structure):
    _fields_ = [('skip', C.c_int32), ('thin', C.c_int32), ('mean', C.c_void_p), ('cov', C.c_void_p),
                ('diag_from', C.c_int32), ('diag', C.c_void_p)]


FLOAT_STATS = ('logp', 'energy', 'mean_tree_accept', 'step_size', 'step_size_bar', 'energy_change',
               'max_energy_change')
INT_STATS = ('tree_depth', 'tree_size', 'diverging')

_lib = None
_lock = threading.Lock()


class BfbError(RuntimeError):
    pass


def lib():
    """Load libbfb200.so; raises if it has not been built (python __graft_entry__.py / make -C bayesfast_b200/csrc)."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise BfbError('libbfb200.so is missing at {}: build it with `make -C bayesfast_b200/csrc` '
                               '(there is no CPU fallback).'.format(LIB_PATH))
            L = C.CDLL(LIB_PATH)
            L.bfb_last_error.restype = C.c_char_p
            L.bfb_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
            L.bfb_destroy.argtypes = [C.c_void_p]
            L.bfb_set_stream.argtypes = [C.c_void_p, C.c_void_p]
            L.bfb_synchronize.argtypes = [C.c_void_p]
            L.bfb_set_model.argtypes = [C.c_void_p, C.POINTER(ModelDesc)]
            L.bfb_poly_eval_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int]
            L.bfb_logp_and_grad_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int]
            L.bfb_fit_begin.argtypes = [C.c_void_p, C.c_void_p]
            L.bfb_set_epilogue.argtypes = [C.c_void_p, C.c_int, C.c_double]
            L.bfb_set_prior.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_double]
            L.bfb_sampler_init.argtypes = [C.c_void_p, C.POINTER(SamplerCfg), C.c_int64, _dp, _dp, _dp, _dp]
            L.bfb_sampler_init_dense.argtypes = [C.c_void_p, C.POINTER(SamplerCfg), C.c_int64, _dp, _dp, _dp, _dp]
            L.bfb_sampler_get_cov.argtypes = [C.c_void_p, _dp, _ip]
            L.bfb_sampler_reset.argtypes = [C.c_void_p]
            L.bfb_sampler_run.argtypes = [C.c_void_p, C.c_int, C.c_int32, C.POINTER(RunOut), C.c_int, _lp]
            L.bfb_sampler_run_ex.argtypes = [C.c_void_p, C.c_int, C.c_int32, C.POINTER(RunOut), C.c_int, C.POINTER(RunOpts), _lp]
            L.bfb_tsampler_init.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.POINTER(SamplerCfg), C.c_int64, _dp, _dp, _dp, _dp, _dp]
            L.bfb_tsampler_run.argtypes = [C.c_void_p, C.c_int, C.c_int32, C.POINTER(RunOut), C.c_void_p, C.c_void_p, C.c_int, _lp]
            L.bfb_sampler_get_state.argtypes = [C.c_void_p, _dp, _dp, _lp, _ip, _dp]
            L.bfb_last_kernel_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
            L.bfb_launch_count.argtypes = [C.c_void_p]
            L.bfb_launch_count.restype = C.c_int64
            L.bfb_rng_fill.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int64, _dp, _dp]
            L.bfb_fp64_peak.argtypes = [C.c_void_p, C.c_int, _dp]
            L.bfb_dmma_issue_test.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _dp]
            L.bfb_sampler_last_path.argtypes = [C.c_void_p]
            L.bfb_eval_last_path.argtypes = [C.c_void_p]
            for name, args, res in (
                    ('bfb_fit_accumulate', [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int], C.c_int),
                    ('bfb_fit_buffer_size', [C.c_void_p], C.c_int64),
                    ('bfb_fit_buffer', [C.c_void_p, C.POINTER(C.c_void_p)], C.c_int),
                    ('bfb_fit_exchange_pack', [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)], C.c_int),
                    ('bfb_fit_exchange_host', [C.c_void_p, C.c_void_p, C.c_int], C.c_int),
                    ('bfb_fit_exchange_unpack', [C.c_void_p], C.c_int),
                    ('bfb_fit_solve', [C.c_void_p, _dp, _dp], C.c_int),
                    ('bfb_fit_moments', [C.c_void_p, _dp, _dp], C.c_int),
                    ('bfb_fit_max_beta', [C.c_void_p, C.c_void_p, C.c_int64, _dp, _dp, C.POINTER(C.c_double), C.c_void_p, C.c_int], C.c_int),
                    ('bfb_chain_diagnostics', [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int,
                                               C.c_void_p], C.c_int),
                    ('bfb_norminv_fill', [C.c_void_p, _dp, C.c_int64, _dp, _dp], C.c_int),
                    ):
                if hasattr(L, name):
                    f = getattr(L, name)
                    f.argtypes, f.restype = args, res
            _lib = L
    return _lib


def exported_symbols():
    """Names declared in include/bfb200.h (used by the CPU-side ABI test)."""
    import re
    hdr = os.path.join(_HERE, '..', 'include', 'bfb200.h')
    txt = open(hdr).read()
    return sorted(set(re.findall(r'\b(bfb_[a-z0-9_]+)\s*\(', txt)))


def check(rc):
    if rc != 0:
        raise BfbError('libbfb200: {} (code {})'.format(lib().bfb_last_error().decode(), rc))


def _d(a):
    return a.ctypes.data_as(_dp)


def f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def n_packed(order, n_in):
    """poly.py:110-129 (_a_shape)"""
    return {'linear': n_in + 1, 'quadratic': n_in * (n_in + 1) // 2, 'cubic-2': n_in * n_in,
            'cubic-3': n_in * (n_in - 1) * (n_in - 2) // 6}[order]


class Handle:
    """One device context (one CUDA stream, one model, one set of chains)."""

    def __init__(self, device=0):
        self._h = C.c_void_p()
        self._L = lib()
        check(self._L.bfb_create(int(device), C.byref(self._h)))
        self.device = int(device)
        self.n = self.m = None
        self._keep = None

    def close(self):
        if getattr(self, '_h', None) is not None and self._h.value:
            self._L.bfb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream_ptr):
        check(self._L.bfb_set_stream(self._h, C.c_void_p(int(cuda_stream_ptr))))

    def synchronize(self):
        check(self._L.bfb_synchronize(self._h))

    # ------------------------------------------------------------------ model
    def set_model(self, spec):
        """spec: the dict produced by PolyModel.to_spec() / Density.to_spec() with packed coefficients
        (key 'packed' per config, shape (n_out, n_packed))."""
        n, m = int(spec['n']), int(spec['m'])
        self.generation = getattr(self, 'generation', 0) + 1      # chains set up before this call belong to another model
        cfgs = spec['configs']
        d = ModelDesc()
        order = np.array([ORDER_CODE[c['order']] for c in cfgs], np.int32)
        n_in = np.array([len(c['input_mask']) for c in cfgs], np.int32)
        n_out = np.array([len(c['output_mask']) for c in cfgs], np.int32)
        im = np.concatenate([np.asarray(c['input_mask'], np.int64) for c in cfgs])
        om = np.concatenate([np.asarray(c['output_mask'], np.int64) for c in cfgs])
        parts = []
        for c in cfgs:
            npk = n_packed(c['order'], len(c['input_mask']))
            p = c.get('packed', None)
            p = np.zeros((len(c['output_mask']), npk)) if p is None else f64(p).reshape(len(c['output_mask']), npk)
            parts.append(p.ravel())
        coef = f64(np.concatenate(parts))
        keep = [order, n_in, n_out, im, om, coef]
        d.n, d.m, d.n_config = n, m, len(cfgs)
        d.cfg_order, d.cfg_n_in, d.cfg_n_out = (a.ctypes.data_as(_ip) for a in (order, n_in, n_out))
        d.cfg_in_mask, d.cfg_out_mask = im.ctypes.data_as(_lp), om.ctypes.data_as(_lp)
        d.cfg_coef = _d(coef)
        d.use_bound = int(bool(spec.get('use_bound', False)))
        if d.use_bound:
            mu, hess, fmu = f64(spec['mu']), f64(spec['hess']), f64(np.atleast_1d(spec['f_mu']))
            keep += [mu, hess, fmu]
            d.mu, d.hess, d.f_mu, d.alpha = _d(mu), _d(hess), _d(fmu), float(spec['alpha'])
        sc = spec.get('input_scales', None)
        d.use_scales = int(sc is not None)
        if sc is not None:
            sc = f64(sc)
            s0, sd = f64(sc[:, 0]), f64(sc[:, 1] - sc[:, 0])
            keep += [s0, sd]
            d.s0, d.sdiff = _d(s0), _d(sd)
        d.use_decay = int(bool(spec.get('use_decay', False)))
        if d.use_decay:
            dmu, dh = f64(spec['d_mu']), f64(spec['d_hess'])
            keep += [dmu, dh]
            d.d_mu, d.d_hess = _d(dmu), _d(dh)
            d.d_alpha2, d.d_gamma = float(spec['d_alpha2']), float(spec['d_gamma'])
        tr = spec.get('transform_ranges', None)
        d.use_transform = int(tr is not None)
        if tr is not None:
            rg, hb = f64(tr), np.ascontiguousarray(spec['hard_bounds'], np.uint8)
            keep += [rg, hb]
            d.ranges, d.hard_bounds = _d(rg), hb.ctypes.data_as(_bp)
        check(self._L.bfb_set_model(self._h, C.byref(d)))
        self.n, self.m = n, m
        self._keep = keep
        pr = spec.get('prior', None)              # dict(idx, mu, sig, c0): Gaussian prior on original-space inputs (third module)
        if pr is not None:
            w, mu = np.zeros(n), np.zeros(n)
            idx = np.asarray(pr['idx'], dtype=np.int64)
            w[idx] = 1. / np.asarray(pr['sig'], dtype=np.float64)**2
            mu[idx] = np.asarray(pr['mu'], dtype=np.float64)
            check(self._L.bfb_set_prior(self._h, w.ctypes.data, mu.ctypes.data, float(pr.get('c0', 0.))))
        ss = spec.get('epilogue_sumsq', None)     # set by Density._sync: logp = c0 - 1/2 sum_o f_o^2 over whitened outputs
        if ss is not None:
            check(self._L.bfb_set_epilogue(self._h, 1, float(ss)))

    def poly_eval_batch(self, X, want_jac=True):
        X = f64(X).reshape(-1, self.n)
        F = np.empty((X.shape[0], self.m))
        J = np.empty((X.shape[0], self.m, self.n)) if want_jac else None
        check(self._L.bfb_poly_eval_batch(self._h, X.ctypes.data, X.shape[0], F.ctypes.data,
                                          J.ctypes.data if want_jac else None, BFB_HOST))
        return F, J

    def logp_and_grad_batch(self, X):
        X = f64(X).reshape(-1, self.n)
        lp = np.empty(X.shape[0])
        g = np.empty((X.shape[0], self.n))
        check(self._L.bfb_logp_and_grad_batch(self._h, X.ctypes.data, X.shape[0], lp.ctypes.data, g.ctypes.data,
                                              BFB_HOST))
        return lp, g

    # device-pointer variants (torch tensors): pointers are ints
    def poly_eval_batch_dev(self, x_ptr, C_, f_ptr, j_ptr):
        check(self._L.bfb_poly_eval_batch(self._h, x_ptr, int(C_), f_ptr, j_ptr, BFB_DEVICE))

    def logp_and_grad_batch_dev(self, x_ptr, C_, lp_ptr, g_ptr):
        check(self._L.bfb_logp_and_grad_batch(self._h, x_ptr, int(C_), lp_ptr, g_ptr, BFB_DEVICE))

    # ------------------------------------------------------------------ sampler
    def sampler_init(self, cfg, x0, step0, var0, mean0, dense=False):
        n = self.n
        self.generation = getattr(self, 'generation', 0) + 1      # a TraceTuple of earlier chains can no longer be continued
        x0 = f64(x0).reshape(-1, n)
        nc = x0.shape[0]
        c = SamplerCfg()
        for k, v in cfg.items():
            setattr(c, k, v)
        step0 = f64(np.broadcast_to(step0, (nc,)))
        mean0 = f64(np.broadcast_to(mean0, (nc, n)))
        # dense: var0 is a covariance (n, n) / (C, n, n) -- dense mass matrix (metrics.py:94-132, 240-330)
        self.dense = bool(dense)
        if self.dense:
            cov0 = f64(np.broadcast_to(var0, (nc, n, n)))
            check(self._L.bfb_sampler_init_dense(self._h, C.byref(c), nc, _d(x0), _d(step0), _d(cov0), _d(mean0)))
        else:
            var0 = f64(np.broadcast_to(var0, (nc, n)))
            check(self._L.bfb_sampler_init(self._h, C.byref(c), nc, _d(x0), _d(step0), _d(var0), _d(mean0)))
        self.n_chain = nc

    def sampler_run(self, sampler, n_iter, out_ptrs=None, fields=None, skip=0, thin=1, summaries=False, diag_from=None):
        """Host outputs (default): returns dict of numpy arrays [C, n_keep(, n)], n_keep = ceil((n_iter - skip) / thin):
        the records of the first `skip` iterations are not produced, of the rest every thin-th is kept ('iters': their
        iteration index within this call).  summaries: 'mean' [n] and 'cov' [n, n] of the samples of all iterations after
        `skip` over all chains, accumulated on the device (bfb_sampler_run_ex).  diag_from: 'diag_partials' [n, L + 3] of the
        split-R-hat / ESS diagnostics over iterations diag_from .. n_iter - 1, L = (n_iter - diag_from) // 2 (bfb_chain_diagnostics).
        out_ptrs: dict name -> device pointer (int) for device-resident outputs, laid out [C, n_iter - skip(, n)]."""
        ro = RunOut()
        res = {}
        nc, n = self.n_chain, self.n
        skip, thin = int(skip), int(thin)
        n_keep = (int(n_iter) - skip + thin - 1) // thin
        if out_ptrs is None:
            want = fields if fields is not None else ('samples',) + FLOAT_STATS + INT_STATS
            from . import _pinned
            for k in want:
                if k == 'samples':
                    res[k] = _pinned.empty((nc, n_keep, n))
                elif k in FLOAT_STATS:
                    res[k] = _pinned.empty((nc, n_keep))
                else:
                    res[k] = _pinned.empty((nc, n_keep), np.int32)
                setattr(ro, k, res[k].ctypes.data)
            loc = BFB_HOST
        else:
            for k, p in out_ptrs.items():
                setattr(ro, k, int(p))
            loc = BFB_DEVICE
        op = RunOpts()
        op.skip, op.thin = skip, thin
        if summaries:
            res['mean'], res['cov'] = np.empty(n), np.empty((n, n))
            op.mean, op.cov = res['mean'].ctypes.data, res['cov'].ctypes.data
        if diag_from is not None:
            res['diag_partials'] = np.empty((n, (int(n_iter) - int(diag_from)) // 2 + 3))
            op.diag_from, op.diag = int(diag_from), res['diag_partials'].ctypes.data
        tot = C.c_int64(0)
        check(self._L.bfb_sampler_run_ex(self._h, SAMPLER_CODE[sampler.upper()], int(n_iter), C.byref(ro), loc,
                                         C.byref(op), C.byref(tot)))
        res['total_tree_size'] = int(tot.value)
        res['iters'] = skip + thin * np.arange(n_keep)
        self.generation_runs = getattr(self, 'generation_runs', 0) + 1
        return res

    # ------------------------------------------------------------------ tempered samplers (TNUTS / THMC)
    def tsampler_init(self, base, logxi, cfg, x0, u0, step0, var0, mean0):
        """base: Handle holding the base density's model (TNTrace.density_base); u0 [C]: tempering variable of the first iteration"""
        n = self.n
        self.generation = getattr(self, 'generation', 0) + 1
        x0 = f64(x0).reshape(-1, n)
        nc = x0.shape[0]
        c = SamplerCfg()
        for k, v in cfg.items():
            setattr(c, k, v)
        step0 = f64(np.broadcast_to(step0, (nc,)))
        mean0 = f64(np.broadcast_to(mean0, (nc, n)))
        var0 = f64(np.broadcast_to(var0, (nc, n)))
        u0 = f64(np.broadcast_to(u0, (nc,)))
        self.dense = False
        self._tbase = base                                         # keeps the base handle alive as long as these chains
        check(self._L.bfb_tsampler_init(self._h, base._h, float(logxi), C.byref(c), nc, _d(x0), _d(u0), _d(step0), _d(var0),
                                        _d(mean0)))
        self.n_chain = nc

    def tsampler_run(self, sampler, n_iter, fields=None):
        """sampler 'TNUTS' / 'THMC'; returns dict of host arrays [C, n_iter(, n)] incl. 'u' and 'weight'"""
        ro = RunOut()
        res = {}
        nc, n, n_iter = self.n_chain, self.n, int(n_iter)
        want = fields if fields is not None else ('samples', 'u', 'weight') + FLOAT_STATS + INT_STATS
        for k in want:
            if k == 'samples':
                res[k] = np.empty((nc, n_iter, n))
            elif k in FLOAT_STATS or k in ('u', 'weight'):
                res[k] = np.empty((nc, n_iter))
            else:
                res[k] = np.empty((nc, n_iter), np.int32)
            if k not in ('u', 'weight'):
                setattr(ro, k, res[k].ctypes.data)
        tot = C.c_int64(0)
        pu = res['u'].ctypes.data if 'u' in res else None
        pw = res['weight'].ctypes.data if 'weight' in res else None
        check(self._L.bfb_tsampler_run(self._h, SAMPLER_CODE[sampler.upper()[1:]], n_iter, C.byref(ro), pu, pw, BFB_HOST,
                                       C.byref(tot)))
        res['total_tree_size'] = int(tot.value)
        res['iters'] = np.arange(n_iter)
        return res

    def sampler_reset(self):
        check(self._L.bfb_sampler_reset(self._h))

    def sampler_state(self):
        nc, n = self.n_chain, self.n
        fs, fv, q = np.empty((nc, 4)), np.empty((nc, n)), np.empty((nc, n))
        nd, stt = np.empty(nc, np.int64), np.empty(nc, np.int32)
        check(self._L.bfb_sampler_get_state(self._h, _d(fs), _d(fv), nd.ctypes.data_as(_lp), stt.ctypes.data_as(_ip),
                                            _d(q)))
        res = dict(final_step=fs, final_var=fv, n_draws=nd, status=stt, q=q)
        if getattr(self, 'dense', False):
            cov, ce = np.empty((nc, n, n)), np.empty(nc, np.int32)
            check(self._L.bfb_sampler_get_cov(self._h, _d(cov), ce.ctypes.data_as(_ip)))
            res['final_var'] = cov
            res['chol_error'] = ce
        return res

    def chain_diagnostics(self, x, C_, T, t0, N, n, loc):
        """partials [n, N // 2 + 3] of bfb_chain_diagnostics; x: host array (loc BFB_HOST) or device pointer (BFB_DEVICE)"""
        P = np.empty((int(n), int(N) // 2 + 3))
        ptr = x.ctypes.data if loc == BFB_HOST else int(x)
        check(self._L.bfb_chain_diagnostics(self._h, ptr, int(C_), int(T), int(t0), int(N), int(n), loc, P.ctypes.data))
        return P

    def last_kernel_ms(self):
        ms = C.c_float(0)
        check(self._L.bfb_last_kernel_ms(self._h, C.byref(ms)))
        return float(ms.value)

    def sampler_last_path(self):
        """kernel family of the last sampler run: 'generic', or a tensor-core family: 'dmma' (one warp per 8 chains), 'team', 'pair'"""
        return {0: 'generic', 2: 'dmma', 3: 'team', 4: 'pair'}.get(int(self._L.bfb_sampler_last_path(self._h)), 'none')

    def eval_last_path(self):
        """evaluator of the last logp_and_grad_batch: 'generic', 'dmma', 'lik_dmma' (tensor-core likelihood pipeline, one n x n
        product per output), 'lik_feat' (its feature form Phi(x) C^T) or 'team' (four warps per 8 points, 32 < n <= 64)"""
        return {0: 'generic', 2: 'dmma', 3: 'lik_dmma', 4: 'lik_feat', 5: 'team'}.get(int(self._L.bfb_eval_last_path(self._h)), 'none')

    def dmma_issue_test(self, nacc, src, warps_per_sm):
        v = C.c_double(0)
        check(self._L.bfb_dmma_issue_test(self._h, int(nacc), int(src), int(warps_per_sm), C.byref(v)))
        return float(v.value)

    def launch_count(self):
        return int(self._L.bfb_launch_count(self._h))

    def rng_fill(self, seed, chain, t0, count):
        u, z = np.empty(count), np.empty(count)
        check(self._L.bfb_rng_fill(self._h, int(seed), int(chain), int(t0), int(count), _d(u), _d(z)))
        return u, z

    def norminv_fill(self, p):
        p = np.ascontiguousarray(p, dtype=np.float64)
        z, z_ref = np.empty_like(p), np.empty_like(p)
        check(self._L.bfb_norminv_fill(self._h, _d(p), p.size, _d(z), _d(z_ref)))
        return z, z_ref

    def fp64_peak(self, kind=0):
        v = C.c_double(0)
        check(self._L.bfb_fp64_peak(self._h, int(kind), C.byref(v)))
        return float(v.value)
