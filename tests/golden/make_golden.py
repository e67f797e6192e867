"""
Generates tests/golden/*.npz by running the REAL reference (h3jia/bayesfast, /root/reference).

Run in the authoring container only (the reference does not exist on the GPU box):

    python tests/golden/make_golden.py

It copies /root/reference/bayesfast to a scratch directory, compiles its four Cython files there
(recipe of SURVEY.md section 8c), imports it through a small shim (numpy-2 aliases, stub matplotlib /
numdifftools) and records inputs + outputs of the hot path:

    poly_kat.npz      the reference's own tests/test_poly.py case (+ bound / far-point values)
    poly_eval.npz     PolyModel._fun_and_jac / fun_and_jac for injected coefficients (all orders, masks, bound)
    density.npz       Density.logp_and_grad(x, original_space=False) with decay + transform + module rescale
    fit.npz           PolyModel.fit (+ _set_bound) results
    sampler.npz       NUTS / HMC chains driven by a replayed random stream (include/bfb_rng.h draws)
    pipeline.npz      surrogate + Gaussian-likelihood module pipelines (2-D donut of examples/2d-donut.ipynb, multi-output)
    pipeline_ext.npz  the same with radial bound + module rescale + variable transform + decay + cubic-2 configs (pins the oracle)
    sampler_dense.npz the same with the dense mass matrix (metric='full' or a covariance; QuadMetricFull / FullAdapt)
    sampler_tempered.npz  TNUTS / THMC chains (samplers/tnuts.py, thmc.py) against a second, base density

The random stream: the reference's per-chain numpy Generator is replaced (after _init_chain) by a
duck-typed object that serves draw t of the Philox stream -- normal(size=k) consumes k draws through
Phi^-1, uniform() consumes one -- so the reference, the oracle and the CUDA kernels see the same numbers.
"""
import os
import shutil
import subprocess
import sys
import types
import warnings
from copy import deepcopy

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
SCRATCH = os.environ.get('BF_REF_SCRATCH', '/tmp/bf_ref')

BUILD_PY = '''
from setuptools import setup, Extension
from Cython.Build import cythonize
import numpy as np
names = ["bayesfast/modules/_poly", "bayesfast/transforms/_constraint", "bayesfast/utils/_cubic", "bayesfast/utils/_sobol"]
exts = [Extension(n.replace("/", "."), [n + ".pyx"], include_dirs=[np.get_include()],
                  extra_compile_args=["-fopenmp", "-O3"],
                  extra_link_args=["-B/usr/lib/gcc/x86_64-linux-gnu/13/", "-fopenmp"]) for n in names]
setup(name="bf_ref_ext", ext_modules=cythonize(exts, language_level="3"), script_args=["build_ext", "--inplace"])
'''


def import_reference():
    if not os.path.exists(os.path.join(SCRATCH, 'bayesfast')):
        os.makedirs(SCRATCH, exist_ok=True)
        shutil.copytree('/root/reference/bayesfast', os.path.join(SCRATCH, 'bayesfast'))
    import glob
    if not glob.glob(os.path.join(SCRATCH, 'bayesfast', 'modules', '_poly*.so')):
        with open(os.path.join(SCRATCH, 'build_ext.py'), 'w') as f:
            f.write(BUILD_PY)
        subprocess.check_call([sys.executable, 'build_ext.py'], cwd=SCRATCH, stdout=subprocess.DEVNULL)
    np.int = int
    np.float = float
    for name in ('matplotlib', 'matplotlib.pyplot', 'numdifftools'):
        sys.modules[name] = types.ModuleType(name)
    sys.modules['matplotlib'].pyplot = sys.modules['matplotlib.pyplot']
    for a in ('Gradient', 'Hessian', 'Jacobian', 'Hessdiag'):
        setattr(sys.modules['numdifftools'], a, None)
    sys.path.insert(0, SCRATCH)
    import bayesfast
    return bayesfast


bf = import_reference()
from bayesfast.modules.poly import PolyModel, PolyConfig  # noqa: E402
from bayesfast.samplers import NUTS, HMC, NTrace, HTrace  # noqa: E402
from bayesfast.samplers.hmc_utils.metrics import QuadMetricFull  # noqa: E402
from oracle import bf_oracle  # noqa: E402  (only for the Philox draws)
import _golden_io as gio  # noqa: E402


# ---------------------------------------------------------------------------------------------
def clean_coef(conf):
    """Dense _coef with the never-read entries (np.empty garbage, poly.py:146) zeroed."""
    c = np.array(conf._coef, copy=True)
    n = conf.input_size
    if conf.order == 'quadratic':
        c = np.triu(c)
    elif conf.order == 'cubic-3':
        mask = np.zeros((n, n, n), bool)
        for j in range(n):
            for k in range(j + 1, n):
                mask[j, k, k + 1:] = True
        c = np.where(mask, c, 0.)
    return c


def poly_spec(sur):
    spec = dict(n=sur._input_size, m=sur._output_size, configs=[])
    for conf in sur._configs:
        spec['configs'].append(dict(order=conf.order, input_mask=np.asarray(conf._input_mask, np.int64),
                                    output_mask=np.asarray(conf._output_mask, np.int64), coef=clean_coef(conf)))
    ub = bool(sur._use_bound and not sur._all_linear and hasattr(sur, '_mu'))
    spec['use_bound'] = ub
    if ub:
        spec.update(mu=sur._mu, hess=sur._hess, alpha=float(sur._alpha), f_mu=np.atleast_1d(sur._f_mu))
    spec['input_scales'] = None if sur._input_scales is None else np.array(sur._input_scales)
    return spec


def density_spec(den):
    sur = den._surrogate_list[0]
    spec = poly_spec(sur)
    spec['use_decay'] = bool(den._use_decay)
    if den._use_decay:
        spec.update(d_mu=den._mu, d_hess=den._hess, d_alpha2=float(den._alpha_2), d_gamma=float(den._gamma))
    if den._input_scales is None:
        spec['transform_ranges'] = None
    else:
        spec['transform_ranges'] = np.array(den._input_scales)
        hb = den._hard_bounds
        if isinstance(hb, bool):
            hb = hb * np.ones((spec['n'], 2), np.uint8)
        spec['hard_bounds'] = np.asarray(hb, np.uint8)
    return spec


def inject(sur, rng, scale=0.3):
    """Random independent coefficients through PolyConfig._set (poly.py:131-158)."""
    for conf in sur._configs:
        for i in range(conf.output_size):
            a = rng.normal(size=conf._a_shape) * scale
            if conf.order == 'quadratic':
                a *= 0.5
            elif conf.order in ('cubic-2', 'cubic-3'):
                a *= 0.1
            conf._set(a, i)


def set_bound_from(sur, pts):
    sur._set_bound(pts, None) if False else None
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        sur._set_bound(pts, np.arange(pts.shape[0], dtype=float))


# ---------------------------------------------------------------------------------------------
def make_poly_kat():
    bf.utils.random.set_generator(0)
    rng = bf.utils.random.get_generator()
    x = rng.normal(size=(50, 4))

    def poly_f(x):
        return (x[..., 0]**3 - 2 * x[..., 1]**3 + 3 * x[..., 1] * x[..., 2] * x[..., 3]
                - 4 * x[..., 2]**2 * x[..., 3] + 5 * x[..., 0]**2 - 6 * x[..., 0] * x[..., 2]
                + 7 * x[..., 1] - 8)[..., np.newaxis]

    y = poly_f(x)
    out = dict(x=x, y=y)
    for tag, logp in (('nologp', None), ('logp', y[:, 0])):
        s = PolyModel('cubic-3', input_size=4, output_size=1)
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            s.fit(x, y, logp)
        vals = np.concatenate([s(xi) for xi in x])
        far = 5 * x[0]
        ff, jf = s._fun_and_jac(far)
        out[tag] = dict(spec=poly_spec(s), values=vals, jac0=s.jac(x[0])[0], far=far, far_f=ff, far_j=jf)
    gio.save('poly_kat.npz', out)


def make_poly_eval():
    rng = np.random.default_rng(11)
    cases = []

    def add(name, sur, n, pts_scale=1., with_bound=True, input_scales=None):
        inject(sur, rng)
        train = rng.normal(size=(6 * n + 10, n)) * pts_scale
        if with_bound:
            set_bound_from(sur, train)
        else:
            sur._use_bound = False
        X = np.concatenate((rng.normal(size=(8, n)) * pts_scale * 0.7,
                            rng.normal(size=(4, n)) * pts_scale * 6.))
        raw_f, raw_j, wrp_f, wrp_j = [], [], [], []
        for xi in X:
            f, j = sur._fun_and_jac(xi)
            raw_f.append(f), raw_j.append(j)
            f, j = sur.fun_and_jac(xi)
            wrp_f.append(np.concatenate(f)), wrp_j.append(np.concatenate(j))
        cases.append(dict(name=name, spec=poly_spec(sur), X=X, raw_f=np.array(raw_f), raw_j=np.array(raw_j),
                          wrapped_f=np.array(wrp_f), wrapped_j=np.array(wrp_j)))

    add('quad_n2', PolyModel('quadratic', input_size=2, output_size=1), 2)
    add('c2_n16', PolyModel('cubic-2', input_size=16, output_size=1), 16)
    add('c2_n26', PolyModel('cubic-2', input_size=26, output_size=1), 26)
    add('c2_n26_nobound', PolyModel('cubic-2', input_size=26, output_size=1), 26, with_bound=False)
    add('c3_n8', PolyModel('cubic-3', input_size=8, output_size=1), 8)
    add('c3_n40', PolyModel('cubic-3', input_size=40, output_size=1), 40, pts_scale=0.5)
    add('linear_n5_m2', PolyModel('linear', input_size=5, output_size=2), 5)
    sc = np.stack((rng.normal(size=7) - 2., rng.normal(size=7) + 3.), axis=1)
    add('c2_n7_scaled', PolyModel('cubic-2', input_size=7, output_size=1, input_scales=sc), 7)
    cfgs = [PolyConfig('linear'),
            PolyConfig('quadratic', input_mask=[0, 2, 3], output_mask=[0, 2]),
            PolyConfig('cubic-2', input_mask=[1, 4, 5], output_mask=[1]),
            PolyConfig('cubic-3', input_mask=[0, 1, 2, 3, 4], output_mask=[2]),
            PolyConfig('cubic-2', input_mask=[0, 5], output_mask=[0, 2])]
    add('masked_n6_m3', PolyModel(cfgs, input_size=6, output_size=3), 6)
    gio.save('poly_eval.npz', dict(cases=cases))


def target_logp(P):
    def f(x):
        return np.atleast_1d(-0.5 * x @ P @ x - 0.02 * np.sum(x**3 * np.exp(-0.1 * x**2)))
    return f


def make_density(n, order, rng, transform=False, decay=False, module_scales=False, n_fit_mult=4, spread=1.):
    A = rng.normal(size=(n, n))
    cov = A @ A.T / n + np.eye(n)
    P = np.linalg.inv(cov)
    mod = bf.Module(fun=target_logp(P), input_vars='x', output_vars='logp')
    kw = {}
    if module_scales:
        kw['input_scales'] = np.stack((-2. + 0.1 * rng.normal(size=n), 3. + 0.1 * rng.normal(size=n)), axis=1)
    sur = PolyModel(order, input_size=n, output_size=1, input_vars='x', output_vars='logp', **kw)
    dkw = {}
    if transform:
        ranges = np.stack((-12. - rng.uniform(size=n), 12. + rng.uniform(size=n)), axis=1)
        hb = np.zeros((n, 2), np.uint8)
        hb[0] = (1, 1)
        if n > 2:
            hb[2] = (1, 0)
        if n > 3:
            hb[3] = (0, 1)
        dkw.update(input_scales=ranges, hard_bounds=hb)
    den = bf.Density(density_name='logp', module_list=[mod], surrogate_list=[sur], input_vars='x',
                     decay_options={'use_decay': decay}, **dkw)
    L = np.linalg.cholesky(cov)
    xf = (L @ rng.normal(size=(n, n_fit_mult * sur.n_param))).T * spread
    vd = [den.fun(x, original_space=True, use_surrogate=False) for x in xf]
    den.fit(vd)
    den.use_surrogate = True
    return den, cov, xf


def make_density_cases():
    rng = np.random.default_rng(23)
    cases = []
    for name, n, order, tr, dc, ms in (('c2_n4_all', 4, 'cubic-2', True, True, True),
                                       ('c2_n6_tr_decay', 6, 'cubic-2', True, True, False),
                                       ('quad_n3_plain', 3, 'quadratic', False, False, False),
                                       ('c3_n5_decay', 5, 'cubic-3', False, True, False),
                                       ('c2_n26_decay', 26, 'cubic-2', False, True, False)):
        den, cov, xf = make_density(n, order, rng, tr, dc, ms)
        L = np.linalg.cholesky(cov)
        Xo = np.concatenate(((L @ rng.normal(size=(n, 8))).T * 0.8, (L @ rng.normal(size=(n, 6))).T * 4.))
        if tr:
            Xo = np.clip(Xo, -11.5, 11.5)
        Xt = np.array([den.from_original(x) for x in Xo])
        lp, gr = [], []
        for x in Xt:
            a, b = den.logp_and_grad(x, original_space=False)
            lp.append(float(a)), gr.append(np.array(b))
        cases.append(dict(name=name, spec=density_spec(den), X=Xt, logp=np.array(lp), grad=np.array(gr)))
    gio.save('density.npz', dict(cases=cases))


def make_fit():
    rng = np.random.default_rng(5)
    cases = []

    def run(name, configs, n, m, N, w=None, scale=1., alpha_p=100., center_max=True):
        sur = PolyModel(configs, input_size=n, output_size=m,
                        bound_options=dict(alpha_p=alpha_p, center_max=center_max))
        x = rng.normal(size=(N, n)) * scale + 0.3
        tmp = PolyModel(deepcopy(configs), input_size=n, output_size=m)
        inject(tmp, rng, 1.)
        tmp._use_bound = False
        y = np.array([tmp._fun(xi) for xi in x]) + 1e-3 * rng.normal(size=(N, m))
        logp = y[:, 0].copy()
        sur.fit(x, y, logp, w)
        cases.append(dict(name=name, x=x, y=y, logp=logp, w=w, alpha_p=alpha_p, center_max=center_max,
                          spec=poly_spec(sur)))

    run('quad_n2', 'quadratic', 2, 1, 30)
    run('c2_n6_w', 'cubic-2', 6, 1, 300, w=rng.uniform(0.5, 1.5, size=300))
    run('c3_n5', 'cubic-3', 5, 1, 250, scale=0.7)
    run('c2_n8_m2_p90', 'cubic-2', 8, 2, 500, alpha_p=90., center_max=False)
    cfgs = [PolyConfig('linear'), PolyConfig('quadratic', input_mask=[0, 2, 3], output_mask=[0, 2]),
            PolyConfig('cubic-2', input_mask=[1, 4, 5], output_mask=[1])]
    run('masked_n6_m3', cfgs, 6, 3, 200)
    run('c2_n16', 'cubic-2', 16, 1, 4 * 409)
    gio.save('fit.npz', dict(cases=cases))


class Replay:
    """Duck-typed stand-in for numpy.random.Generator: serves the Philox draws of include/bfb_rng.h."""

    def __init__(self, u, z):
        self.u, self.z, self.t = u, z, 0

    def normal(self, *args, size=None):
        if len(args) == 1:                      # normal(size=k) of metrics.py:85; normal(0, 1) of base_hmc.py:245
            size = args[0]
        else:
            assert args in ((), (0, 1))
        k = 1 if size is None else int(size)
        v = self.z[self.t:self.t + k].copy()
        assert v.size == k, 'replay stream exhausted'
        self.t += k
        return v if size is not None else float(v[0])

    def uniform(self):
        v = self.u[self.t]
        self.t += 1
        return float(v)


def run_reference_chains(den, sampler, trace_kw, x0, seed, n_draw_cap):
    n_chain = x0.shape[0]
    cls, tcls = (NUTS, NTrace) if sampler == 'NUTS' else (HMC, HTrace)
    base = tcls(n_chain=n_chain, x_0=x0, random_generator=0, **trace_kw)
    res = dict(samples=[], final_step=[], final_var=[], n_draws=[], draws_u=[], draws_z=[])
    names = ('logp', 'energy', 'tree_depth', 'tree_size', 'mean_tree_accept', 'step_size', 'step_size_bar',
             'energy_change', 'max_energy_change', 'diverging') if sampler == 'NUTS' else \
            ('logp', 'energy', 'n_int_step', 'accept_stat', 'accepted', 'step_size', 'step_size_bar',
             'energy_change', 'diverging')
    for k in names:
        res[k] = []
    step0 = var0 = None
    for i in range(n_chain):
        t = deepcopy(base)
        t._init_chain(i)
        u, z = bf_oracle.rng_fill(seed, i, 0, n_draw_cap)
        rep = Replay(u, z)
        t._random_generator = rep
        if i == 0:
            step0 = float(np.exp(t.step_size._log_step))
            var0 = np.array(t.metric._cov if hasattr(t.metric, '_cov') else t.metric._var)
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            cls(logp_and_grad=lambda x: den.logp_and_grad(x, original_space=False), sample_trace=t).run(verbose=False)
        res['samples'].append(np.array(t._samples))
        for k in names:
            res[k].append(np.array(getattr(t.stats, '_' + k), dtype=float))
        ss = t.step_size
        res['final_step'].append([ss._log_step, ss._log_bar, ss._hbar, ss._count])
        res['final_var'].append(np.array(t.metric._cov if hasattr(t.metric, '_cov') else t.metric._var))
        res['n_draws'].append(rep.t)
        res['draws_u'].append(u), res['draws_z'].append(z)
    nmax = max(res['n_draws']) + 4
    out = {k: np.array(v) for k, v in res.items()}
    out['draws_u'] = out['draws_u'][:, :nmax]
    out['draws_z'] = out['draws_z'][:, :nmax]
    out['step0'] = step0
    out['var0'] = var0
    return out


def run_reference_tempered(den, den_base, logxi, sampler, trace_kw, x0, u0, seed, n_draw_cap=60000):
    """TNUTS / THMC of the real reference, driven directly (core/sample.py:64-70 tests isinstance(trace, NTrace) first, so
    bf.sample() would run plain NUTS on a TNTrace).  The tempering variable of the first iteration comes from numpy's GLOBAL
    generator in the reference (base_hmc.py:242): served from u0 here.  THTrace.__init__ raises in the reference
    (sample_trace.py:600 calls HTrace.__init__ without self, and never installs THStats), so for THMC the trace object is
    assembled from the two base initialisers by hand -- the sampler code that then runs is the unmodified reference."""
    from bayesfast.samplers import TNUTS, THMC, TNTrace
    from bayesfast.samplers.sample_trace import THTrace, _TTrace
    from bayesfast.samplers.hmc_utils.stats import THStats
    n_chain = x0.shape[0]
    if sampler == 'TNUTS':
        cls = TNUTS
        base = TNTrace(den_base, logxi, n_chain=n_chain, x_0=x0, random_generator=0, **trace_kw)
        names = ('u', 'weight', 'logp', 'energy', 'tree_depth', 'tree_size', 'mean_tree_accept', 'step_size', 'step_size_bar',
                 'energy_change', 'max_energy_change', 'diverging')
    else:
        cls = THMC
        base = THTrace.__new__(THTrace)
        _TTrace.__init__(base, den_base, logxi)
        HTrace.__init__(base, n_chain=n_chain, x_0=x0, random_generator=0, **trace_kw)
        base._stats = THStats()
        names = ('u', 'weight', 'logp', 'energy', 'n_int_step', 'accept_stat', 'accepted', 'step_size', 'step_size_bar',
                 'energy_change', 'diverging')
    res = dict(samples=[], final_step=[], final_var=[], n_draws=[], draws_u=[], draws_z=[])
    for k in names:
        res[k] = []
    step0 = var0 = None
    for i in range(n_chain):
        t = deepcopy(base)
        t._init_chain(i)
        u, z = bf_oracle.rng_fill(seed, i, 0, n_draw_cap)
        rep = Replay(u, z)
        t._random_generator = rep
        if i == 0:
            step0 = float(np.exp(t.step_size._log_step))
            var0 = np.array(t.metric._var)
        keep = np.random.normal
        np.random.normal = lambda *a, **k: float(u0[i])
        try:
            with warnings.catch_warnings():
                warnings.simplefilter('ignore')
                cls(logp_and_grad=lambda x: den.logp_and_grad(x, original_space=False), sample_trace=t).run(verbose=False)
        finally:
            np.random.normal = keep
        res['samples'].append(np.array(t._samples))
        for k in names:
            res[k].append(np.array(getattr(t.stats, '_' + k), dtype=float))
        ss = t.step_size
        res['final_step'].append([ss._log_step, ss._log_bar, ss._hbar, ss._count])
        res['final_var'].append(np.array(t.metric._var))
        res['n_draws'].append(rep.t)
        res['draws_u'].append(u), res['draws_z'].append(z)
    nmax = max(res['n_draws']) + 4
    out = {k: np.array(v) for k, v in res.items()}
    out['draws_u'] = out['draws_u'][:, :nmax]
    out['draws_z'] = out['draws_z'][:, :nmax]
    out['step0'] = step0
    out['var0'] = var0
    return out


def make_tempered_pair(n, order, rng, transform=False, decay=False, temperature=3.):
    """target: `order` surrogate of the usual test density; base: quadratic surrogate of the same density at a higher
    temperature (a broad Gaussian), same variable transform."""
    A = rng.normal(size=(n, n))
    cov = A @ A.T / n + np.eye(n)
    P = np.linalg.inv(cov)
    dkw = {}
    if transform:
        ranges = np.stack((-12. - rng.uniform(size=n), 12. + rng.uniform(size=n)), axis=1)
        hb = np.zeros((n, 2), np.uint8)
        hb[0] = (1, 1)
        if n > 2:
            hb[2] = (1, 0)
        dkw.update(input_scales=ranges, hard_bounds=hb)
    L = np.linalg.cholesky(cov)
    dens = []
    for o, fun, dc, spread in ((order, target_logp(P), decay, 1.), ('quadratic', target_logp(P / temperature), False, 1.5)):
        mod = bf.Module(fun=fun, input_vars='x', output_vars='logp')
        sur = PolyModel(o, input_size=n, output_size=1, input_vars='x', output_vars='logp')
        den = bf.Density(density_name='logp', module_list=[mod], surrogate_list=[sur], input_vars='x',
                         decay_options={'use_decay': dc}, **dkw)
        xf = (L @ rng.normal(size=(n, 4 * sur.n_param))).T * spread
        if transform:
            xf = np.clip(xf, -11., 11.)
        den.fit([den.fun(x, original_space=True, use_surrogate=False) for x in xf])
        den.use_surrogate = True
        dens.append(den)
    return dens[0], dens[1], xf


def make_sampler_tempered():
    rng = np.random.default_rng(4242)
    cases = []

    def add(name, sampler, den, db, logxi, x0, u0, seed, **trace_kw):
        r = run_reference_tempered(den, db, logxi, sampler, trace_kw, x0, u0, seed)
        cases.append(dict(name=name, sampler=sampler, spec=density_spec(den), base_spec=density_spec(db), logxi=logxi,
                          x0=x0, u0=np.asarray(u0, dtype=float), seed=seed,
                          trace_kw={k: (v if not isinstance(v, bool) else int(v)) for k, v in trace_kw.items()}, result=r))
        print(name, 'mean depth', np.mean(r['tree_depth']) if sampler == 'TNUTS' else '-', 'n_div', int(np.sum(r['diverging'])),
              'draws', r['n_draws'], 'u range', float(np.min(r['u'])), float(np.max(r['u'])),
              'weight range', float(np.min(r['weight'])), float(np.max(r['weight'])))

    den, db, xf = make_tempered_pair(3, 'quadratic', rng)
    add('tnuts_quad_n3', 'TNUTS', den, db, 0., xf[:2].copy() / 1.5, [0.3, -1.2], 11, n_iter=50, n_warmup=25)
    add('thmc_quad_n3', 'THMC', den, db, 0.1, xf[:2].copy() / 1.5, [-0.4, 0.9], 44, n_iter=40, n_warmup=20, n_int_step=6)
    den, db, xf = make_tempered_pair(6, 'cubic-2', rng, transform=True, decay=True)
    x0 = np.array([den.from_original(x / 1.5) for x in xf[:3]])
    add('tnuts_c2_n6_tr_decay', 'TNUTS', den, db, 0.4, x0, [0.5, 2.0, -0.7], 22, n_iter=40, n_warmup=20)
    add('tnuts_c2_n6_depthcap', 'TNUTS', den, db, -0.2, x0[:2], [0., 1.], 33, n_iter=24, n_warmup=8, max_treedepth=3)
    den, db, xf = make_tempered_pair(16, 'cubic-2', rng)
    add('tnuts_c2_n16', 'TNUTS', den, db, 0., xf[:2].copy() / 1.5, [1.1, -0.3], 55, n_iter=30, n_warmup=15)
    gio.save('sampler_tempered.npz', dict(cases=cases))


def make_sampler():
    rng = np.random.default_rng(77)
    cases = []

    def add(name, sampler, den, x0, seed, n_draw_cap=60000, **trace_kw):
        r = run_reference_chains(den, sampler, trace_kw, x0, seed, n_draw_cap)
        cases.append(dict(name=name, sampler=sampler, spec=density_spec(den), x0=x0, seed=seed,
                          trace_kw={k: (v if not isinstance(v, bool) else int(v)) for k, v in trace_kw.items()},
                          result=r))
        print(name, 'mean depth', np.mean(r['tree_depth']) if sampler == 'NUTS' else '-',
              'n_div', int(np.sum(r['diverging'])), 'draws', r['n_draws'])

    den, cov, xf = make_density(2, 'quadratic', rng)
    add('nuts_quad_n2', 'NUTS', den, xf[:4].copy(), 101, n_iter=80, n_warmup=40)

    den, cov, xf = make_density(6, 'cubic-2', rng, transform=True, decay=True)
    x0 = np.array([den.from_original(np.clip(x, -11., 11.)) for x in xf[:3]])
    add('nuts_c2_n6_tr_decay', 'NUTS', den, x0, 202, n_iter=50, n_warmup=25)
    L = np.linalg.cholesky(cov)
    far = np.array([den.from_original(np.clip((L @ rng.normal(size=6)) * 3.5, -11., 11.)) for _ in range(2)])
    add('nuts_c2_n6_far_start', 'NUTS', den, far, 303, n_iter=30, n_warmup=15)
    add('nuts_c2_n6_depthcap', 'NUTS', den, x0[:2], 404, n_iter=30, n_warmup=10, max_treedepth=2)
    add('nuts_c2_n6_divergent', 'NUTS', den, x0[:2], 505, n_iter=30, n_warmup=10, max_change=3.0,
        step_size=1.1, adapt_step_size=False)
    add('nuts_c2_n6_noadapt', 'NUTS', den, x0[:2], 606, n_iter=25, n_warmup=10, adapt_step_size=False,
        adapt_metric=False, step_size=0.6)
    add('hmc_c2_n6', 'HMC', den, x0[:2], 707, n_iter=30, n_warmup=15, n_int_step=8)

    den, cov, xf = make_density(16, 'cubic-2', rng)
    add('nuts_c2_n16', 'NUTS', den, xf[:2].copy(), 808, n_iter=40, n_warmup=20)

    den, cov, xf = make_density(5, 'cubic-3', rng, decay=True)
    add('nuts_c3_n5', 'NUTS', den, xf[:2].copy(), 909, n_iter=40, n_warmup=20)
    gio.save('sampler.npz', dict(cases=cases))


def make_sampler_dense():
    """dense mass matrix (metric='full': QuadMetricFull / QuadMetricFullAdapt, metrics.py:94-132, 240-330)"""
    rng = np.random.default_rng(78)
    cases = []

    def add(name, sampler, den, x0, seed, n_draw_cap=60000, **trace_kw):
        r = run_reference_chains(den, sampler, trace_kw, x0, seed, n_draw_cap)
        kw = {k: (int(v) if isinstance(v, bool) else v) for k, v in trace_kw.items() if k != 'metric'}
        if isinstance(trace_kw['metric'], QuadMetricFull):       # a fixed covariance (a QuadMetric instance is used as is)
            kw['adapt_metric'] = 0
        cases.append(dict(name=name, sampler=sampler, spec=density_spec(den), x0=x0, seed=seed, trace_kw=kw, result=r))
        print(name, 'mean depth', np.mean(r['tree_depth']) if sampler == 'NUTS' else '-',
              'n_div', int(np.sum(r['diverging'])), 'draws', r['n_draws'])

    den, cov, xf = make_density(6, 'cubic-2', rng, transform=True, decay=True)
    x0 = np.array([den.from_original(np.clip(x, -11., 11.)) for x in xf[:3]])
    add('nuts_c2_n6_full_adapt', 'NUTS', den, x0, 1101, n_iter=60, n_warmup=30, metric='full')
    add('hmc_c2_n6_full_adapt', 'HMC', den, x0[:2], 1202, n_iter=30, n_warmup=15, n_int_step=8, metric='full')
    den, cov, xf = make_density(16, 'cubic-2', rng)
    add('nuts_c2_n16_full_fixed', 'NUTS', den, xf[:2].copy(), 1303, n_iter=30, n_warmup=15, metric=QuadMetricFull(0.7 * cov + 0.3 * np.eye(16)))
    add('nuts_c2_n16_full_adapt', 'NUTS', den, xf[:2].copy(), 1404, n_iter=40, n_warmup=30, metric='full', adapt_window=12)
    gio.save('sampler_dense.npz', dict(cases=cases))


def make_pipeline():
    """Two-module pipelines: PolyModel surrogate (x -> m outputs) followed by a Gaussian-likelihood module
    logp = c - 1/2 (f - d)^T Cinv (f - d) written as a user bf.Module (fun + jac), as in examples/2d-donut.ipynb (m = 1,
    d = 5, Cinv = 4: f_1 = -(m - 5)^2 / 0.5) and, multi-output with masked configs, like the DES-Y1 example.  Records
    Density.logp_and_grad of the real reference and NUTS runs driven by the replayed stream."""
    rng = np.random.default_rng(91)
    cases = []

    def lik_module(d, cinv, c0):
        cs = 0.5 * (cinv + cinv.T)
        return bf.Module(fun=lambda f: np.atleast_1d(c0 - 0.5 * (f - d) @ cinv @ (f - d)),
                         jac=lambda f: np.atleast_2d(-(cs @ (f - d))), input_vars='m', output_vars='logp')

    def finish(name, den, ep, Xt, x0, seed, **trace_kw):        # appends to the `cases` list current at call time
        lp, gr = [], []
        for x in Xt:
            a_, b_ = den.logp_and_grad(x, original_space=False)
            lp.append(float(a_)), gr.append(np.array(b_))
        r = run_reference_chains(den, 'NUTS', trace_kw, x0, seed, 60000)
        spec = density_spec(den)
        spec['epilogue'] = ep
        cases.append(dict(name=name, spec=spec, X=Xt, logp=np.array(lp), grad=np.array(gr), x0=x0, seed=seed,
                          trace_kw=trace_kw, result=r))
        print(name, 'mean depth', np.mean(r['tree_depth']), 'n_div', int(np.sum(r['diverging'])), 'draws', r['n_draws'])

    # --- BASELINE configs[0]: 2-D donut, quadratic surrogate of m = |x|, analytic f_1, decay on, bound off, 4 chains ---
    a, b = 5., 0.5
    m0 = bf.Module(fun=lambda x: np.atleast_1d(np.linalg.norm(x, 2, -1)), input_vars='x', output_vars='m')
    m1 = bf.Module(fun=lambda x: -(x - a)**2 / b, jac=lambda x: np.atleast_2d(-2 * (x - a) / b), input_vars='m',
                   output_vars='logp')
    sur = PolyModel('quadratic', input_size=2, output_size=1, input_vars='x', output_vars='m')
    sur.set_bound_options(use_bound=False)
    den = bf.Density(module_list=[m0, m1], surrogate_list=[sur], input_shapes=[2], input_vars='x', density_name='logp')
    den.set_decay_options(use_decay=True)
    th = rng.uniform(0., 2. * np.pi, size=30)                 # 5 P = 30 fit points on the ring (recipe.py:84-86)
    rad = 5. + 0.5 * rng.normal(size=30)
    xf = np.stack((rad * np.cos(th), rad * np.sin(th)), axis=1)
    den.fit([den.fun(x, original_space=True, use_surrogate=False) for x in xf])
    den.use_surrogate = True
    Xt = np.concatenate((xf[:6] * 1.02, rng.normal(size=(4, 2)) * 2., xf[6:9] * 2.5))
    finish('donut_quadratic', den, dict(d=np.array([a]), cinv=np.array([[2. / b]]), c0=0.), Xt, xf[10:14].copy(), 2101,
           n_iter=40, n_warmup=20)       # short: the ring amplifies rounding differences ~1.3x per iteration

    # --- multi-output: n = 5 inputs, m = 6 outputs from two masked quadratic configs + a linear one, full Cinv ---
    n, m = 5, 6
    cfgs = [PolyConfig('linear', input_mask=None, output_mask=None),
            PolyConfig('quadratic', input_mask=[0, 1, 3], output_mask=[0, 1, 2]),
            PolyConfig('quadratic', input_mask=[1, 2, 3, 4], output_mask=[3, 4, 5])]
    W = rng.normal(size=(m, n)) * 0.6
    truth = lambda x: W @ x + 0.15 * np.array([x[0] * x[1], x[3]**2, x[0] * x[3], x[2] * x[4], x[1]**2, x[3] * x[4]])
    d = rng.normal(size=m) * 0.3
    B = rng.normal(size=(m, m))
    cinv = B @ B.T / m + 0.5 * np.eye(m)
    mA = bf.Module(fun=truth, input_vars='x', output_vars='m')
    sur = PolyModel(cfgs, input_size=n, output_size=m, input_vars='x', output_vars='m')
    den = bf.Density(module_list=[mA, lik_module(d, cinv, -1.25)], surrogate_list=[sur], input_shapes=[n], input_vars='x',
                     density_name='logp', decay_options={'use_decay': True})
    xf = rng.normal(size=(4 * sur.n_param, n)) * 1.5
    den.fit([den.fun(x, original_space=True, use_surrogate=False) for x in xf])
    den.use_surrogate = True
    Xt = np.concatenate((xf[:8] * 0.7, xf[8:14] * 3.))
    finish('multi_output_n5_m6', den, dict(d=d, cinv=cinv, c0=-1.25), Xt, xf[20:23] * 0.5, 2202, n_iter=60, n_warmup=30)
    gio.save('pipeline.npz', dict(cases=cases))

    # --- second file (oracle pin only): multi-output pipeline with everything on -- radial bound (default bound options, so
    # far points take PolyModel._fj_bound for every output), module-level input_scales, variable transform with hard bounds,
    # decay, cubic-2 + quadratic + linear configs ---
    cases = []
    n, m = 4, 3
    cfgs = [PolyConfig('linear'), PolyConfig('quadratic', input_mask=[0, 1, 2], output_mask=[0, 2]), PolyConfig('cubic-2', output_mask=[1])]
    W = rng.normal(size=(m, n)) * 0.5
    truth = lambda x: W @ x + 0.1 * np.array([x[0] * x[1], x[2]**2 * x[3], x[1] * x[2]])
    d = rng.normal(size=m) * 0.2
    B = rng.normal(size=(m, m))
    cinv = B @ B.T / m + 0.4 * np.eye(m)
    ranges = np.stack((-9. - rng.uniform(size=n), 9. + rng.uniform(size=n)), axis=1)
    hb = np.array([[1, 1], [0, 0], [1, 0], [0, 1]], np.uint8)
    mA = bf.Module(fun=truth, input_vars='x', output_vars='m')
    sur = PolyModel(cfgs, input_size=n, output_size=m, input_vars='x', output_vars='m',
                    input_scales=np.stack((-1.5 + 0.1 * rng.normal(size=n), 2. + 0.1 * rng.normal(size=n)), axis=1))
    den = bf.Density(module_list=[mA, lik_module(d, cinv, 0.3)], surrogate_list=[sur], input_shapes=[n], input_vars='x',
                     density_name='logp', decay_options={'use_decay': True}, input_scales=ranges, hard_bounds=hb)
    xf = rng.normal(size=(4 * sur.n_param, n)) * 1.2
    den.fit([den.fun(x, original_space=True, use_surrogate=False) for x in xf])
    den.use_surrogate = True
    Xo = np.clip(np.concatenate((xf[:8] * 0.8, xf[8:16] * 4.)), -8.5, 8.5)
    Xt = np.array([den.from_original(x) for x in Xo])
    x0 = np.array([den.from_original(x) for x in xf[30:33] * 0.5])
    finish('multi_output_bound_transform_decay', den, dict(d=d, cinv=cinv, c0=0.3), Xt, x0, 2303, n_iter=40, n_warmup=20)
    for c in cases:          # trees 8 doublings deep use 1.5 MB of draws: kept as a digest, the test regenerates them
        r = c['result']
        r['draws_sha256'] = gio.draws_digest(r.pop('draws_u'), r.pop('draws_z'))
    gio.save('pipeline_ext.npz', dict(cases=cases))


def make_sampler_d26():
    """The headline shape pinned directly: d = 26 cubic-2 surrogate with the radial bound, 4 chains x 60 iterations, and the
    same with the logit transform on 5 coordinates (SURVEY 8d config 3)."""
    rng = np.random.default_rng(2626)
    cases = []

    def add(name, den, x0, seed, **trace_kw):
        r = run_reference_chains(den, 'NUTS', trace_kw, x0, seed, 60000)
        cases.append(dict(name=name, sampler='NUTS', spec=density_spec(den), x0=x0, seed=seed,
                          trace_kw={k: (v if not isinstance(v, bool) else int(v)) for k, v in trace_kw.items()}, result=r))
        print(name, 'mean depth', np.mean(r['tree_depth']), 'n_div', int(np.sum(r['diverging'])), 'draws', r['n_draws'])

    den, cov, xf = make_density(26, 'cubic-2', rng)
    assert den._surrogate_list[0]._use_bound
    add('nuts_c2_n26_bound', den, xf[:4].copy(), 2601, n_iter=60, n_warmup=30)
    # hard bounds (logit transform) on 5 coordinates, soft ranges elsewhere, like cell 16 of the DES notebook
    n = 26
    A = rng.normal(size=(n, n))
    cov = A @ A.T / n + np.eye(n)
    P = np.linalg.inv(cov)
    mod = bf.Module(fun=target_logp(P), input_vars='x', output_vars='logp')
    sur = PolyModel('cubic-2', input_size=n, output_size=1, input_vars='x', output_vars='logp')
    ranges = np.stack((-9. - rng.uniform(size=n), 9. + rng.uniform(size=n)), axis=1)
    hb = np.zeros((n, 2), np.uint8)
    for j in (0, 4, 6, 16, 17):
        hb[j] = (1, 1)
    den = bf.Density(density_name='logp', module_list=[mod], surrogate_list=[sur], input_vars='x',
                     decay_options={'use_decay': False}, input_scales=ranges, hard_bounds=hb)
    L = np.linalg.cholesky(cov)
    xf = np.clip((L @ rng.normal(size=(n, 4 * sur.n_param))).T, -8.5, 8.5)
    den.fit([den.fun(x, original_space=True, use_surrogate=False) for x in xf])
    den.use_surrogate = True
    x0 = np.array([den.from_original(x) for x in xf[:4]])
    add('nuts_c2_n26_bound_transform5', den, x0, 2602, n_iter=60, n_warmup=30)
    gio.save('sampler_d26.npz', dict(cases=cases))


def seeded_coefs(n, orders, seed, scales):
    """packed coefficient vectors from a seed: the test regenerates them instead of storing 2 MB of cubic-3 coefficients"""
    rng = np.random.default_rng(seed)
    shapes = {'linear': n + 1, 'quadratic': n * (n + 1) // 2, 'cubic-2': n * n, 'cubic-3': n * (n - 1) * (n - 2) // 6}
    return [rng.normal(size=shapes[o]) * scales[o] for o in orders]


def make_poly_eval_c3n64():
    """BASELINE configs[3]: 64-D cubic-3 stack (P = 47905) with injected coefficients and the radial bound"""
    n = 64
    orders = ('linear', 'quadratic', 'cubic-2', 'cubic-3')
    scales = {'linear': 0.3, 'quadratic': 0.15 / np.sqrt(n), 'cubic-2': 0.03 / n, 'cubic-3': 0.03 / n}
    sur = PolyModel('cubic-3', input_size=n, output_size=1)
    for conf, a in zip(sur._configs, seeded_coefs(n, orders, 6464, scales)):
        assert conf.order == orders[sur._configs.index(conf)]
        conf._set(a.reshape(conf._a_shape) if hasattr(conf, '_a_shape') else a, 0)
    rng = np.random.default_rng(65)
    train = rng.normal(size=(6 * n + 10, n)) * 0.5
    set_bound_from(sur, train)
    X = np.concatenate((rng.normal(size=(8, n)) * 0.35, rng.normal(size=(4, n)) * 3.))
    raw_f, raw_j = [], []
    for xi in X:
        f, j = sur._fun_and_jac(xi)
        raw_f.append(f), raw_j.append(j)
    gio.save('poly_eval_c3n64.npz', dict(n=n, seed=6464, scales=scales, X=X, raw_f=np.array(raw_f), raw_j=np.array(raw_j),
                                         mu=sur._mu, hess=sur._hess, alpha=float(sur._alpha), f_mu=np.atleast_1d(sur._f_mu)))
    print('c3_n64 beta/alpha of the points', [float(np.sqrt((x - sur._mu) @ sur._hess @ (x - sur._mu)) / sur._alpha) for x in X])


def make_pipeline_des():
    """The DES-Y1 example's density shape (examples/des-y1-w-cosmosis.ipynb cells 12-18): three modules -- surrogate
    x (27) -> m outputs from a linear config plus a quadratic config on the SHARED mask `nonlinear_indices`, module
    input_scales = para_range; chi2 module like = -1/2 |m - d|^2 + norm; posterior module logp = like + Gaussian prior on 13 of
    the x -- in a Density with input_scales = para_range and hard_bounds = True (logit transform on every coordinate), radial
    bound on (default bound options).  m = 40 here to keep the fixture small."""
    rng = np.random.default_rng(1812)
    n, m = 27, 40
    para_range = np.array([[0.1, 0.9], [0.55, 0.9], [0.03, 0.07], [0.87, 1.07], [0.5e-9, 5.0e-9], [0.0006, 0.01], [-2, -0.333],
                           [0.8, 3.0], [0.8, 3.0], [0.8, 3.0], [0.8, 3.0], [0.8, 3.0], [-0.1, 0.1], [-0.1, 0.1], [-0.1, 0.1],
                           [-0.1, 0.1], [-5.0, 5.0], [-5.0, 5.0], [-0.1, 0.1], [-0.1, 0.1], [-0.1, 0.1], [-0.1, 0.1],
                           [-0.05, 0.05], [-0.05, 0.05], [-0.05, 0.05], [-0.05, 0.05], [-0.05, 0.05]])
    nonlinear_indices = np.array([0, 1, 2, 3, 4, 5, 6, 16, 17])
    prior_idx = np.array([18, 19, 20, 21, 12, 13, 14, 15, 22, 23, 24, 25, 26])
    prior_mu = np.array([-0.001, -0.019, 0.009, -0.018, 0.012, 0.012, 0.012, 0.012, 0.008, -0.005, 0.006, 0.0, 0.0])
    prior_sig = np.array([0.016, 0.013, 0.011, 0.022, 0.023, 0.023, 0.023, 0.023, 0.007, 0.007, 0.006, 0.01, 0.01]) * 3.
    prior_c0 = -1.75
    width = para_range[:, 1] - para_range[:, 0]
    mid = para_range.mean(axis=1)
    W1 = rng.normal(size=(m, n)) * 1.5
    W2 = rng.normal(size=(m, 9, 9)) * 0.8

    def theory(x):
        u = (x - mid) / width
        v = u[nonlinear_indices]
        return W1 @ u + np.einsum('ojk,j,k->o', W2, v, v) + 0.05 * np.sin(3. * (W1 @ u))

    u_true = rng.normal(size=n) * 0.05
    d_vec = theory(mid + u_true * width) + 0.05 * rng.normal(size=m)
    norm_c = 3.25

    def prior_f(x):
        return -0.5 * np.sum(((x[prior_idx] - prior_mu) / prior_sig)**2) + prior_c0

    def prior_j(x):
        foo = np.zeros((1, n))
        foo[0, prior_idx] = -(x[prior_idx] - prior_mu) / prior_sig**2
        return foo

    module_0 = bf.Module(fun=theory, input_vars='x', output_vars='m')
    module_1 = bf.Module(fun=lambda mm: np.atleast_1d(-0.5 * np.sum((mm - d_vec)**2) + norm_c),
                         fun_and_jac=lambda mm: (np.atleast_1d(-0.5 * np.sum((mm - d_vec)**2) + norm_c), -(mm - d_vec)[np.newaxis]),
                         input_vars='m', output_vars='like')
    module_2 = bf.Module(fun=lambda like, x: like + prior_f(x),
                         fun_and_jac=lambda like, x: (like + prior_f(x), np.concatenate((np.ones((1, 1)), prior_j(x)), axis=-1)),
                         input_vars=['like', 'x'], output_vars='logp')
    den = bf.Density(density_name='logp', module_list=[module_0, module_1, module_2], input_vars='x', input_shapes=n,
                     input_scales=para_range, hard_bounds=True)
    sur = PolyModel([PolyConfig('linear'), PolyConfig('quadratic', input_mask=nonlinear_indices)], input_size=n, output_size=m,
                    input_vars='x', output_vars='m', input_scales=para_range)
    den.surrogate_list = [sur]
    xf = mid + np.clip(rng.normal(size=(3 * sur.n_param, n)) * 0.08, -0.45, 0.45) * width
    den.fit([den.fun(x, original_space=True, use_surrogate=False) for x in xf])
    den.use_surrogate = True
    assert sur._use_bound
    Xo = np.concatenate((xf[:8], mid + np.clip(rng.normal(size=(6, n)) * 0.3, -0.47, 0.47) * width))
    Xt = np.array([den.from_original(x) for x in Xo])
    lp, gr = [], []
    for x in Xt:
        a_, b_ = den.logp_and_grad(x, original_space=False)
        lp.append(float(a_)), gr.append(np.array(b_))
    x0 = np.array([den.from_original(x) for x in xf[20:24]])
    r = run_reference_chains(den, 'NUTS', dict(n_iter=40, n_warmup=20), x0, 2404, 60000)
    spec = density_spec(den)
    spec['epilogue'] = dict(d=d_vec, cinv=np.eye(m), c0=norm_c)
    spec['prior'] = dict(idx=prior_idx, mu=prior_mu, sig=prior_sig, c0=prior_c0)
    print('des_shaped mean depth', np.mean(r['tree_depth']), 'n_div', int(np.sum(r['diverging'])), 'draws', r['n_draws'],
          'outside', [float(np.sqrt(((x - mid) / width * 0 + 1) @ np.ones(n))) for x in Xo[:1]])
    gio.save('pipeline_des.npz', dict(cases=[dict(name='des_shaped_n27_m40', spec=spec, X=Xt, logp=np.array(lp), grad=np.array(gr),
                                                  x0=x0, seed=2404, trace_kw=dict(n_iter=40, n_warmup=20), result=r)]))


def make_post():
    """SystematicResampler.run of the real reference (utils/misc.py:21-110) on seeded arrays, and PostStep's weight lines"""
    from bayesfast.utils.misc import SystematicResampler
    rng = np.random.default_rng(404)
    cases = []
    for name, m, n, nodes, weights in (('default', 5000, 400, (1., 100.), None), ('three_nodes', 20000, 1500, (0., 50., 100.), (1., 3.)),
                                       ('small', 97, 31, (1., 100.), None), ('ragged', 30011, 4216, (1., 99.5, 100.), (40., 1.))):
        a = rng.normal(size=m) * 3. - 10.
        i = SystematicResampler(nodes=nodes, weights=weights).run(a, n)
        cases.append(dict(name=name, a=a, n=n, nodes=np.asarray(nodes), weights=weights, idx=np.asarray(i, np.int64)))
    logp, logq = rng.normal(size=2000) - 5., rng.normal(size=2000) * 0.9 - 5.
    weights = np.exp(logp - logq)
    wt = np.clip(weights, 0, np.mean(weights) * 2000**0.25)                 # recipe.py:1291-1297 with n_is = 2000, k_trunc = 0.25
    gio.save('post.npz', dict(cases=cases, logp=logp, logq=logq, k_trunc=0.25, weights=weights, weights_trunc=wt))


def make_sobol_x0():
    """default x_0 of bayesfast.sample (core/sample.py:107-112): utils.sobol.multivariate_normal of the real reference"""
    from bayesfast.utils.sobol import multivariate_normal
    out = {}
    for d, n in ((2, 4), (26, 37), (64, 50)):
        out['d%d_n%d' % (d, n)] = multivariate_normal(np.zeros(d), np.eye(d), n)
    np.savez_compressed(os.path.join(gio.GOLDEN_DIR, 'sobol_x0.npz'), **out)


if __name__ == '__main__':
    which = sys.argv[1:] or ['poly_kat', 'poly_eval', 'density', 'fit', 'sampler', 'sampler_dense', 'pipeline']
    if 'poly_kat' in which:
        make_poly_kat()
    if 'poly_eval' in which:
        make_poly_eval()
    if 'density' in which:
        make_density_cases()
    if 'fit' in which:
        make_fit()
    if 'sampler' in which:
        make_sampler()
    if 'sampler_tempered' in which:
        make_sampler_tempered()
    if 'sampler_d26' in which:
        make_sampler_d26()
    if 'poly_eval_c3n64' in which:
        make_poly_eval_c3n64()
    if 'pipeline_des' in which:
        make_pipeline_des()
    if 'post' in which:
        make_post()
    if 'sobol_x0' in which:
        make_sobol_x0()
    if 'sampler_dense' in which:
        make_sampler_dense()
    if 'pipeline' in which:
        make_pipeline()
    for f in sorted(os.listdir(gio.GOLDEN_DIR)):
        if f.endswith('.npz'):
            print(f, os.path.getsize(os.path.join(gio.GOLDEN_DIR, f)))
