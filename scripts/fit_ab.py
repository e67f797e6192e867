"""Fit outputs of two builds of libbfb200.so on the same seeded inputs, compared bit for bit.

    python scripts/fit_ab.py --lib-a OLD.so --lib-b NEW.so --out-dir fit_ab

Each build runs in a process of its own (BFB200_LIB) and fits: the cases of tests/golden/fit.npz, the shapes of
test_gpu_fit.py::test_fit_vs_lstsq, a Density with the decay ellipsoid, and cubic-2 at n = 53 / 54 / 60 and quadratic at n = 64
(P = 4294 / 4510 / 5491 / 2145).  Per case it stores every coefficient block, _mu, _hess, _alpha, _f_mu (and the Density's
decay ellipsoid), or the error the fit raised.  The comparison prints, per case, whether each build ran and whether all outputs
are np.array_equal, and the median of five warm fits at the headline size (cubic-2, n = 26, N = 4216) for each build.
"""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
import numpy as np


def _model_outputs(s, out, name):
    for i, c in enumerate(s.configs):
        out[name + '/coef%d' % i] = np.asarray(c._coef)
    for k in ('_mu', '_hess', '_alpha', '_f_mu'):
        out[name + '/' + k] = np.asarray(getattr(s, k))


def dump(path):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    import bayesfast_b200 as bfb
    import _golden_io as gio
    out, status = {}, {}

    def case(name, fn):
        try:
            fn(name)
            status[name] = 'ok'
        except Exception as e:                     # recorded: a build that cannot run a case says why
            status[name] = 'error: ' + str(e).splitlines()[0][:300]
        print(name, status[name], flush=True)

    for c in gio.load('fit.npz')['cases']:
        def golden(name, c=c):
            spec = c['spec']
            cfgs = [bfb.PolyConfig(cf['order'], cf['input_mask'], cf['output_mask']) for cf in spec['configs']]
            s = bfb.PolyModel(cfgs, input_size=int(spec['n']), output_size=int(spec['m']),
                              bound_options=dict(alpha_p=float(c['alpha_p']), center_max=bool(c['center_max'])))
            s.fit(c['x'], c['y'], c['logp'], c['w'])
            _model_outputs(s, out, name)
        case('golden_' + c['name'], golden)

    for n, N, scale in ((26, 4216, 1.0), (16, 1636, 1.0), (26, 4216, 0.3), (32, 20000, 1.0)):
        def lstsq_shape(name, n=n, N=N, scale=scale):
            rng = np.random.default_rng(n)
            A = rng.normal(size=(n, n))
            P = A @ A.T / n + np.eye(n)
            x = rng.normal(size=(N, n)) * scale
            y = (-0.5 * np.einsum('ij,jk,ik->i', x, P, x) - 0.02 * np.sum(x**3 * np.exp(-0.1 * x**2), axis=1))[:, None]
            s = bfb.PolyModel('cubic-2', input_size=n, output_size=1)
            s.fit(x, y, logp=y[:, 0])
            _model_outputs(s, out, name)
        case('lstsq_n%d_N%d_s%g' % (n, N, scale), lstsq_shape)

    def density(name):
        n = 8
        rng = np.random.default_rng(1)
        A = rng.normal(size=(n, n))
        cov = A @ A.T / n + np.eye(n)
        xf = (np.linalg.cholesky(cov) @ rng.normal(size=(n, 2000))).T
        logp = -0.5 * np.einsum('ij,jk,ik->i', xf, np.linalg.inv(cov), xf)
        sur = bfb.PolyModel('cubic-2', input_size=n, output_size=1)
        den = bfb.Density(sur, decay_options=dict(use_decay=True))
        den.fit(xf, logp)
        _model_outputs(sur, out, name)
        out[name + '/d_mu'], out[name + '/d_hess'], out[name + '/d_alpha'] = den._mu, den._hess, np.asarray(den._alpha)
    case('density_decay_n8', density)

    for order, n in (('cubic-2', 53), ('cubic-2', 54), ('cubic-2', 60), ('quadratic', 64)):
        def wide(name, order=order, n=n):
            s = bfb.PolyModel(order, input_size=n, output_size=1)
            rng = np.random.default_rng(n)
            x = rng.normal(size=(2 * s.n_param, n))
            y = (-0.5 * np.sum(x**2, axis=1) + 0.1 * x[:, 0] * x[:, -1]**2 + 1e-3 * rng.normal(size=x.shape[0]))[:, None]
            s.fit(x, y, logp=y[:, 0])
            _model_outputs(s, out, name)
        case('%s_n%d' % (order, n), wide)

    n, N = 26, 4216                                # headline fit size: warm wall time
    rng = np.random.default_rng(n)
    x = rng.normal(size=(N, n))
    y = (-0.5 * np.sum(x**2, axis=1) + 0.1 * x[:, 0] * x[:, 1]**2)[:, None]
    s = bfb.PolyModel('cubic-2', input_size=n, output_size=1)
    s.fit(x, y, logp=y[:, 0])
    ts = []
    for _ in range(5):
        t0 = time.perf_counter()
        s.fit(x, y, logp=y[:, 0])
        ts.append(time.perf_counter() - t0)
    out['__headline_fit_s'] = np.asarray(ts)
    out['__status_names'] = np.asarray(list(status.keys()))
    out['__status'] = np.asarray(list(status.values()))
    np.savez(path, **out)


def compare(pa, pb):
    a, b = np.load(pa), np.load(pb)
    sa = dict(zip(a['__status_names'], a['__status']))
    sb = dict(zip(b['__status_names'], b['__status']))
    all_equal = True
    for name in sa:
        keys = sorted(k for k in b.files if k.startswith(name + '/'))
        if sa[name] == 'ok' and sb[name] == 'ok':
            eq = all(np.array_equal(a[k], b[k]) for k in keys)
            all_equal &= eq
            print('%-28s both ran, %d outputs, %s' % (name, len(keys), 'all np.array_equal' if eq else 'DIFFERENT'))
        else:
            print('%-28s A: %s | B: %s' % (name, sa[name], sb[name]))
    for tag, d in (('A', a), ('B', b)):
        t = d['__headline_fit_s']
        print('%s warm PolyModel.fit cubic-2 n=26 N=4216: median %.2f ms (min %.2f, max %.2f)'
              % (tag, 1e3 * np.median(t), 1e3 * t.min(), 1e3 * t.max()))
    print('outputs of the cases both builds ran:', 'bit-identical' if all_equal else 'NOT identical')
    return all_equal


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--lib-a', required=True)
    ap.add_argument('--lib-b', required=True)
    ap.add_argument('--out-dir', required=True)
    ap.add_argument('--dump', default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.dump:
        return dump(a.dump)
    os.makedirs(a.out_dir, exist_ok=True)
    paths = []
    for tag, lib in (('a', a.lib_a), ('b', a.lib_b)):
        p = os.path.join(a.out_dir, 'fit_ab_%s.npz' % tag)
        env = dict(os.environ, BFB200_LIB=os.path.abspath(lib))
        print('== build %s: %s' % (tag.upper(), lib), flush=True)
        subprocess.run([sys.executable, os.path.abspath(__file__), '--lib-a', lib, '--lib-b', lib, '--out-dir', a.out_dir,
                        '--dump', p], env=env, check=True)
        paths.append(p)
    sys.exit(0 if compare(*paths) else 1)


if __name__ == '__main__':
    main()
