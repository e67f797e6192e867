"""Nested dict <-> flat .npz helpers shared by tests/ and tests/golden/make_golden.py."""
import hashlib
import os
import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def flatten(d, prefix=''):
    out = {}
    if isinstance(d, dict):
        for k, v in d.items():
            out.update(flatten(v, prefix + str(k) + '/'))
    elif isinstance(d, (list, tuple)) and len(d) > 0 and isinstance(d[0], (dict, list, tuple)):
        out[prefix + '__len__'] = np.asarray(len(d))
        for i, v in enumerate(d):
            out.update(flatten(v, prefix + str(i) + '/'))
    elif d is None:
        out[prefix + '__none__'] = np.asarray(0)
    else:
        out[prefix[:-1]] = np.asarray(d)
    return out


def unflatten(flat):
    root = {}
    for key in flat:
        parts = key.split('/')
        cur = root
        for p in parts[:-1]:
            cur = cur.setdefault(p, {})
        cur[parts[-1]] = flat[key]

    def fix(node):
        if not isinstance(node, dict):
            a = np.asarray(node)
            if a.dtype.kind in 'US' and a.ndim == 0:
                return str(a)
            if a.ndim == 0 and a.dtype.kind == 'b':
                return bool(a)
            return a
        if '__none__' in node:
            return None
        if '__len__' in node:
            return [fix(node[str(i)]) for i in range(int(node['__len__']))]
        return {k: fix(v) for k, v in node.items()}

    return fix(root)


def draws_digest(u, z):
    """sha256 of a run's uniform and normal draws (float64, little-endian): pins draws a golden file regenerates instead of
    storing them"""
    h = hashlib.sha256(np.ascontiguousarray(u, '<f8').tobytes())
    h.update(np.ascontiguousarray(z, '<f8').tobytes())
    return h.hexdigest()


def save(name, d):
    np.savez_compressed(os.path.join(GOLDEN_DIR, name), **flatten(d))


def load(name):
    with np.load(os.path.join(GOLDEN_DIR, name), allow_pickle=False) as z:
        return unflatten({k: z[k] for k in z.files})
