"""The NumPy gradient oracle of BodyMeasurements (tests/measure_grad_oracle.py) against the reference's own autograd
(tests/golden/measure_grad.npz, written by tools/make_golden.py measure_grad) on the four real bodies, and its
homogeneity: with the barycentrics fixed, mass is homogeneous of degree 3 in the vertices and height and the
circumferences of degree 1, so <v, dm/dv> = deg * m (Euler)."""
import os

import numpy as np
import pytest

import measure_grad_oracle as mgo
from oracle import measure_oracle
from shapy_b200 import synth


@pytest.fixture(scope='module')
def data(golden_dir):
    g = np.load(os.path.join(golden_dir, 'img00_body.npz'))
    ref = np.load(os.path.join(golden_dir, 'measure_grad.npz'))
    bodies = np.concatenate([g['v_shaped'][None], g['extra_v_shaped']], 0).astype(np.float32)
    lm = synth.load_landmarks()
    grads = [mgo.measure_grad(v, g['faces'], lm) for v in bodies]
    return g, ref, bodies, lm, grads


def ref_dense(ref, name, b, V):
    """The reference gradient of measurement `name` for body b as a dense (V, 3) array."""
    if name == 'mass':
        return ref['mass_grad'][b].astype(np.float64)
    out = np.zeros((V, 3), np.float64)
    sel = ref[f'{name}_body'] == b
    out[ref[f'{name}_vertex'][sel]] = ref[f'{name}_grad'][sel]
    return out


def test_oracle_gradient_matches_reference_autograd(data):
    g, ref, bodies, lm, grads = data
    V = bodies.shape[1]
    for b in range(len(bodies)):
        for i, name in enumerate(mgo.NAMES):
            if name == 'mass' and b >= len(ref['mass_grad']):
                continue
            r = ref_dense(ref, name, b, V)
            tol = (1e-6 if name in ('mass', 'height') else 1e-5) * np.abs(r).max()
            err = np.abs(grads[b][i] - r).max()
            assert err <= tol, (b, name, err, tol)
            if name != 'mass':
                assert ((np.abs(grads[b][i]).sum(-1) > 0) == (np.abs(r).sum(-1) > 0)).all(), (b, name)


def test_oracle_gradient_is_homogeneous(data):
    g, ref, bodies, lm, grads = data
    for b, v in enumerate(bodies):
        m = measure_oracle.measure(v, g['faces'], lm)
        for i, (name, deg) in enumerate(zip(mgo.NAMES, (3, 1, 1, 1, 1))):
            lhs = float((v.astype(np.float64) * grads[b][i]).sum())
            assert abs(lhs - deg * m[name]) <= 1e-5 * deg * abs(m[name]), (b, name, lhs, deg * m[name])
