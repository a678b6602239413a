"""NumPy restatement of the gradient of BodyMeasurements (the reference's autograd through
mesh-mesh-intersection/body_measurements/body_measurements.py:132-215), on top of oracle/measure_oracle.

  mass    analytic: corner k of face f gets sign(sum det) 985/6 (T_k+1 x T_k+2)
  height  analytic: the y components of the two landmark faces, +/- sign(y_ht - y_hl) bc_k
  chest / waist / hips  the oracle's own collision records (face, barycentrics) and the qhull simplices the reference
          sums over: each hull edge (a, b) adds -/+ (p_b - p_a) / |p_b - p_a| to its points, each point bc_k times
          that to the corners of its face (the barycentrics and the plane height are constants, as under the
          reference's no_grad).

Pinned to the reference's own autograd by tests/golden/measure_grad.npz (tests/test_measure_grad_cpu.py).
"""
import numpy as np

from oracle import measure_oracle

NAMES = ('mass', 'height', 'chest', 'waist', 'hips')


def periphery_grad(tris, face_idx, bc, max_collisions=256):
    """(value, d value / d tris (F,3,3) float64) for one circumference of one body."""
    from scipy.spatial import ConvexHull
    bc = np.asarray(bc, np.float32)
    vertex = (tris[face_idx] * bc.reshape(3, 1)).sum(axis=0, dtype=np.float32)
    q = measure_oracle.plane_quad(np.float32(vertex[1]))
    faces, bcs = measure_oracle.mesh_to_mesh_forward(q[None], tris[None], max_collisions)
    faces, bcs = faces[0], bcs[0]
    valid = np.where(faces > 0)[0]
    pts = (tris[faces[valid]][:, None] * bcs[valid][..., None]).sum(axis=-2, dtype=np.float32)  # (n,2,3)
    flat = pts.reshape(-1, 3)
    hull = ConvexHull(flat[:, [0, 2]])
    gp = np.zeros(flat.shape, np.float64)
    value = 0.0
    for a, b in hull.simplices:
        d = flat[b].astype(np.float64) - flat[a]
        n = np.sqrt((d * d).sum())
        value += n
        gp[a] -= d / n
        gp[b] += d / n
    g = np.zeros(tris.shape, np.float64)
    rec_face = np.repeat(faces[valid], 2)           # point j = record j // 2, copy j % 2
    rec_bc = bcs[valid].reshape(-1, 3).astype(np.float64)
    np.add.at(g, rec_face, rec_bc[:, :, None] * gp[:, None, :])
    return value, g


def measure_grad_tris(tris, lm, max_collisions=256):
    """tris (F,3,3) float32 -> (5, F, 3, 3) float64: d(mass, height, chest, waist, hips) / d tris."""
    tris = np.ascontiguousarray(tris, np.float32)
    out = np.zeros((5,) + tris.shape, np.float64)
    t = tris.astype(np.float64)
    x, y, z = tris[..., 0], tris[..., 1], tris[..., 2]
    vol = (-x[:, 2] * y[:, 1] * z[:, 0] + x[:, 1] * y[:, 2] * z[:, 0] + x[:, 2] * y[:, 0] * z[:, 1]
           - x[:, 0] * y[:, 2] * z[:, 1] - x[:, 1] * y[:, 0] * z[:, 2] + x[:, 0] * y[:, 1] * z[:, 2])
    s = np.sign(vol.sum(dtype=np.float32))
    for k in range(3):
        out[0, :, k] = s * measure_oracle.DENSITY / 6.0 * np.cross(t[:, (k + 1) % 3], t[:, (k + 2) % 3])
    ht, hl = lm['head_top'], lm['left_heel']
    yht = (tris[ht['face_idx']] * np.asarray(ht['bc'], np.float32).reshape(3, 1)).sum(0)[1]
    yhl = (tris[hl['face_idx']] * np.asarray(hl['bc'], np.float32).reshape(3, 1)).sum(0)[1]
    sh = np.sign(np.float32(yht) - np.float32(yhl))
    out[1, ht['face_idx'], :, 1] += sh * np.asarray(ht['bc'], np.float64)
    out[1, hl['face_idx'], :, 1] -= sh * np.asarray(hl['bc'], np.float64)
    for i, name in enumerate(NAMES[2:]):
        out[2 + i] = periphery_grad(tris, lm[name]['face_idx'], lm[name]['bc'], max_collisions)[1]
    return out


def measure_grad(v_shaped, faces, lm=None, max_collisions=256):
    """v_shaped (V,3) float32, faces (F,3) -> (5, V, 3) float64: d(mass, height, chest, waist, hips) / d v_shaped."""
    lm = lm or measure_oracle.load_landmarks()
    faces = np.asarray(faces, np.int64)
    gt = measure_grad_tris(np.asarray(v_shaped, np.float32)[faces], lm, max_collisions)
    out = np.zeros((5,) + np.shape(v_shaped), np.float64)
    for k in range(3):
        np.add.at(out, (slice(None), faces[:, k]), gt[:, :, k])
    return out
