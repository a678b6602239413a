"""shapy_mmi_forward against the REFERENCE's own CUDA kernel (SURVEY.md 8c: the patched build of the reference operator is
the GPU-side oracle).  tests/golden/ref_mmi.npz holds what that kernel returned on a B200 for the inputs below:
tools/make_golden.py mmi runs it (oracle/build_ref.py compiles it into oracle/_ref/, oracle/run_ref_mmi.py runs it in a
process of its own because it exit(0)s on CUDA errors) and stores every collision slot and the barycentrics of the filled
ones.  The C restatement oracle/mmi_oracle.c, pinned by the img_00 golden, is the other checker.
The reference is compiled with nvcc's default FMA contraction, shapy_b200's predicates with -fmad=false (to be bit-equal
to the plain-C oracle), so a pair sitting exactly on a tolerance (SAT `CMP`, |det| < 1e-4) may legitimately fall on
different sides: the bars below allow a handful of such pairs and are otherwise exact."""
import os

import numpy as np
import pytest
import torch

from shapy_b200 import synth

pytestmark = pytest.mark.gpu
PLANE_M, SOUP_M = 256, 64


def plane_queries(golden_dir):
    """The two triangles of the chest measurement plane of each of the four real bodies, and the bodies' triangles."""
    g = np.load(os.path.join(golden_dir, 'img00_body.npz'))
    lm = synth.load_landmarks()
    bodies = np.concatenate([g['v_shaped'][None], g['extra_v_shaped']], 0).astype(np.float32)
    tris = bodies[:, g['faces']]                                               # (4, F, 3, 3)
    queries = []
    for b in range(bodies.shape[0]):
        h = float((tris[b, lm['chest']['face_idx']] * np.float32(lm['chest']['bc'])[:, None]).sum(0)[1])
        quad = np.float32([[-1, h, -1], [1, h, -1], [1, h, 1], [-1, h, 1]])     # body_measurements.py:90-97
        queries.append(np.stack([quad[[0, 1, 2]], quad[[0, 2, 3]]]))
    return np.stack(queries).astype(np.float32), np.ascontiguousarray(tris)


def reference(golden_dir, tag):
    """The stored arrays of one case: `faces` (B, Q*M) and `bcs` (B, Q*M, 2, 3) of the reference kernel (the barycentrics
    are stored for the filled slots only), and the inputs where the test cannot rebuild them."""
    g = np.load(os.path.join(golden_dir, 'ref_mmi.npz'))
    out = {k[len(tag) + 1:]: g[k] for k in g.files if k.startswith(tag + '_')}
    bcs = np.zeros(out['faces'].shape + (2, 3), np.float32)
    bcs[out['faces'] >= 0] = out['bcs']
    out['bcs'] = bcs
    return out


def compare(r, m, max_set_diff, what):
    """r, m: {(query, face): bcs}.  Collision sets equal up to max_set_diff borderline pairs; barycentrics of the common
    pairs equal to 1e-4 for all but 1 % (a borderline ray test flips which edge supplies the point)."""
    diff = set(r) ^ set(m)
    assert len(diff) <= max_set_diff, (what, len(diff), sorted(diff)[:8])
    common = sorted(set(r) & set(m))
    bad = [k for k in common if np.abs(r[k] - m[k]).max() > 1e-4]
    assert len(bad) <= max(1, len(common) // 100), (what, len(bad), len(common), bad[:4])
    return len(common)


def as_dict(faces, bcs, M):
    """{(query, face): bcs (2,3)} of one body."""
    out = {}
    for s in np.nonzero(faces >= 0)[0]:
        out[(int(s) // M, int(faces[s]))] = bcs[s]
    return out


def test_plane_queries_on_real_bodies(golden_dir):
    """The hot-path use: the two triangles of a measurement plane against the 20 908 body triangles."""
    from shapy_b200 import ops
    query, tris = plane_queries(golden_dir)
    M = PLANE_M
    ref = reference(golden_dir, 'plane')
    ref_f, ref_b = ref['faces'], ref['bcs']
    mine_f, mine_b = ops.mesh_to_mesh_forward(torch.from_numpy(query).cuda(), torch.from_numpy(tris).cuda(), M)
    mine_f, mine_b = mine_f.cpu().numpy(), mine_b.cpu().numpy()
    for b in range(query.shape[0]):
        r, m = as_dict(ref_f[b], ref_b[b], M), as_dict(mine_f[b], mine_b[b], M)
        assert compare(r, m, 2, f'body {b}') > 50


def test_random_mesh_against_mesh(golden_dir):
    """General use of the operator: every triangle of one mesh against another."""
    from shapy_b200 import ops
    M = SOUP_M
    ref = reference(golden_dir, 'soup')        # ~180 colliding pairs, at most 5 per query (C oracle)
    query, target, ref_f, ref_b = ref['query'], ref['target'], ref['faces'], ref['bcs']
    mine_f, mine_b = ops.mesh_to_mesh_forward(torch.from_numpy(query).cuda(), torch.from_numpy(target).cuda(), M)
    mine_f, mine_b = mine_f.cpu().numpy(), mine_b.cpu().numpy()
    total = 0
    for b in range(query.shape[0]):
        r, m = as_dict(ref_f[b], ref_b[b], M), as_dict(mine_f[b], mine_b[b], M)
        total += compare(r, m, max(2, len(r) // 100), f'soup {b}')
    assert total > 100
