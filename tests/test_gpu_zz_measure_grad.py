"""GPU backward of BodyMeasurements (csrc/measure_grad.cu) and of SMPLX.forward_shape (smplx_shape_backward_kernel):
against the reference's own autograd (tests/golden/measure_grad.npz) and the NumPy oracle
(tests/measure_grad_oracle.py), homogeneity, determinism, the unchanged forward, and a first-order fit of shape
coefficients to measurements."""
import os

import numpy as np
import pytest
import torch

import measure_grad_oracle as mgo
from shapy_b200 import ops, synth

pytestmark = pytest.mark.gpu
DEG = np.array([3.0, 1.0, 1.0, 1.0, 1.0])


@pytest.fixture(scope='module')
def data(golden_dir):
    g = np.load(os.path.join(golden_dir, 'img00_body.npz'))
    ref = np.load(os.path.join(golden_dir, 'measure_grad.npz'))
    bodies = np.concatenate([g['v_shaped'][None], g['extra_v_shaped']], 0).astype(np.float32)
    lm = synth.load_landmarks()
    return g, ref, bodies, lm, ops.make_landmarks(lm)


def one_hot_grads(lmk, v, faces, triangles=False):
    """(5, B, ...) gradients of the five measurements of every body of v, one backward call."""
    B = v.shape[0]
    rep = v.repeat(5, 1, 1)                                            # row j * B + b: body b, measurement j
    g = torch.eye(5, device=v.device).repeat_interleave(B, 0)
    if triangles:
        tris = rep[:, faces.long()].contiguous()
        return ops.measure_backward(lmk, g, triangles=tris).view(5, B, -1, 3, 3)
    return ops.measure_backward(lmk, g, v_shaped=rep.contiguous(), faces_i32=faces).view(5, B, -1, 3)


def tris_to_verts(gt, faces, V):
    out = torch.zeros(gt.shape[0], V, 3, dtype=torch.float64, device=gt.device)
    for k in range(3):
        out.index_add_(1, faces[:, k].long(), gt[:, :, k].double())
    return out


def test_golden_bodies_both_entries(data):
    g, ref, bodies, lm, lmk = data
    v = torch.from_numpy(bodies).cuda()
    f = torch.from_numpy(g['faces']).cuda()
    gv = one_hot_grads(lmk, v, f).double().cpu().numpy()
    gt = one_hot_grads(lmk, v, f, triangles=True)
    V = bodies.shape[1]
    for b in range(len(bodies)):
        gt_v = tris_to_verts(gt[:, b], f, V).cpu().numpy()
        oracle_mass = None
        for i, name in enumerate(mgo.NAMES):
            if name == 'mass' and b >= len(ref['mass_grad']):
                if oracle_mass is None:
                    oracle_mass = mgo.measure_grad(bodies[b], g['faces'], lm)[0]
                r = oracle_mass
            else:
                r = np.zeros((V, 3))
                if name == 'mass':
                    r = ref['mass_grad'][b].astype(np.float64)
                else:
                    sel = ref[f'{name}_body'] == b
                    r[ref[f'{name}_vertex'][sel]] = ref[f'{name}_grad'][sel]
            scale = np.abs(r).max()
            assert np.abs(gv[i, b] - r).max() <= 1e-5 * scale, (b, name, np.abs(gv[i, b] - r).max() / scale)
            assert np.abs(gt_v[i] - r).max() <= 1e-5 * scale, (b, name, 'triangles')
            assert np.abs(gt_v[i] - gv[i, b]).max() <= 1e-6 * np.abs(gv[i, b]).max(), (b, name, 'entries')


def _random_beta_bodies():
    smplx = synth.make_smplx()
    packed = ops.SmplxModel(dict(smplx), 'cuda')
    betas = torch.randn(4096, 10, generator=torch.Generator().manual_seed(3)).clamp(-3, 3)
    vs = ops.smplx_forward_shape(packed, betas.cuda())
    return smplx, vs, smplx['faces_tensor'].to(torch.int32).cuda()


def test_random_beta_bodies_vs_oracle_and_nan_rows(data):
    """64 of the 4 096 random-beta bodies of configs[3] (60 seeded rows + 4 whose forward overflows to NaN)."""
    g, ref, bodies, lm, lmk = data
    smplx, vs, faces = _random_beta_bodies()
    out = ops.measure(lmk, v_shaped=vs, faces_i32=faces).cpu().numpy()
    nan_rows = np.nonzero(np.isnan(out).any(1))[0][:4]
    assert len(nan_rows) > 0
    finite = np.nonzero(~np.isnan(out).any(1))[0]
    rows = list(np.random.default_rng(5).choice(finite, 60, replace=False)) + list(nan_rows)
    sub = vs[torch.tensor(rows, device='cuda')].contiguous()
    gv = one_hot_grads(lmk, sub, faces).double().cpu().numpy()
    f = smplx['faces_tensor'].numpy()
    for j, r in enumerate(rows):
        if r in nan_rows:
            for i in range(5):
                assert np.isnan(gv[i, j]).all() == bool(np.isnan(out[r, i])), (int(r), i)
            continue
        want = mgo.measure_grad(sub[j].cpu().numpy(), f, lm, max_collisions=4096)
        for i, name in enumerate(mgo.NAMES):
            scale = np.abs(want[i]).max()
            err = np.abs(gv[i, j] - want[i]).max()
            assert err <= 1e-5 * scale, (int(r), name, err / scale)
    # a zero upstream entry for the NaN measurement contributes exactly nothing
    r = int(nan_rows[0])
    mask = torch.tensor([[1.0, 1.0] + [0.0 if np.isnan(out[r, 2 + p]) else 1.0 for p in range(3)]], device='cuda')
    x = vs[r:r + 1].contiguous()
    masked = ops.measure_backward(lmk, mask, v_shaped=x, faces_i32=faces)
    assert torch.isfinite(masked).all()
    parts = sum(ops.measure_backward(lmk, mask * torch.eye(5, device='cuda')[i], v_shaped=x, faces_i32=faces).double()
                for i in range(5) if mask[0, i] != 0)
    assert float((masked.double() - parts).abs().max()) <= 1e-6 * float(parts.abs().max())


def test_homogeneity_on_gpu_gradients(data):
    """<v, dm/dv> = deg * m for every finite row: the backward rebuilt the forward's hull."""
    g, ref, bodies, lm, lmk = data
    smplx, vs, faces = _random_beta_bodies()
    v = torch.cat([torch.from_numpy(bodies).cuda(), vs[:252]]).contiguous()
    m = ops.measure(lmk, v_shaped=v, faces_i32=faces).double()
    gv = one_hot_grads(lmk, v, faces).double()
    lhs = (gv * v.double()[None]).sum((2, 3)).t()                    # (B, 5)
    rhs = m * torch.tensor(DEG, device='cuda')
    fin = torch.isfinite(m)
    assert int(fin.all(1).sum()) > 200
    rel = ((lhs - rhs).abs() / rhs.abs())[fin]
    assert float(rel.max()) <= 1e-5, float(rel.max())


def test_determinism_and_batch_position(data):
    g, ref, bodies, lm, lmk = data
    f = torch.from_numpy(g['faces']).cuda()
    base = torch.from_numpy(bodies).cuda()
    big = base[torch.arange(1024) % 4]
    scale = (1.0 + 0.05 * torch.sin(torch.arange(1024, dtype=torch.float32))).view(-1, 1, 1).cuda()
    big = (big * scale).contiguous()
    gout = torch.randn(1024, 5, generator=torch.Generator().manual_seed(1)).cuda()
    a = ops.measure_backward(lmk, gout, v_shaped=big, faces_i32=f)
    b = ops.measure_backward(lmk, gout, v_shaped=big, faces_i32=f)
    assert torch.equal(a, b)
    for r in (0, 517, 1023):
        one = ops.measure_backward(lmk, gout[r:r + 1].contiguous(), v_shaped=big[r:r + 1].contiguous(), faces_i32=f)
        assert torch.equal(one[0], a[r])
    tris = big[:64][:, f.long()].contiguous()
    ta = ops.measure_backward(lmk, gout[:64].contiguous(), triangles=tris)
    assert torch.equal(ta, ops.measure_backward(lmk, gout[:64].contiguous(), triangles=tris))
    assert torch.equal(ta[7], ops.measure_backward(lmk, gout[7:8].contiguous(), triangles=tris[7:8].contiguous())[0])


def test_module_forward_unchanged_and_first_derivative_only(data):
    from shapy_b200.body_measurements import BodyMeasurements
    g, ref, bodies, lm, lmk = data
    bm = BodyMeasurements({'landmarks': lm}).cuda()
    f = torch.from_numpy(g['faces']).cuda()
    v = torch.from_numpy(bodies).cuda()
    with torch.no_grad():
        plain = bm.forward_vertices(v, f)['measurements']
        plain_t = bm(v[:, f.long()].contiguous())['measurements']
    x = v.clone().requires_grad_(True)
    out = bm.forward_vertices(x, f)['measurements']
    xt = v[:, f.long()].contiguous().requires_grad_(True)
    out_t = bm(xt, compute_waist=False)['measurements']
    for k in plain:
        assert torch.equal(out[k]['tensor'], plain[k]['tensor']), k
        assert out[k]['tensor'].requires_grad
        if k != 'waist':
            assert torch.equal(out_t[k]['tensor'], plain_t[k]['tensor']), k
    assert bm.last_status is not None and int(bm.last_status.item()) == 0
    # module autograd == the op with the same upstream gradient; a dropped measurement gets none
    w = torch.tensor([1.0, 100.0, 2000.0, 1000.0, 1000.0], device='cuda')
    loss = sum(w[i] * out[k]['tensor'].sum() for i, k in enumerate(mgo.NAMES))
    loss.backward()
    want = ops.measure_backward(lmk, w.expand(4, 5).contiguous(), v_shaped=v, faces_i32=f)
    assert torch.equal(x.grad, want)
    loss_t = sum(w[i] * out_t[k]['tensor'].sum() for i, k in enumerate(mgo.NAMES) if k in out_t)
    loss_t.backward()
    wt = w.clone()
    wt[3] = 0
    assert torch.equal(xt.grad, ops.measure_backward(lmk, wt.expand(4, 5).contiguous(), triangles=xt.detach()))
    # second derivatives are not supported: differentiating the gradient raises
    x2 = v.clone().requires_grad_(True)
    m = bm.forward_vertices(x2, f)['measurements']['chest']['tensor'].sum()
    gx, = torch.autograd.grad(m, x2, create_graph=True)
    with pytest.raises(RuntimeError):
        gx.sum().backward()


def _smplx_module(shapedirs=None):
    from shapy_b200.human_shape.models.body_models.body_models import SMPLX
    ds = synth.make_smplx()
    if shapedirs is not None:
        ds['shapedirs'] = shapedirs
    return SMPLX(data_struct=ds).cuda(), ds


@pytest.mark.parametrize('B', [1, 64, 4096])
def test_forward_shape_backward(B):
    model, ds = _smplx_module()
    nb = model.packed('cuda').NB
    betas = torch.randn(B, nb, generator=torch.Generator().manual_seed(B)).cuda().requires_grad_(True)
    vs = model.forward_shape(betas)['v_shaped']
    with torch.no_grad():
        assert torch.equal(vs, model.forward_shape(betas)['v_shaped'])
    gv = torch.randn(vs.shape, generator=torch.Generator().manual_seed(B + 1)).cuda()
    vs.backward(gv)
    S = ds['shapedirs'].double().reshape(-1, betas.shape[1])           # (3V, NB)
    want = gv.double().reshape(B, -1).cpu() @ S
    got = betas.grad.double().cpu()
    assert float((got - want).abs().max() / want.abs().max()) <= 1e-5
    if B == 4096:           # a body's gradient does not depend on its position in the batch
        one = ops.smplx_shape_backward(model.packed('cuda'), gv[1234:1235].contiguous())
        assert torch.equal(one[0], betas.grad[1234])


def smooth_shape_basis(vt, landmarks, faces):
    """Ten smooth directions (low-frequency scalings of the template): overall size, height, and girth bumps around
    the chest, waist and hip planes and between them."""
    vt = vt.double()
    c = vt.mean(0)
    d = vt - c
    ys = [float((vt[faces[landmarks[n]['face_idx']]] * torch.tensor(landmarks[n]['bc'], dtype=torch.float64)[:, None])
                .sum(0)[1]) for n in ('chest', 'waist', 'hips')]
    girth = torch.stack([d[:, 0], torch.zeros_like(d[:, 0]), d[:, 2]], 1)
    dirs = [0.05 * d, 0.05 * torch.stack([torch.zeros_like(d[:, 0]), d[:, 1], torch.zeros_like(d[:, 0])], 1)]
    for y in ys + [(ys[0] + ys[1]) / 2, (ys[1] + ys[2]) / 2, ys[2] - 0.25, ys[0] + 0.2]:
        dirs.append(0.05 * girth * torch.exp(-((vt[:, 1:2] - y) / 0.12) ** 2))
    dirs.append(0.05 * girth)
    return torch.stack(dirs, -1).float()                               # (V, 3, 10)


FIT_STEPS = 30


def test_fit_betas_to_measurements():
    """forward_shape -> forward_vertices -> the reference example's weighted loss -> backward, torch.optim.LBFGS on 64
    bodies whose targets are the measurements of seeded beta* bodies."""
    from shapy_b200.body_measurements import BodyMeasurements
    lm = synth.load_landmarks()
    ds0 = synth.make_smplx()
    S = smooth_shape_basis(ds0['v_template'], lm, ds0['faces_tensor'])
    model, ds = _smplx_module(S)
    bm = BodyMeasurements({'landmarks': lm}).cuda()
    f = model.faces_i32
    B = 64
    beta_star = (torch.randn(B, 10, generator=torch.Generator().manual_seed(7)) * 0.7).clamp(-1.5, 1.5).cuda()
    w = torch.tensor([1.0, 100.0, 2000.0, 1000.0, 1000.0], device='cuda')
    with torch.no_grad():
        target = bm.forward_vertices(model.forward_shape(beta_star)['v_shaped'], f)['measurements']
        target = torch.stack([target[k]['tensor'] for k in mgo.NAMES], 1)
    assert torch.isfinite(target).all()
    betas = torch.zeros(B, 10, device='cuda', requires_grad=True)
    opt = torch.optim.LBFGS([betas], lr=1.0, max_iter=20, history_size=20, line_search_fn='strong_wolfe',
                            tolerance_grad=0.0, tolerance_change=0.0)

    def closure():
        opt.zero_grad()
        m = bm.forward_vertices(model.forward_shape(betas)['v_shaped'], f)['measurements']
        est = torch.stack([m[k]['tensor'] for k in mgo.NAMES], 1)
        loss = ((target - est) ** 2 * w).sum()
        loss.backward()
        return loss
    for _ in range(FIT_STEPS):
        opt.step(closure)
    with torch.no_grad():
        m = bm.forward_vertices(model.forward_shape(betas)['v_shaped'], f)['measurements']
        est = torch.stack([m[k]['tensor'] for k in mgo.NAMES], 1)
    err = (est - target).abs()
    print('fit: max |error| mass %.2e kg, height / chest / waist / hips %s m' % (
        float(err[:, 0].max()), ['%.2e' % float(e) for e in err[:, 1:].max(0).values]))
    assert float(err[:, 0].max()) <= 0.1
    assert float(err[:, 1:].max()) <= 1e-3
