"""Tensor-level wrappers over the C ABI (include/shapy_b200.h).

PyTorch is used for device memory and streams only: every function takes CUDA fp32 tensors, allocates
the outputs with torch, and launches the hand-written sm_100a kernels on the current stream.  Nothing
here computes with torch ops, and nothing falls back to the CPU: non-CUDA inputs raise.
"""
import ctypes as C
import weakref

import numpy as np
import torch

from . import _lib
from ._lib import check, lib, ptr, stream_ptr


def _cuda_f32(t, name):
    if not (torch.is_tensor(t) and t.is_cuda):
        raise RuntimeError(f'shapy_b200: `{name}` must be a CUDA tensor (there is no CPU path)')
    if t.dtype != torch.float32:
        raise RuntimeError(f'shapy_b200: `{name}` must be float32, got {t.dtype}')
    return t.contiguous()


class _Workspace:
    """Grow-only per-device scratch buffer (plumbing, not math)."""

    def __init__(self):
        self.bufs = {}

    def get(self, key, nbytes, device):
        k = (key, device.index)
        b = self.bufs.get(k)
        if b is None or b.numel() < nbytes:
            b = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
            self.bufs[k] = b
        return b


_WS = _Workspace()


# ------------------------------------------------------------------------------------------ SMPL-X
class SmplxModel:
    """Device-side packed SMPL-X constants (shapy_smplx_create).  `tensors` uses the reference's
    buffer names (body_models.py:112-166, 563-597)."""

    def __init__(self, tensors: dict, device):
        self.device = torch.device(device)
        h = {}

        def host(name, dtype, required=True):
            t = tensors.get(name)
            if t is None or (torch.is_tensor(t) and t.numel() == 0):
                if required:
                    raise RuntimeError(f'SMPL-X tensor `{name}` missing')
                return None
            a = np.ascontiguousarray(t.detach().cpu().numpy().astype(dtype))
            h[name] = a
            return a

        vt = host('v_template', np.float32)
        sd = host('shapedirs', np.float32)
        ed = host('expr_dirs', np.float32, False)
        pd = host('posedirs', np.float32)
        jr = host('J_regressor', np.float32)
        lw = host('lbs_weights', np.float32)
        par = host('parents', np.int64)
        fc = host('faces_tensor', np.int64)
        lf = host('lmk_faces_idx', np.int64, False)
        lb = host('lmk_bary_coords', np.float32, False)
        df = host('dynamic_lmk_faces_idx', np.int64, False)
        db = host('dynamic_lmk_bary_coords', np.float32, False)
        nk = host('neck_kin_chain', np.int64, False)
        ex = host('extra_joint_regressor', np.float32, False)
        si = host('source_idxs', np.int64, False)
        ti = host('target_idxs', np.int64, False)
        d = _lib.SmplxDesc()
        d.num_verts, d.num_joints = vt.shape[0], jr.shape[0]
        d.num_betas = sd.shape[-1]
        d.num_expr = 0 if ed is None else ed.shape[-1]
        d.num_faces = fc.shape[0]
        ap = lambda a: None if a is None else a.ctypes.data  # noqa: E731
        d.v_template, d.shapedirs, d.expr_dirs, d.posedirs = ap(vt), ap(sd), ap(ed), ap(pd)
        d.J_regressor, d.lbs_weights, d.parents, d.faces = ap(jr), ap(lw), ap(par), ap(fc)
        d.num_static_lmk = 0 if lf is None else lf.shape[0]
        d.lmk_faces_idx, d.lmk_bary_coords = ap(lf), ap(lb)
        use_dyn = df is not None and tensors.get('use_face_contour', True)
        d.num_dyn_lmk = df.shape[1] if use_dyn else 0
        d.num_dyn_rows = df.shape[0] if use_dyn else 0
        d.dynamic_lmk_faces_idx, d.dynamic_lmk_bary_coords = (ap(df), ap(db)) if use_dyn else (None, None)
        d.neck_chain_len = 0 if nk is None else nk.shape[0]
        d.neck_kin_chain = ap(nk)
        d.num_extra = 0 if ex is None else ex.shape[0]
        d.extra_joint_regressor = ap(ex)
        d.num_overwrite = 0 if si is None else si.shape[0]
        d.source_idxs, d.target_idxs = ap(si), ap(ti)
        self.V, self.J, self.NB, self.NE, self.F = d.num_verts, d.num_joints, d.num_betas, d.num_expr, d.num_faces
        handle = C.c_void_p()
        with torch.cuda.device(self.device):
            check(lib().shapy_smplx_create(C.byref(handle), C.byref(d)), 'smplx_create')
        self.handle = handle
        self.K = lib().shapy_smplx_num_keypoints(handle)
        self._fin = weakref.finalize(self, lib().shapy_smplx_destroy, handle)
        self._faces_ptr = lib().shapy_smplx_faces_i32(handle)

    @property
    def faces_ptr(self):
        return C.c_void_p(self._faces_ptr)


def decode_rot6d(raw: torch.Tensor) -> torch.Tensor:
    """(B, 6n) -> (B, n, 3, 3)  (ContinuousRotReprDecoder.forward, pose_utils.py:138-153)."""
    raw = _cuda_f32(raw, 'raw')
    B = raw.shape[0]
    n = raw.numel() // 6
    out = torch.empty(n, 3, 3, dtype=torch.float32, device=raw.device)
    if n == 0:            # empty batch: nothing to launch (torch semantics: empty in, empty out)
        return out.view(B, raw.shape[1] // 6 if raw.dim() > 1 else 0, 3, 3)
    with torch.cuda.device(raw.device):
        check(lib().shapy_decode_rot6d(ptr(raw), n, ptr(out), stream_ptr()), 'decode_rot6d')
    return out.view(B, -1, 3, 3)


def smplx_forward(model: SmplxModel, betas, rot, expr=None, camera=None, want_vertices=True, want_v_shaped=True,
                  want_joints=True):
    """rot (B, n_rot, 3, 3): rotations of the first n_rot joints of the full pose; the rest is identity."""
    betas = _cuda_f32(betas, 'betas')
    rot = _cuda_f32(rot, 'rot')
    B, n_rot = rot.shape[0], rot.shape[1]
    if betas.shape != (B, model.NB):
        raise RuntimeError(f'betas must be ({B}, {model.NB}), got {tuple(betas.shape)}')
    dev = betas.device
    expr = None if expr is None else _cuda_f32(expr, 'expression')
    camera = None if camera is None else _cuda_f32(camera, 'camera')
    mk = lambda *s: torch.empty(*s, dtype=torch.float32, device=dev)  # noqa: E731
    vertices = mk(B, model.V, 3) if want_vertices else None
    v_shaped = mk(B, model.V, 3) if want_v_shaped else None
    joints = mk(B, model.K, 3) if want_joints else None
    proj = mk(B, model.K, 2) if (want_joints and camera is not None) else None
    if B == 0:
        return dict(vertices=vertices, v_shaped=v_shaped, joints=joints, proj_joints=proj)
    with torch.cuda.device(dev):
        nbytes = lib().shapy_smplx_workspace_bytes(model.handle, B)
        ws = _WS.get('smplx', nbytes, dev)
        check(lib().shapy_smplx_forward(model.handle, ptr(betas), ptr(rot), n_rot, ptr(expr), ptr(camera), B,
                                        ptr(vertices), ptr(v_shaped), ptr(joints), ptr(proj), ptr(ws), ws.numel(),
                                        stream_ptr()), 'smplx_forward')
    return dict(vertices=vertices, v_shaped=v_shaped, joints=joints, proj_joints=proj)


def smplx_forward_shape(model: SmplxModel, betas) -> torch.Tensor:
    betas = _cuda_f32(betas, 'betas')
    B = betas.shape[0]
    out = torch.empty(B, model.V, 3, dtype=torch.float32, device=betas.device)
    if B == 0:
        return out
    with torch.cuda.device(betas.device):
        check(lib().shapy_smplx_forward_shape(model.handle, ptr(betas), B, ptr(out), stream_ptr()), 'forward_shape')
    return out


def smplx_shape_backward(model: SmplxModel, grad_v_shaped) -> torch.Tensor:
    """(B, V, 3) gradient of v_shaped -> (B, num_betas) gradient of betas (backward of smplx_forward_shape)."""
    g = _cuda_f32(grad_v_shaped, 'grad_v_shaped')
    B = g.shape[0]
    if g.shape != (B, model.V, 3):
        raise RuntimeError(f'grad_v_shaped must be ({B}, {model.V}, 3), got {tuple(g.shape)}')
    out = torch.empty(B, model.NB, dtype=torch.float32, device=g.device)
    if B == 0:
        return out
    with torch.cuda.device(g.device):
        check(lib().shapy_smplx_shape_backward(model.handle, ptr(g), B, ptr(out), stream_ptr()), 'smplx_shape_backward')
    return out


# ------------------------------------------------------------------------------------ measurements
def make_landmarks(lm: dict) -> _lib.MeasureLandmarks:
    """lm: {'head_top','left_heel','chest','waist','hips'} -> {'face_idx', 'bc'}."""
    s = _lib.MeasureLandmarks()
    for i, k in enumerate(('head_top', 'left_heel', 'chest', 'waist', 'hips')):
        s.face_idx[i] = int(lm[k]['face_idx'])
        for c in range(3):
            s.bc[i][c] = float(lm[k]['bc'][c])
    return s


def measure(landmarks: _lib.MeasureLandmarks, v_shaped=None, faces_i32=None, triangles=None, return_points=False,
            max_points=1024, strict=False):
    """Returns (B, 5) = mass, height, chest, waist, hips.  Either (v_shaped, faces_i32) or triangles (B,F,3,3).

    The kernel's point / candidate buffers have a fixed capacity (1024 points per plane; the reference's
    `max_collisions` has no equivalent).  A body that overflows them gets NaN circumferences, never a truncated value,
    and the device status word is set: it is returned as `out.status` (a 1-element int32 CUDA tensor, readable at the
    caller's next synchronisation point) and `strict=True` checks it here (one host synchronisation) and raises."""
    if triangles is not None:
        x = _cuda_f32(triangles, 'triangles')
        B, F = x.shape[0], x.shape[1]
    else:
        x = _cuda_f32(v_shaped, 'v_shaped')
        B, V = x.shape[0], x.shape[1]
        if not (torch.is_tensor(faces_i32) and faces_i32.is_cuda and faces_i32.dtype == torch.int32):
            raise RuntimeError('faces_i32 must be a CUDA int32 tensor')
        faces_i32 = faces_i32.contiguous()
        F = faces_i32.shape[0]
    dev = x.device
    out = torch.empty(B, 5, dtype=torch.float32, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    pts = cnt = None
    if return_points:
        pts = torch.zeros(B, 3, max_points, 3, dtype=torch.float32, device=dev)
        cnt = torch.zeros(B, 3, dtype=torch.int32, device=dev)
    if B == 0:
        out.status = status
        return (out, pts, cnt, status) if return_points else out
    with torch.cuda.device(dev):
        if triangles is not None:
            check(lib().shapy_measure_forward_tris(ptr(x), B, F, C.byref(landmarks), ptr(out), ptr(pts), ptr(cnt),
                                                   max_points, ptr(status), stream_ptr()), 'measure')
        else:
            check(lib().shapy_measure_forward(ptr(x), ptr(faces_i32), B, V, F, C.byref(landmarks), ptr(out), ptr(pts),
                                              ptr(cnt), max_points, ptr(status), stream_ptr()), 'measure')
    out.status = status
    if strict and int(status.item()) != 0:
        raise RuntimeError('shapy_b200 measure: a slicing plane produced more intersection points than the kernel can '
                           'hold (the affected circumferences are NaN)')
    if return_points:
        return out, pts, cnt, status
    return out


def measure_backward(landmarks: _lib.MeasureLandmarks, grad_out, v_shaped=None, faces_i32=None, triangles=None):
    """Backward of `measure`: grad_out (B, 5) -> the gradient of v_shaped (B, V, 3) or of triangles (B, F, 3, 3).

    First derivative only, with the intersection barycentrics and the slicing heights held constant.  Where `measure`
    returned a NaN circumference, the body's gradient is NaN if its grad_out entry is non-zero; a zero entry
    contributes nothing."""
    g = _cuda_f32(grad_out, 'grad_out')
    if triangles is not None:
        x = _cuda_f32(triangles, 'triangles')
        B, F = x.shape[0], x.shape[1]
    else:
        x = _cuda_f32(v_shaped, 'v_shaped')
        B, V = x.shape[0], x.shape[1]
        if not (torch.is_tensor(faces_i32) and faces_i32.is_cuda and faces_i32.dtype == torch.int32):
            raise RuntimeError('faces_i32 must be a CUDA int32 tensor')
        faces_i32 = faces_i32.contiguous()
        F = faces_i32.shape[0]
    if g.shape != (B, 5):
        raise RuntimeError(f'grad_out must be ({B}, 5), got {tuple(g.shape)}')
    dev = x.device
    grad = torch.empty_like(x)
    if B == 0:
        return grad
    with torch.cuda.device(dev):
        if triangles is not None:
            check(lib().shapy_measure_backward_tris(ptr(x), B, F, C.byref(landmarks), ptr(g), ptr(grad),
                                                    stream_ptr()), 'measure_backward')
        else:
            ws = _WS.get('measure_bwd', lib().shapy_measure_backward_workspace_bytes(V, F), dev)
            check(lib().shapy_measure_backward(ptr(x), ptr(faces_i32), B, V, F, C.byref(landmarks), ptr(g), ptr(grad),
                                               ptr(ws), ws.numel(), stream_ptr()), 'measure_backward')
    return grad


def mesh_to_mesh_forward(query_triangles, target_triangles, max_collisions=16, print_timings=False):
    """Drop-in for mesh_mesh_intersect_cuda.mesh_to_mesh_forward (bind.cpp:59-64)."""
    for name, t in (('query_triangles', query_triangles), ('target_triangles', target_triangles)):
        if not (torch.is_tensor(t) and t.is_cuda):
            raise RuntimeError(f'{name} must be a CUDA tensor')
        if not t.is_contiguous():
            raise RuntimeError(f'{name} must be contiguous')
    if query_triangles.dtype != torch.float32 or target_triangles.dtype != torch.float32:
        raise RuntimeError('shapy_b200 mesh_to_mesh_forward supports float32 triangles only')
    B, Q = query_triangles.shape[:2]
    F = target_triangles.shape[1]
    dev = query_triangles.device
    M = int(max_collisions)
    faces = torch.empty(B, Q * M, dtype=torch.int64, device=dev)
    bcs = torch.empty(B, Q * M, 2, 3, dtype=torch.float32, device=dev)
    if B == 0 or Q == 0:
        return [faces, bcs]
    if F == 0:            # nothing to collide with: every slot is "no collision"
        return [faces.fill_(-1), bcs.zero_()]
    with torch.cuda.device(dev):
        nbytes = lib().shapy_mmi_workspace_bytes(B, Q, F)
        ws = _WS.get('mmi', nbytes, dev)
        check(lib().shapy_mmi_forward(ptr(query_triangles), ptr(target_triangles), B, Q, F, M, ptr(faces), ptr(bcs),
                                      ptr(ws), ws.numel(), stream_ptr()), 'mmi_forward')
    return [faces, bcs]


# -------------------------------------------------------------------------------------------- head
def head_forward(feats, W0, b0, W1, b1, W2, b2, mean, num_stages=3):
    feats = _cuda_f32(feats, 'features')
    B, Fd = feats.shape
    P = mean.numel()
    h0, h1 = W0.shape[0], W1.shape[0]
    out = torch.empty(num_stages, B, P, dtype=torch.float32, device=feats.device)
    ts = [_cuda_f32(t, 'head weight') for t in (W0, b0, W1, b1, W2, b2, mean)]
    if B == 0:
        return out
    with torch.cuda.device(feats.device):
        nbytes = lib().shapy_head_workspace_bytes(B, Fd, P, h0, h1)
        ws = _WS.get('head', nbytes, feats.device)
        check(lib().shapy_head_forward(ptr(feats), B, Fd, P, h0, h1, *[ptr(t) for t in ts], num_stages, ptr(out),
                                       ptr(ws), ws.numel(), stream_ptr()), 'head_forward')
    return out


def collapse_head(W0, b0, W1, b1, W2, b2, feat_dim):
    """Contracts the activation-free 3-layer MLP into (MfT, MpT, c) in fp64 (host, once per weight load)."""
    d = lambda t: t.detach().double().cpu()  # noqa: E731
    W0, b0, W1, b1, W2, b2 = map(d, (W0, b0, W1, b1, W2, b2))
    W21 = W2 @ W1
    Mf = W21 @ W0[:, :feat_dim]
    Mp = W21 @ W0[:, feat_dim:]
    c = W2 @ (W1 @ b0 + b1) + b2
    return Mf.t().contiguous().float(), Mp.t().contiguous().float(), c.float()


def head_forward_collapsed(feats, MfT, Mp, c, mean, num_stages=3):
    feats = _cuda_f32(feats, 'features')
    B, Fd = feats.shape
    P = mean.numel()
    out = torch.empty(num_stages, B, P, dtype=torch.float32, device=feats.device)
    ts = [_cuda_f32(t, 'head matrix') for t in (MfT, Mp, c, mean)]
    if B == 0:
        return out
    with torch.cuda.device(feats.device):
        ws = _WS.get('headc', B * P * 4, feats.device)
        check(lib().shapy_head_forward_collapsed(ptr(feats), B, Fd, P, *[ptr(t) for t in ts], num_stages, ptr(out),
                                                 ptr(ws), ws.numel(), stream_ptr()), 'head_forward_collapsed')
    return out


# ------------------------------------------------------------------------------------------- HRNet
class HrnetPlan:
    """Owns a shapy_hrnet_t built from a conv table + op program (see human_shape/models/backbone/hrnet.py)."""

    def __init__(self, convs, ops, slots, feat_slot, feat_dim, mode, engine, device):
        self.device = torch.device(device)
        self._keep = []
        cd = (_lib.ConvDesc * len(convs))()
        for i, c in enumerate(convs):
            def hp(t):
                if t is None:
                    return None
                a = np.ascontiguousarray(t.detach().float().cpu().numpy())
                self._keep.append(a)
                return a.ctypes.data
            cd[i].cin, cd[i].cout, cd[i].ksize, cd[i].stride = c['cin'], c['cout'], c['ksize'], c['stride']
            cd[i].weight, cd[i].bias = hp(c['weight']), hp(c.get('bias'))
            bn = c.get('bn')
            if bn is not None:
                cd[i].bn_weight, cd[i].bn_bias = hp(bn['weight']), hp(bn['bias'])
                cd[i].bn_mean, cd[i].bn_var = hp(bn['mean']), hp(bn['var'])
                cd[i].bn_eps = float(bn['eps'])
        od = (_lib.Op * len(ops))()
        for i, o in enumerate(ops):
            od[i].kind, od[i].conv = o['kind'], o.get('conv', -1)
            od[i].in_slot, od[i].out_slot, od[i].out_coff = o.get('in_slot', -1), o.get('out_slot', -1), o.get('out_coff', 0)
            od[i].res_slot, od[i].relu = o.get('res_slot', -1), int(o.get('relu', 0))
            od[i].lane = int(o.get('lane', 0))
            ins = o.get('fuse_in', [])
            od[i].n_in = len(ins)
            for k, (s, sh) in enumerate(zip(ins, o.get('fuse_shift', []))):
                od[i].fuse_in[k], od[i].fuse_shift[k] = s, sh
        sd = (_lib.Slot * len(slots))()
        for i, s in enumerate(slots):
            sd[i].channels, sd[i].div = s['channels'], s['div']
        self.slots, self.feat_dim, self.mode, self.engine = slots, feat_dim, mode, engine
        handle = C.c_void_p()
        with torch.cuda.device(self.device):
            check(lib().shapy_hrnet_create(C.byref(handle), cd, len(convs), od, len(ops), sd, len(slots), feat_slot,
                                           mode, engine), 'hrnet_create')
        self._keep = []
        self.handle = handle
        self._fin = weakref.finalize(self, lib().shapy_hrnet_destroy, handle)
        self._ws = None
        self._shape = None

    def forward(self, images: torch.Tensor) -> torch.Tensor:
        images = _cuda_f32(images, 'images')
        B, Cc, H, W = images.shape
        if Cc != 3:
            raise RuntimeError('images must be (B, 3, H, W)')
        feats = torch.empty(B, self.feat_dim, dtype=torch.float32, device=images.device)
        if H % 32 or W % 32 or H == 0 or W == 0:
            raise RuntimeError(f'image size {H}x{W} must be a multiple of 32')
        if B == 0:
            return feats
        with torch.cuda.device(images.device):
            nbytes = lib().shapy_hrnet_workspace_bytes(self.handle, B, H, W)
            if nbytes == 0:
                raise RuntimeError(f'image size {H}x{W} must be a multiple of 32')
            if self._ws is None or self._ws.numel() < nbytes or self._shape != (B, H, W):
                self._ws = torch.empty(nbytes, dtype=torch.uint8, device=images.device)
                self._shape = (B, H, W)
            check(lib().shapy_hrnet_forward(self.handle, ptr(images), B, H, W, ptr(feats), ptr(self._ws),
                                            self._ws.numel(), stream_ptr()), 'hrnet_forward')
        return feats

    def read_slot(self, slot: int) -> torch.Tensor:
        B, H, W = self._shape
        s = self.slots[slot]
        out = torch.empty(B, s['channels'], H // s['div'], W // s['div'], dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(lib().shapy_hrnet_read_slot(self.handle, slot, ptr(out), stream_ptr()), 'hrnet_read_slot')
        return out

    def flops(self, B, H, W) -> float:
        return lib().shapy_hrnet_flops(self.handle, B, H, W)


def conv_test(x_nhwc, weight, bias=None, bn=None, stride=1, res_nhwc=None, relu=False, mode=1, engine=0):
    """Single convolution through either engine on fp32 NHWC tensors (unit tests)."""
    x = _cuda_f32(x_nhwc, 'x')
    B, H, W, Cin = x.shape
    Cout, _, k, _ = weight.shape
    keep = []

    def hp(t):
        if t is None:
            return None
        a = np.ascontiguousarray(t.detach().float().cpu().numpy())
        keep.append(a)
        return a.ctypes.data
    d = _lib.ConvDesc()
    d.cin, d.cout, d.ksize, d.stride = Cin, Cout, k, stride
    d.weight, d.bias = hp(weight), hp(bias)
    if bn is not None:
        d.bn_weight, d.bn_bias, d.bn_mean, d.bn_var = hp(bn['weight']), hp(bn['bias']), hp(bn['mean']), hp(bn['var'])
        d.bn_eps = float(bn['eps'])
    Ho, Wo = (H // 2, W // 2) if stride == 2 else (H, W)
    y = torch.empty(B, Ho, Wo, Cout, dtype=torch.float32, device=x.device)
    res = None if res_nhwc is None else _cuda_f32(res_nhwc, 'res')
    with torch.cuda.device(x.device):
        check(lib().shapy_conv_test(C.byref(d), ptr(x), ptr(res), B, H, W, int(relu), mode, engine, ptr(y),
                                    stream_ptr()), 'conv_test')
    return y
