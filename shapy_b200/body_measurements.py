"""BodyMeasurements, host mirror of mesh-mesh-intersection/body_measurements/body_measurements.py:17-246.

Same constructor (a cfg with `meas_definition_path` / `meas_vertices_path` / `max_collisions`), same
registered buffers (left_heel_bc, head_top_bc, chest_bcs, belly_bcs, hips_bcs) and the same output
structure {'measurements': {name: {'tensor': (B,)}}}.  The reference runs, per body and per measurement,
a BVH build + 2-thread traversal on the GPU and scipy's ConvexHull on the CPU; here all five values of all
bodies come from ONE kernel launch (csrc/measure.cu) with the reference's exact point-selection rule.
"""
import os.path as osp

import torch
import torch.nn as nn
from torch.autograd.function import once_differentiable

from . import ops as _ops


class _Measure(torch.autograd.Function):
    """(B, 5) measurements of `x` = v_shaped (with faces_i32) or triangles, differentiable once in `x`."""

    @staticmethod
    def forward(ctx, x, faces_i32, landmarks):
        if faces_i32 is None:
            out = _ops.measure(landmarks, triangles=x)
        else:
            out = _ops.measure(landmarks, v_shaped=x, faces_i32=faces_i32)
        ctx.landmarks = landmarks
        ctx.save_for_backward(x, faces_i32)
        ctx.mark_non_differentiable(out.status)
        return out, out.status

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out, _grad_status):
        x, faces_i32 = ctx.saved_tensors
        if faces_i32 is None:
            return _ops.measure_backward(ctx.landmarks, grad_out, triangles=x), None, None
        return _ops.measure_backward(ctx.landmarks, grad_out, v_shaped=x, faces_i32=faces_i32), None, None


def _measure(landmarks, x, faces_i32=None):
    if torch.is_grad_enabled() and x.requires_grad:
        out, status = _Measure.apply(x, faces_i32, landmarks)
        out.status = status
        return out
    if faces_i32 is None:
        return _ops.measure(landmarks, triangles=x)
    return _ops.measure(landmarks, v_shaped=x, faces_i32=faces_i32)


class BodyMeasurements(nn.Module):
    DENSITY = 985

    def __init__(self, cfg, **kwargs):
        super().__init__()
        lm = cfg.get('landmarks', None)
        if lm is None:
            import yaml
            with open(osp.expanduser(osp.expandvars(cfg.get('meas_definition_path', ''))), 'r') as f:
                defs = yaml.safe_load(f)
            with open(osp.expanduser(osp.expandvars(cfg.get('meas_vertices_path', ''))), 'r') as f:
                mv = yaml.safe_load(f)
            lm = {'head_top': mv['HeadTop'], 'left_heel': mv['HeelLeft'], 'chest': mv[defs['CW_p'][0]],
                  'waist': mv[defs['BW_p'][0]], 'hips': mv[defs['IW_p'][0]]}
        self.left_heel_face_idx = lm['left_heel']['face_idx']
        self.head_top_face_idx = lm['head_top']['face_idx']
        self.chest_face_index = lm['chest']['face_idx']
        self.belly_face_index = lm['waist']['face_idx']
        self.hips_face_index = lm['hips']['face_idx']
        self.register_buffer('left_heel_bc', torch.tensor(lm['left_heel']['bc'], dtype=torch.float32))
        self.register_buffer('head_top_bc', torch.tensor(lm['head_top']['bc'], dtype=torch.float32))
        self.register_buffer('chest_bcs', torch.tensor(lm['chest']['bc'], dtype=torch.float32))
        self.register_buffer('belly_bcs', torch.tensor(lm['waist']['bc'], dtype=torch.float32))
        self.register_buffer('hips_bcs', torch.tensor(lm['hips']['bc'], dtype=torch.float32))
        # accepted for config compatibility; the fused kernel has its own fixed capacity (1024 points per plane,
        # 4x the reference default) and reports overflow through NaN + `last_status` instead of truncating
        self.max_collisions = cfg.get('max_collisions', 256)
        self.last_status = None
        self._lm = None

    def extra_repr(self):
        return f'Human Body Density: {self.DENSITY}'

    def _landmarks(self):
        # rebuilt from the buffers so that a loaded checkpoint's barycentrics are honoured
        lm = {'head_top': dict(face_idx=self.head_top_face_idx, bc=self.head_top_bc.tolist()),
              'left_heel': dict(face_idx=self.left_heel_face_idx, bc=self.left_heel_bc.tolist()),
              'chest': dict(face_idx=self.chest_face_index, bc=self.chest_bcs.tolist()),
              'waist': dict(face_idx=self.belly_face_index, bc=self.belly_bcs.tolist()),
              'hips': dict(face_idx=self.hips_face_index, bc=self.hips_bcs.tolist())}
        return _ops.make_landmarks(lm)

    def landmarks(self):
        if self._lm is None:
            self._lm = self._landmarks()
        return self._lm

    def _load_from_state_dict(self, *args, **kwargs):
        self._lm = None
        return super()._load_from_state_dict(*args, **kwargs)

    def _pack(self, out):
        names = ('mass', 'height', 'chest', 'waist', 'hips')
        # device status word of the launch (non-zero: some body overflowed the kernel's fixed point capacity and its
        # circumferences are NaN); kept for callers that want to check it at their next synchronisation point
        self.last_status = getattr(out, 'status', None)
        return {'measurements': {n: {'tensor': out[:, i]} for i, n in enumerate(names)}}

    def check_status(self):
        """Raises if the last launch overflowed the kernel's point buffers (one host synchronisation)."""
        st = getattr(self, 'last_status', None)
        if st is not None and int(st.item()) != 0:
            raise RuntimeError('BodyMeasurements: intersection-point capacity exceeded; affected values are NaN')

    def forward_vertices(self, v_shaped, faces_i32):
        """Fast path: (B, V, 3) vertices + (F, 3) int32 faces; no (B, F, 3, 3) tensor is materialised.
        Differentiable once in v_shaped when grad mode is on and it requires grad (see ops.measure_backward)."""
        return self._pack(_measure(self.landmarks(), v_shaped, faces_i32))

    def forward(self, triangles, compute_mass=True, compute_height=True, compute_chest=True, compute_waist=True,
                compute_hips=True, **kwargs):
        """triangles: (B, F, 3, 3), as in the reference; differentiable once in triangles when grad mode is on and
        they require grad.  A measurement turned off by its compute_* flag receives no gradient."""
        out = self._pack(_measure(self.landmarks(), triangles))
        drop = [n for n, f in (('mass', compute_mass), ('height', compute_height), ('chest', compute_chest),
                               ('waist', compute_waist), ('hips', compute_hips)) if not f]
        for n in drop:
            out['measurements'].pop(n)
        return out
