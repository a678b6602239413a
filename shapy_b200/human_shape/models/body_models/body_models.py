"""SMPL-X body model, host mirror of regressor/human_shape/models/body_models/body_models.py
(SMPL.__init__ 73-203, SMPLX.__init__ 535-597, SMPLX.forward 628-767, forward_shape 292-302).

Same buffer names (v_template, shapedirs, posedirs, J_regressor, lbs_weights, parents, faces_tensor,
expr_dirs, lmk_*, dynamic_lmk_*, neck_kin_chain, extra_joint_regressor, source_idxs, target_idxs,
head_vertices_ids) so `model.*` checkpoint entries load; the buffers are the source of truth and the
packed device-side model (shapy_smplx_create) is rebuilt lazily after load_state_dict / .to() / deepcopy.
The forward pass is three launches of csrc/smplx.cu; there is no PyTorch fallback.
"""
import os.path as osp
import pickle
from collections import defaultdict

import numpy as np
import torch
import torch.nn as nn
from torch.autograd.function import once_differentiable

from .... import ops as _ops
from .utils import KeypointTensor, find_joint_kin_chain, to_tensor

J14_NAMES = ['right_ankle', 'right_knee', 'right_hip', 'left_hip', 'left_knee', 'left_ankle', 'right_wrist',
             'right_elbow', 'right_shoulder', 'left_shoulder', 'left_elbow', 'left_wrist', 'neck', 'head']


def _to_np(array, dtype=np.float32):
    if 'scipy.sparse' in str(type(array)):
        array = array.todense()
    if torch.is_tensor(array):
        array = array.detach().cpu().numpy()
    return np.array(array, dtype=dtype)


# The 22 body joints of the public SMPL / SMPL-X kinematic tree, in model order.  Pure data (the reference lists the same
# names first in human_shape/data/utils/keypoint_names.py, SMPLX_KEYPOINT_NAMES = SMPL_KEYPOINT_NAMES[:-2] + ...); the
# J14 overwrite (body_models.py:184-197) finds its 14 names among exactly these.
SMPLX_BODY_JOINT_NAMES = [
    'pelvis', 'left_hip', 'right_hip', 'spine1', 'left_knee', 'right_knee', 'spine2', 'left_ankle', 'right_ankle',
    'spine3', 'left_foot', 'right_foot', 'neck', 'left_collar', 'right_collar', 'head', 'left_shoulder',
    'right_shoulder', 'left_elbow', 'right_elbow', 'left_wrist', 'right_wrist']


def _keypoint_names(num):
    """SMPL-X keypoint names: the reference's own table (human_shape.data.utils, pure data) when that package is
    importable; otherwise the 22 public body-joint names followed by positional labels (the remaining names only
    label the output; the J14 overwrite needs the body joints)."""
    try:  # pragma: no cover - only inside the reference environment
        from human_shape.data.utils import KEYPOINT_NAMES_DICT
        names = list(KEYPOINT_NAMES_DICT['smplx'])
        if len(names) >= num:
            return names
    except Exception:
        pass
    names = list(SMPLX_BODY_JOINT_NAMES)
    return (names + [f'keypoint_{i:03d}' for i in range(len(names), num)])[:max(num, 0)]


class _ShapeBlend(torch.autograd.Function):
    @staticmethod
    def forward(ctx, betas, model):
        ctx.model = model
        return _ops.smplx_forward_shape(model, betas)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_v_shaped):
        return _ops.smplx_shape_backward(ctx.model, grad_v_shaped), None


class SMPLX(nn.Module):
    NUM_BODY_JOINTS = 21
    NUM_HAND_JOINTS = 15
    NUM_FACE_JOINTS = 3
    NUM_JOINTS = NUM_BODY_JOINTS + 2 * NUM_HAND_JOINTS + NUM_FACE_JOINTS
    SHAPE_SPACE_DIM = 300
    EXPRESSION_SPACE_DIM = 100
    NECK_IDX = 12
    HEAD_IDX = 15
    NAME = 'smplx'

    def __init__(self, model_folder='', is_training=False, expression=None, use_face_contour=False,
                 gender='neutral', dtype=torch.float32, ext='npz', data_struct=None, betas=None,
                 j14_regressor_path='', head_verts_ids_path='', **kwargs):
        super().__init__()
        self.gender, self.dtype, self.use_face_contour = gender, dtype, use_face_contour
        betas = betas if betas is not None else {'num': 10}
        expression = expression if expression is not None else {'num': 10}
        self._num_betas = betas.get('num', 10)
        self._num_expression_coeffs = expression.get('num', 10)
        if data_struct is None:
            path = osp.join(osp.expandvars(model_folder), f'SMPLX_{gender.upper()}.{ext}')
            if ext == 'npz':
                data_struct = dict(np.load(path, allow_pickle=True))
            else:
                with open(path, 'rb') as f:
                    data_struct = pickle.load(f, encoding='latin1')
        ds = data_struct
        if 'faces_tensor' in ds:      # already in buffer form (e.g. shapy_b200.synth.make_smplx)
            bufs = {k: (v.clone() if torch.is_tensor(v) else v) for k, v in ds.items()}
        else:                          # raw SMPL-X model file, as read by the reference (112-166, 563-597)
            nb, ne = self._num_betas, self._num_expression_coeffs
            shapedirs = _to_np(ds['shapedirs'])
            parents = torch.from_numpy(_to_np(ds['kintree_table'][0], np.int64)).long()
            parents[0] = -1
            npose = ds['posedirs'].shape[-1]
            bufs = dict(
                faces_tensor=torch.from_numpy(_to_np(ds['f'], np.int64)),
                v_template=to_tensor(_to_np(ds['v_template']), dtype),
                shapedirs=to_tensor(shapedirs[:, :, :nb], dtype),
                expr_dirs=to_tensor(shapedirs[:, :, self.SHAPE_SPACE_DIM:self.SHAPE_SPACE_DIM + ne], dtype),
                J_regressor=to_tensor(_to_np(ds['J_regressor']), dtype),
                posedirs=to_tensor(np.reshape(_to_np(ds['posedirs']), [-1, npose]).T, dtype),
                parents=parents, lbs_weights=to_tensor(_to_np(ds['weights']), dtype),
                lmk_faces_idx=torch.from_numpy(_to_np(ds['lmk_faces_idx'], np.int64)),
                lmk_bary_coords=to_tensor(_to_np(ds['lmk_bary_coords']), dtype),
                dynamic_lmk_faces_idx=torch.from_numpy(_to_np(ds['dynamic_lmk_faces_idx'], np.int64)),
                dynamic_lmk_bary_coords=to_tensor(_to_np(ds['dynamic_lmk_bary_coords']), dtype))
        self.faces = bufs['faces_tensor'].cpu().numpy().astype(np.int64)
        for name in ('faces_tensor', 'v_template', 'shapedirs', 'J_regressor', 'posedirs', 'parents', 'lbs_weights',
                     'lmk_faces_idx', 'lmk_bary_coords', 'dynamic_lmk_faces_idx', 'dynamic_lmk_bary_coords',
                     'expr_dirs'):
            self.register_buffer(name, bufs[name])
        hv = bufs.get('head_vertices_ids')
        head_verts_ids_path = osp.expandvars(head_verts_ids_path or '')
        if hv is None:
            hv = torch.tensor(np.load(head_verts_ids_path) if osp.exists(head_verts_ids_path) else [],
                              dtype=torch.long)
        self.register_buffer('head_vertices_ids', hv)
        kin = bufs.get('neck_kin_chain')
        if kin is None:
            kin = torch.tensor(find_joint_kin_chain(self.HEAD_IDX, self.parents.tolist()), dtype=torch.long)
        self.register_buffer('neck_kin_chain', kin)
        n_kp = self.NUM_JOINTS + 1 + self.lmk_faces_idx.shape[0] + (
            self.dynamic_lmk_faces_idx.shape[1] if use_face_contour else 0)
        self._keypoint_names = _keypoint_names(n_kp)[:n_kp]
        # J14 regressor (SMPL.__init__ 170-202)
        self.use_joint_regressor = False
        if 'extra_joint_regressor' in bufs:
            self.use_joint_regressor = True
            self.register_buffer('source_idxs', bufs['source_idxs'])
            self.register_buffer('target_idxs', bufs['target_idxs'])
            self.register_buffer('extra_joint_regressor', bufs['extra_joint_regressor'].to(torch.float32))
        else:
            j14_regressor_path = osp.expandvars(j14_regressor_path or '')
            if osp.exists(j14_regressor_path):
                if j14_regressor_path.endswith('.pkl'):
                    with open(j14_regressor_path, 'rb') as f:
                        j14 = pickle.load(f, encoding='latin1')
                else:
                    j14 = np.load(j14_regressor_path)
                source, target = [], []
                for idx, name in enumerate(self._keypoint_names):
                    if name in J14_NAMES:
                        source.append(idx)
                        target.append(J14_NAMES.index(name))
                if len(source) != len(J14_NAMES):
                    raise ValueError(f'J14 regressor: only {len(source)} of the {len(J14_NAMES)} joint names were found '
                                     'among the model\'s keypoint names; refusing to skip the overwrite silently')
                self.use_joint_regressor = True
                self.register_buffer('source_idxs', torch.from_numpy(np.asarray(source, dtype=np.int64)))
                self.register_buffer('target_idxs', torch.from_numpy(np.asarray(target, dtype=np.int64)))
                self.register_buffer('extra_joint_regressor', torch.from_numpy(np.asarray(j14)).to(torch.float32))
        self._packed = None

    # ------------------------------------------------------------------ metadata
    name = property(lambda self: self.NAME)
    num_betas = property(lambda self: self._num_betas)
    num_expression_coeffs = property(lambda self: self._num_expression_coeffs)
    num_body_joints = property(lambda self: self.NUM_BODY_JOINTS)
    num_hand_joints = property(lambda self: self.NUM_HAND_JOINTS)
    keypoint_names = property(lambda self: self._keypoint_names)
    parts = property(lambda self: None)
    connections = property(lambda self: None)
    part_connections = property(lambda self: None)

    def get_num_verts(self):
        return self.v_template.shape[0]

    def get_num_faces(self):
        return self.faces.shape[0]

    def get_head_vertices_ids(self):
        return self.head_vertices_ids

    # ------------------------------------------------------------------ packed device model
    def invalidate(self):
        self._packed = None

    def _apply(self, fn, *args, **kwargs):
        self.invalidate()
        return super()._apply(fn, *args, **kwargs)

    def _load_from_state_dict(self, *args, **kwargs):
        self.invalidate()
        return super()._load_from_state_dict(*args, **kwargs)

    def __deepcopy__(self, memo):
        import copy
        packed, self._packed = self._packed, None
        try:
            new = self.__class__.__new__(self.__class__)
            memo[id(self)] = new
            for k, v in self.__dict__.items():
                new.__dict__[k] = copy.deepcopy(v, memo)
        finally:
            self._packed = packed
        return new

    def packed(self, device=None) -> _ops.SmplxModel:
        device = torch.device(device) if device is not None else self.v_template.device
        if self._packed is None or self._packed.device != device:
            t = {k: v for k, v in self.named_buffers()}
            t['use_face_contour'] = self.use_face_contour
            if not self.use_joint_regressor:
                t.pop('extra_joint_regressor', None)
            self._packed = _ops.SmplxModel(t, device)
        return self._packed

    @property
    def faces_i32(self):
        if getattr(self, '_faces_i32', None) is None or self._faces_i32.device != self.faces_tensor.device:
            self._faces_i32 = self.faces_tensor.to(torch.int32).contiguous()
        return self._faces_i32

    # ------------------------------------------------------------------ forward
    def forward_shape(self, betas=None):
        """v_shaped = v_template + shapedirs . betas; differentiable once in betas when grad mode is on and betas
        require grad."""
        model = self.packed(betas.device)
        if torch.is_grad_enabled() and betas.requires_grad:
            v_shaped = _ShapeBlend.apply(betas, model)
        else:
            v_shaped = _ops.smplx_forward_shape(model, betas)
        return {'vertices': v_shaped, 'betas': betas, 'v_shaped': v_shaped}

    def forward(self, global_rot=None, body_pose=None, left_hand_pose=None, right_hand_pose=None, jaw_pose=None,
                betas=None, expression=None, transl=None, leye_pose=None, reye_pose=None, get_skin=True,
                return_full_pose=False, return_shaped=True, camera=None, **kwargs):
        device = self.shapedirs.device
        bs = 1
        for v in (betas, global_rot, body_pose, transl, left_hand_pose, right_hand_pose, jaw_pose, leye_pose,
                  reye_pose, expression):
            if v is not None:
                bs = max(bs, len(v))
        eye = torch.eye(3, device=device, dtype=torch.float32).view(1, 1, 3, 3)
        if global_rot is None:
            global_rot = eye.expand(bs, 1, -1, -1)
        if body_pose is None:
            body_pose = eye.expand(bs, 21, -1, -1)
        if betas is None:
            betas = torch.zeros(bs, self.num_betas, dtype=torch.float32, device=device)
        parts = [global_rot.reshape(bs, -1, 3, 3), body_pose.reshape(bs, -1, 3, 3)]
        extra = [(jaw_pose, 1), (leye_pose, 1), (reye_pose, 1), (left_hand_pose, 15), (right_hand_pose, 15)]
        # trailing identity joints are never materialised: the kernel skips their (exactly zero) pose-feature rows
        last = max([i for i, (p, _) in enumerate(extra) if p is not None], default=-1)
        for i, (p, n) in enumerate(extra[:last + 1]):
            parts.append(p.reshape(bs, n, 3, 3) if p is not None else eye.expand(bs, n, -1, -1))
        rot = torch.cat([p.to(torch.float32) for p in parts], dim=1).contiguous()
        out = _ops.smplx_forward(self.packed(device), betas, rot, expr=expression, camera=camera,
                                 want_vertices=True, want_v_shaped=return_shaped, want_joints=True)
        vertices, joints = out['vertices'], out['joints']
        if transl is not None:
            joints += transl.unsqueeze(dim=1)
            vertices += transl.unsqueeze(dim=1)
        output = defaultdict(lambda: None,
                             joints=KeypointTensor(joints, source=self.name, keypoint_names=self.keypoint_names),
                             faces=self.faces)
        if get_skin:
            output['vertices'] = vertices
        if return_full_pose:
            full = torch.cat([rot, eye.expand(bs, self.NUM_JOINTS + 1 - rot.shape[1], -1, -1)], dim=1)
            output['full_pose'] = full
        if return_shaped:
            output['v_shaped'] = out['v_shaped']
        if out['proj_joints'] is not None:
            output['proj_joints'] = out['proj_joints']
        return output


def build_body_model(body_model_cfg, **kwargs):
    """Mirror of regressor/human_shape/models/body_models/build.py:10-29 (smplx only).  A `data_struct`
    entry inside the `smplx` node supplies the model tensors directly (synthetic models in tests)."""
    model_type = body_model_cfg.get('type', 'smplx')
    if model_type.lower() != 'smplx':
        raise ValueError(f'shapy_b200 implements the smplx body model only, got: {model_type}')
    model_folder = osp.expandvars(body_model_cfg.get('model_folder', 'data/models') or '')
    cur = body_model_cfg.get(model_type, {}) or {}
    allowed = ('betas', 'expression', 'j14_regressor_path', 'use_face_contour', 'head_verts_ids_path',
               'data_struct', 'ext', 'gender')
    sub = {k: cur.get(k) for k in allowed if cur.get(k) is not None}
    return SMPLX(osp.join(model_folder, model_type), **sub, **kwargs)
