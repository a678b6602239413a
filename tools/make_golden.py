#!/usr/bin/env python
"""Writes tests/golden/* by running the REFERENCE's own code (build container only).

    python tools/make_golden.py            # needs /root/reference

Everything written here is a small fixture that travels to the GPU box, where
/root/reference does not exist.  Fixtures:

  img00_body.npz        real SHAPY_A output shipped by the reference
                        (samples/shapy_fit_for_virtual_measurements/img_00.npz): v_shaped,
                        faces (int32), raw/decoded poses, camera, joints, proj_joints,
                        golden measurements; plus 3 more real v_shaped bodies from
                        regressor/hbw_evaluation/example_shapy_prediction.npz.
  measurement_landmarks.json   the 5 (face_idx, bc) landmarks BodyMeasurements reads from
                        mesh-mesh-intersection/data/{measurement_defitions,smplx_measurements}.yaml
  ref_smplx.npz         reference lbs()/SMPLX.forward outputs on the seeded synthetic model
  ref_head.npz          reference IterativeRegression + ContinuousRotReprDecoder outputs
  ref_hrnet.npz         reference HighResolutionNet outputs on the seeded synthetic checkpoint
  hrnet_keys.json       the 1 967 state-dict keys/shapes of the reference backbone (sha256 + list)
  ref_measure.json      oracle/measure (quirk-faithful op.cu emulation) results on the 4 real bodies
  b2a.npz               reference Polynomial (B2A head) outputs with seeded male / female weights, routed by gender
  p2p.npz               reference v2vhdError (P2P metric) outputs on seeded sparse point regressors and meshes
  v2v.npz               reference PointError(TranslationAlignment / NoAlignment) outputs (`v2v_t` / `v2v`) on two seeded meshes
  preprocess.npz        reference input stage (transf_utils.crop with cv2 + ToTensor + Normalize) on seeded uint8 images:
                        crop windows, crops with OpenCV's portable path (IPP off) and with this container's IPP build
  ref_smplx_seed5.npz   reference SMPLX.forward on a second seeded batch (every 4th vertex)
  keypoint_tensor.json  the reference KeypointTensor class through the tensor methods of test_keypoint_tensor_cpu.py
  camera.npz            the reference weak_persp_to_blender (demo.py) on seeded targets and camera parameters
  ref_mmi.npz           the reference mesh_to_mesh_forward kernel (oracle/_ref; `python tools/make_golden.py mmi` on a
                        GPU) on the cases of test_gpu_zz_reference_op.py
  measure_grad.npz      gradients of the reference's BodyMeasurements under autograd (its mesh_mesh_intersection module
                        replaced by the C restatement oracle/mmi_oracle.c) on the four bodies of img00_body.npz
"""
import hashlib
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_shim  # noqa: E402

G = os.path.join(ROOT, 'tests', 'golden')
os.makedirs(G, exist_ok=True)
REF = ref_shim.REF


def body_fixture():
    d = ref_shim.load_img00()
    ex = np.load(os.path.join(REF, 'regressor/hbw_evaluation/example_shapy_prediction.npz'))
    np.savez_compressed(
        os.path.join(G, 'img00_body.npz'),
        v_shaped=d['v_shaped'].astype(np.float32), faces=d['faces'].astype(np.int32),
        vertices=d['vertices'].astype(np.float32),
        raw_global_rot=d['raw_global_rot'], global_rot=d['global_rot'],
        raw_body_pose=d['raw_body_pose'], body_pose=d['body_pose'], betas=d['betas'],
        camera=d['camera'], joints=d['joints'], proj_joints=d['proj_joints'],
        meas_names=np.array(['mass', 'height', 'chest', 'waist', 'hips']),
        meas_values=np.array([d['measurements'][k] for k in ['mass', 'height', 'chest', 'waist', 'hips']],
                             dtype=np.float64),
        extra_v_shaped=ex['v_shaped'].astype(np.float32))
    import yaml
    mv = yaml.safe_load(open(os.path.join(REF, 'mesh-mesh-intersection/data/smplx_measurements.yaml')))
    md = yaml.safe_load(open(os.path.join(REF, 'mesh-mesh-intersection/data/measurement_defitions.yaml')))
    lm = {}
    for out_name, src in [('head_top', 'HeadTop'), ('left_heel', 'HeelLeft'), ('chest', md['CW_p'][0]),
                          ('waist', md['BW_p'][0]), ('hips', md['IW_p'][0])]:
        lm[out_name] = dict(name=src, face_idx=int(mv[src]['face_idx']), bc=[float(x) for x in mv[src]['bc']])
    json.dump(lm, open(os.path.join(G, 'measurement_landmarks.json'), 'w'), indent=1)
    print('img00_body.npz, measurement_landmarks.json', lm)


def smplx_fixture():
    from shapy_b200 import synth
    ref = ref_shim.load()
    model = synth.make_smplx()
    g = torch.Generator().manual_seed(11)
    B = 3
    betas = torch.randn(B, 10, generator=g)
    raw = torch.randn(B, 22 * 6, generator=g) * 0.4 + synth.mean_params()[:132]
    dec1, dec21 = ref.pu.ContinuousRotReprDecoder(1), ref.pu.ContinuousRotReprDecoder(21)
    with torch.no_grad():
        grot = dec1(raw[:, :6].contiguous())
        bpose = dec21(raw[:, 6:].contiguous())
        out = ref_shim.smplx_forward_ref(model, betas, grot, bpose)
        # config 1: T-pose, B=1
        eye = torch.eye(3).view(1, 1, 3, 3)
        out_t = ref_shim.smplx_forward_ref(model, betas[:1], eye.clone(), eye.expand(1, 21, -1, -1).contiguous())
        # large head rotation to exercise the dynamic-contour LUT on both sides
        raw2 = raw.clone()
        aa = torch.tensor([[0.0, 0.9, 0.0], [0.0, -1.2, 0.1], [0.2, 0.3, 0.0]])
        R = ref.rot.batch_rodrigues(aa)
        # neck joint 12 sits at body_pose index 11 -> flat offset 6 + 11 * 6
        raw2[:, 6 + 11 * 6: 6 + 12 * 6] = R[:, :, :2].reshape(B, 6)
        grot2, bpose2 = dec1(raw2[:, :6].contiguous()), dec21(raw2[:, 6:].contiguous())
        out2 = ref_shim.smplx_forward_ref(model, betas, grot2, bpose2)
    np.savez_compressed(
        os.path.join(G, 'ref_smplx.npz'), betas=betas.numpy(), raw=raw.numpy(), global_rot=grot.numpy(),
        body_pose=bpose.numpy(), vertices=out['vertices'].numpy(), joints=out['joints'].numpy(),
        v_shaped=out['v_shaped'].numpy(), t_vertices=out_t['vertices'].numpy(), t_joints=out_t['joints'].numpy(),
        raw2=raw2.numpy(), joints2=out2['joints'].numpy(), vertices2_sub=out2['vertices'][:, ::97].numpy())
    print('ref_smplx.npz', out['vertices'].shape, out['joints'].shape)


def head_fixture():
    from shapy_b200 import synth
    ref = ref_shim.load()
    mlp = ref.net.MLP(2048 + 145, 145, layers=[1024, 1024], activation={'type': 'none'},
                      normalization={'type': 'none'}, dropout=0.5, gain=0.01)
    it = ref.net.IterativeRegression(mlp, synth.mean_params().view(1, -1), num_stages=3).eval()
    sd = synth.make_head_state_dict()
    it.load_state_dict({k[len('regressor.'):]: v for k, v in sd.items()})
    g = torch.Generator().manual_seed(12)
    feats = torch.randn(5, 2048, generator=g).abs() * 0.5
    with torch.no_grad():
        params, _ = it(feats)
    np.savez_compressed(os.path.join(G, 'ref_head.npz'), feats=feats.numpy(),
                        params=np.stack([p.numpy() for p in params]))
    print('ref_head.npz', params[-1].shape)


def hrnet_fixture():
    from shapy_b200 import synth
    m = ref_shim.build_hrnet()
    sd0 = m.state_dict()
    keys = [[k, list(v.shape)] for k, v in sd0.items()]
    digest = hashlib.sha256('\n'.join(f'{k} {s}' for k, s in keys).encode()).hexdigest()
    json.dump(dict(sha256=digest, n=len(keys), keys=keys), open(os.path.join(G, 'hrnet_keys.json'), 'w'))
    m.load_state_dict(synth.make_state_dict(sd0, seed=1))
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 3, 224, 224, generator=g)
    with torch.no_grad():
        out = m(x)
        x64 = torch.randn(1, 3, 64, 96, generator=g)
        out64 = m(x64)
    np.savez_compressed(
        os.path.join(G, 'ref_hrnet.npz'), concat=out['concat'].numpy(),
        layer1_sub=out['layer1'][:, ::7, ::5, ::5].numpy(), layer4=out['layer4'][:, ::16].numpy(),
        concat64=out64['concat'].numpy())
    print('ref_hrnet.npz', out['concat'].shape, float(out['concat'].abs().mean()), len(keys), digest[:12])


def preprocess_fixture():
    """Runs the reference's own crop() (regressor/human_shape/utils/transf_utils.py, loaded by path; cv2 is present in the
    build container) followed by the ToTensor / Normalize arithmetic of data/transforms/transforms.py:603-624,710-733."""
    import importlib.util
    import cv2
    import torchvision.transforms.functional as F
    spec = importlib.util.spec_from_file_location('ref_transf_utils', os.path.join(ref_shim.HS, 'utils', 'transf_utils.py'))
    tu = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tu)
    mean, std = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]      # config/datasets_defaults.py:37-38
    rng = np.random.default_rng(20240923)
    out = {'mean': np.float32(mean), 'std': np.float32(std)}
    cases = [  # (H, W, center, scale, size): inside, overhanging every border, strong down- and up-scaling
        (96, 128, (64.0, 48.0), 0.40, 64), (96, 128, (5.5, 90.25), 0.55, 64), (120, 90, (80.0, 10.0), 0.9, 32),
        (70, 70, (35.0, 35.0), 0.12, 64), (150, 200, (100.7, 75.2), 1.35, 32), (64, 48, (24.0, 32.0), 0.32, 64),
    ]
    for i, (H, W, center, scale, size) in enumerate(cases):
        # image-like content: smooth gradients plus noise, uint8
        yy, xx = np.mgrid[0:H, 0:W]
        img = np.stack([(xx * 255.0 / W), (yy * 255.0 / H), ((xx + yy) * 255.0 / (H + W))], -1)
        img = np.clip(img + rng.normal(0, 25, img.shape), 0, 255).astype(np.uint8)
        imgf = np.clip(img.astype(np.float32) / 255.0, 0, 1)                      # read_img, img_utils.py:57-61
        c = np.array(center, dtype=np.float32)
        res = {}
        for tag, ipp in (('portable', False), ('ipp', True)):
            cv2.ipp.setUseIPP(ipp)
            crop = tu.crop(imgf, c, scale, [size, size])
            t = F.to_tensor(crop)
            t = torch.clamp(t, 0, 1)
            res[tag] = F.normalize(t, mean=mean, std=std).numpy()
        cv2.ipp.setUseIPP(True)
        ul = np.array(tu.transform([1, 1], c, scale, [size, size], invert=1)) - 1
        br = np.array(tu.transform([size + 1, size + 1], c, scale, [size, size], invert=1)) - 1
        out[f'img{i}'] = img
        out[f'center{i}'] = c
        out[f'scale{i}'] = np.float64(scale)
        out[f'size{i}'] = np.int64(size)
        out[f'ul{i}'] = ul.astype(np.int64)
        out[f'br{i}'] = br.astype(np.int64)
        out[f'out{i}'] = res['portable']
        out[f'ipp_dev{i}'] = np.float64(np.abs(res['portable'] - res['ipp']).max())   # this container's IPP build vs portable
    out['n'] = np.int64(len(cases))
    np.savez_compressed(os.path.join(G, 'preprocess.npz'), **out)
    print('preprocess.npz', os.path.getsize(os.path.join(G, 'preprocess.npz')), 'bytes; max |portable - ipp| =',
          max(float(out[f'ipp_dev{i}']) for i in range(len(cases))))


def b2a_fixture():
    """Runs the reference's own Polynomial module (attributes/attributes/attributes_betas/polynomial.py, loaded by path behind
    a stub of attributes.utils.typing) with seeded male / female weights, and routes by gender exactly as
    regressor/human_shape/models/common/iterative_regressor.py:761-776 does."""
    import importlib.util
    import types
    from loguru import logger
    logger.remove()
    for name in ('attributes', 'attributes.utils', 'attributes.utils.typing'):
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.__path__ = []
            sys.modules[name] = m
    sys.modules['attributes.utils.typing'].Tensor = torch.Tensor
    sys.modules['attributes.utils.typing'].Array = np.ndarray
    spec = importlib.util.spec_from_file_location(
        'ref_polynomial', os.path.join(REF, 'attributes', 'attributes', 'attributes_betas', 'polynomial.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    torch.manual_seed(31)
    males, females = mod.Polynomial(10, 15, degree=2), mod.Polynomial(10, 15, degree=2)
    for p in (males, females):                      # ratings live in [1, 5]: give the synthetic heads that scale
        with torch.no_grad():
            p.linear.weight.mul_(0.5)
            p.linear.bias.copy_(torch.rand(15) * 4 + 1)
    betas = torch.randn(9, 10) * 1.5
    gender_strs = ['male', 'Female', 'f', '', None, 'M', 'neutral', 'female', 'm']
    genders = np.array([x.lower()[0] if (x is not None and x != '') else 'n' for x in gender_strs])
    gm, gf = np.where(genders == 'm')[0], np.where(genders == 'f')[0]
    with torch.no_grad():
        am, af = males(betas[gm, :]), females(betas[gf, :])
        attributes = torch.zeros(betas.shape[0], am.shape[1])
        attributes[gm, :] = am
        attributes[gf, :] = af
    np.savez_compressed(
        os.path.join(G, 'b2a.npz'), betas=betas.numpy(), genders=np.array([g if g is not None else '<none>' for g in gender_strs]),
        w_male=males.linear.weight.detach().numpy(), b_male=males.linear.bias.detach().numpy(),
        w_female=females.linear.weight.detach().numpy(), b_female=females.linear.bias.detach().numpy(),
        indices_000=males.indices_000.numpy(), indices_001=males.indices_001.numpy(), attributes=attributes.numpy())
    print('b2a.npz', os.path.getsize(os.path.join(G, 'b2a.npz')), 'bytes')


def _load_ref_metrics():
    """The reference's regressor/human_shape/utils/metrics.py loaded by path behind stubs of open3d / .np_utils / .typing."""
    import importlib.util
    import types
    from loguru import logger
    logger.remove()
    if 'ref_hs.utils.metrics' in sys.modules:
        return sys.modules['ref_hs.utils.metrics']
    for name in ('open3d', 'ref_hs', 'ref_hs.utils', 'ref_hs.utils.np_utils', 'ref_hs.utils.typing'):
        m = types.ModuleType(name)
        m.__path__ = []
        sys.modules[name] = m
    sys.modules['ref_hs.utils.np_utils'].np2o3d_pcl = None
    for n in ('Tensor', 'Array', 'IntList'):
        setattr(sys.modules['ref_hs.utils.typing'], n, object)
    spec = importlib.util.spec_from_file_location('ref_hs.utils.metrics', os.path.join(ref_shim.HS, 'utils', 'metrics.py'))
    mod = importlib.util.module_from_spec(spec)
    mod.__package__ = 'ref_hs.utils'
    sys.modules['ref_hs.utils.metrics'] = mod
    spec.loader.exec_module(mod)
    return mod


def v2v_fixture():
    """Runs the reference's own PointError with TranslationAlignment / NoAlignment (metrics.py:232-277, 335-366), i.e. the
    `v2v_t` / `v2v` evaluation metrics (evaluation.py:192-224, 595-602), on two seeded meshes of the same topology."""
    mod = _load_ref_metrics()
    rng = np.random.default_rng(78)
    B, V = 3, 1500
    est = rng.normal(0, 0.4, (B, V, 3)).astype(np.float32)
    gt = (est + rng.normal(0, 0.01, (B, V, 3)) + rng.normal(0, 0.05, (B, 1, 3))).astype(np.float32)
    out = {}
    for tag, name in (('aligned', 'translation'), ('raw', 'none')):
        pe = mod.PointError(mod.build_alignment(name))
        out[f'error_{tag}'] = np.asarray(pe(est.copy(), gt.copy()), np.float64)
    np.savez_compressed(os.path.join(G, 'v2v.npz'), est=est, gt=gt, **out)
    print('v2v.npz', os.path.getsize(os.path.join(G, 'v2v.npz')), 'bytes; mean aligned error', out['error_aligned'].mean())


def p2p_fixture():
    """Runs the reference's own v2vhdError (regressor/human_shape/utils/metrics.py:368-456, loaded by path behind stubs of
    open3d / .np_utils / .typing) on seeded sparse point regressors (3 barycentric weights per point) and meshes, in
    float64 on the CPU as the evaluator does (evaluation.py:258-260)."""
    import pickle
    import tempfile
    import scipy.sparse as sp
    mod = _load_ref_metrics()
    rng = np.random.default_rng(77)
    P, V1, V2, B = 700, 400, 250, 3

    def regressor(V):
        cols = rng.integers(0, V, (P, 3))
        w = rng.dirichlet([1, 1, 1], P)
        # float32-representable weights stored as float64, the dtype of the reference's regressor pickles (the evaluator
        # multiplies them with .double() vertices)
        return sp.csr_matrix((w.reshape(-1).astype(np.float32).astype(np.float64), (np.repeat(np.arange(P), 3), cols.reshape(-1))),
                             shape=(P, V))
    r_in, r_tg = regressor(V1), regressor(V2)
    r_in.sum_duplicates()
    r_tg.sum_duplicates()
    tmp = tempfile.mkdtemp()
    paths = []
    for name, r in (('in', r_in), ('tg', r_tg)):
        paths.append(os.path.join(tmp, name + '.pkl'))
        with open(paths[-1], 'wb') as f:
            pickle.dump(r, f)
    v_in = (rng.normal(0, 0.3, (B, V1, 3)) + [0.1, -0.2, 0.05]).astype(np.float32)
    v_tg = (rng.normal(0, 0.3, (B, V2, 3)) + [-0.3, 0.4, 0.0]).astype(np.float32)
    out = {}
    for align in (True, False):
        metric = mod.v2vhdError(paths[0], paths[1], align=align)
        if align:
            mean, err = metric(torch.from_numpy(v_in).double(), torch.from_numpy(v_tg).double())
        else:       # metrics.py:449-452 only defines t under `if self.align`: the unaligned variant is the same formula with t = 0
            a = metric.sparse_batch_mm(metric.input_point_regressor.double(), torch.from_numpy(v_in).double())
            c = metric.sparse_batch_mm(metric.target_point_regressor.double(), torch.from_numpy(v_tg).double())
            err = torch.sqrt(torch.pow(a - c, 2).sum(axis=-1))
            mean = err.mean(1)
        out['mean_aligned' if align else 'mean_raw'] = mean.numpy()
        out['error_aligned' if align else 'error_raw'] = err.numpy()
    for name, r in (('in', r_in), ('tg', r_tg)):
        out[f'{name}_row_ptr'], out[f'{name}_col'], out[f'{name}_val'] = (r.indptr.astype(np.int32), r.indices.astype(np.int32),
                                                                             r.data.astype(np.float32))
    np.savez_compressed(os.path.join(G, 'p2p.npz'), v_in=v_in, v_tg=v_tg, **out)
    print('p2p.npz', os.path.getsize(os.path.join(G, 'p2p.npz')), 'bytes; mean aligned error', out['mean_aligned'])


def _test_module(name):
    """tests/<name>.py, whose inputs and helpers the fixtures below share."""
    import importlib.util
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, 'tests', name + '.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def smplx_seed5_fixture():
    """ref_shim.smplx_forward_ref on the seed-5 batch of test_oracle_pins.py, the rotations decoded by the oracle's
    decode_6d as the test does; vertices and v_shaped at every 4th vertex (the file stays small)."""
    from oracle import smplx_oracle
    from shapy_b200 import synth
    model = synth.make_smplx()
    g = torch.Generator().manual_seed(5)
    betas = torch.randn(2, 10, generator=g)
    raw = torch.randn(2, 132, generator=g) * 0.3 + synth.mean_params()[:132]
    grot, bpose = smplx_oracle.decode_6d(raw[:, :6]), smplx_oracle.decode_6d(raw[:, 6:])
    ref = ref_shim.smplx_forward_ref(model, betas, grot, bpose)
    np.savez_compressed(os.path.join(G, 'ref_smplx_seed5.npz'), betas=betas.numpy(), raw=raw.numpy(),
                        vertices_sub=ref['vertices'][:, ::4].numpy(), joints=ref['joints'].numpy(),
                        v_shaped_sub=ref['v_shaped'][:, ::4].numpy())
    print('ref_smplx_seed5.npz', os.path.getsize(os.path.join(G, 'ref_smplx_seed5.npz')), 'bytes')


def keypoint_fixture():
    """Runs the reference's own KeypointTensor (regressor/human_shape/models/body_models/utils.py:123-309; the class text
    only, executed from where it lies: the module's other imports are not needed for it) through REFERENCE_OPS of
    test_keypoint_tensor_cpu.py."""
    t = _test_module('test_keypoint_tensor_cpu')
    path = os.path.join(ref_shim.HS, 'models', 'body_models', 'utils.py')
    src = open(path).read()
    start = src.index('class KeypointTensor(object):')
    end = src.index('\nclass ', start + 10) if '\nclass ' in src[start + 10:] else len(src)
    ns = {'torch': torch}
    exec(compile(src[start:end], path, 'exec'), ns)
    k = t.make(ns['KeypointTensor'])
    out = dict(ops=[t.record(f(k)) for f in t.REFERENCE_OPS], index1=k[1].tolist(), index1_type=type(k[1]).__name__,
               numpy=k.numpy().tolist())
    with open(os.path.join(G, 'keypoint_tensor.json'), 'w') as f:
        json.dump(out, f)
    print('keypoint_tensor.json', [r['type'] for r in out['ops']])


def camera_fixture():
    """Runs weak_persp_to_blender of the reference's regressor/demo.py:70-106 (the function text, executed from where it
    lies) on seeded targets and weak-perspective camera parameters."""
    import ast
    from collections import defaultdict
    t = _test_module('test_writer_cpu')
    path = os.path.join(REF, 'regressor', 'demo.py')
    src = open(path).read()
    fn = [n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == 'weak_persp_to_blender'][0]
    ns = {'torch': torch, 'np': np, 'defaultdict': defaultdict}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), path, 'exec'), ns)
    targets = t.make_targets(5, np.random.default_rng(2))
    g = torch.Generator().manual_seed(2)
    scale, transl = torch.rand(5, 1, generator=g) + 0.5, torch.randn(5, 2, generator=g) * 0.1
    ref = ns['weak_persp_to_blender'](targets, scale, transl, H=720, W=1280, sensor_width=36, focal_length=5000)
    np.savez_compressed(
        os.path.join(G, 'camera.npz'), bbox_size=np.array([x.get_field('orig_bbox_size') for x in targets]),
        center=np.stack([x.get_field('orig_center') for x in targets]), scale=scale.numpy(), transl=transl.numpy(),
        keys=np.array(sorted(ref)), **{f'out_{k}': np.asarray(v) for k, v in ref.items()})
    print('camera.npz', sorted(ref))


def mmi_fixture():
    """Runs the reference's own mesh_to_mesh_forward (oracle/_ref, built by oracle/build_ref.py; needs a GPU) in a process
    of its own (oracle/run_ref_mmi.py) on the cases of test_gpu_zz_reference_op.py: the chest-plane queries of the four
    real bodies, and two seeded random triangle soups (~180 colliding pairs, at most 5 per query).  Stores every collision
    slot (face index or -1) and the barycentrics of the filled ones."""
    import subprocess
    import tempfile
    t = _test_module('test_gpu_zz_reference_op')
    rng = np.random.default_rng(11)
    B, Q, F = 2, 96, 400

    def soup(n, spread, size):
        c = rng.uniform(-spread, spread, (B, n, 1, 3))
        return (c + rng.normal(0, size, (B, n, 3, 3))).astype(np.float32)
    soup_query, soup_target = soup(Q, 1.0, 0.15), soup(F, 1.0, 0.15)
    out = dict(soup_query=soup_query, soup_target=soup_target)
    cases = dict(plane=t.plane_queries(G) + (t.PLANE_M,), soup=(soup_query, soup_target, t.SOUP_M))
    with tempfile.TemporaryDirectory() as tmp:
        for tag, (query, target, m) in cases.items():
            inp, outp = os.path.join(tmp, tag + '_in.npz'), os.path.join(tmp, tag + '_out.npz')
            np.savez(inp, query=query, target=target, max_collisions=np.int64(m))
            subprocess.run([sys.executable, os.path.join(ROOT, 'oracle', 'run_ref_mmi.py'), inp, outp], check=True, timeout=600)
            d = np.load(outp)
            faces = d['faces']
            assert faces.shape == (query.shape[0], query.shape[1] * m), faces.shape
            out[f'{tag}_faces'] = faces.astype(np.int32)
            out[f'{tag}_bcs'] = d['bcs'][faces >= 0].astype(np.float32)
            print(tag, 'collisions per batch entry', (faces >= 0).sum(1))
    np.savez_compressed(os.path.join(G, 'ref_mmi.npz'), **out)
    print('ref_mmi.npz', os.path.getsize(os.path.join(G, 'ref_mmi.npz')), 'bytes')



def measure_grad_fixture():
    """The reference's body_measurements.py loaded verbatim, its CUDA collision module replaced by
    oracle.measure_oracle.mesh_to_mesh_forward (the C restatement of op.cu the golden measurements pin), run under
    autograd on the four bodies of img00_body.npz.  Each measurement's gradient with respect to v_shaped is stored
    on its own: mass dense for bodies 0 and 1 (it touches every vertex), height and the circumferences sparse as
    (body, vertex) indices + values.  The mass gradient is the reference's compute_mass differentiated in float64: in
    float32 its autograd loses ~1e-5 of max|grad| to cancellation between the faces around a vertex."""
    import importlib.util
    import types
    from oracle import measure_oracle
    mmi = types.ModuleType('mesh_mesh_intersection')

    class MeshMeshIntersection(torch.nn.Module):
        def __init__(self, max_collisions=16):
            super().__init__()
            self.max_collisions = max_collisions

        def forward(self, query, target):
            f, b = measure_oracle.mesh_to_mesh_forward(query.detach().numpy(), target.detach().numpy(),
                                                       self.max_collisions)
            return torch.from_numpy(f), torch.from_numpy(b)
    mmi.MeshMeshIntersection = MeshMeshIntersection
    saved = sys.modules.get('mesh_mesh_intersection')
    sys.modules['mesh_mesh_intersection'] = mmi
    try:
        R = os.path.join(REF, 'mesh-mesh-intersection')
        spec = importlib.util.spec_from_file_location('ref_body_measurements',
                                                      os.path.join(R, 'body_measurements', 'body_measurements.py'))
        bm = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(bm)
        module = bm.BodyMeasurements({'meas_definition_path': os.path.join(R, 'data', 'measurement_defitions.yaml'),
                                      'meas_vertices_path': os.path.join(R, 'data', 'smplx_measurements.yaml')})
    finally:
        if saved is None:
            sys.modules.pop('mesh_mesh_intersection', None)
        else:
            sys.modules['mesh_mesh_intersection'] = saved
    g = np.load(os.path.join(G, 'img00_body.npz'))
    bodies = np.concatenate([g['v_shaped'][None], g['extra_v_shaped']], 0).astype(np.float32)
    faces = torch.from_numpy(g['faces'].astype(np.int64))
    out = dict(values=np.zeros((len(bodies), 5), np.float32))
    names = ('mass', 'height', 'chest', 'waist', 'hips')
    sparse = {n: ([], [], []) for n in names[1:]}
    mass = []
    for b, v in enumerate(bodies):
        vs = torch.from_numpy(v)[None].requires_grad_(True)
        meas = module(vs[:, faces])['measurements']
        for i, n in enumerate(names):
            val = meas[n]['tensor']
            out['values'][b, i] = float(val[0].detach())
            grad, = torch.autograd.grad(val.sum(), vs, retain_graph=i < 4)
            grad = grad[0].numpy()
            if n == 'mass':
                if b < 2:
                    v64 = torch.from_numpy(v).double()[None].requires_grad_(True)
                    mass.append(torch.autograd.grad(module.compute_mass(v64[:, faces]).sum(), v64)[0][0].numpy())
                continue
            idx = np.where(np.abs(grad).sum(-1) > 0)[0]
            sparse[n][0].append(np.full(len(idx), b, np.int32))
            sparse[n][1].append(idx.astype(np.int32))
            sparse[n][2].append(grad[idx].astype(np.float32))
        print('body', b, dict(zip(names, out['values'][b])))
    out['mass_grad'] = np.stack(mass).astype(np.float32)
    for n, (bb, idx, val) in sparse.items():
        out[f'{n}_body'], out[f'{n}_vertex'], out[f'{n}_grad'] = map(np.concatenate, (bb, idx, val))
        print(n, 'non-zero vertices per body', np.bincount(out[f'{n}_body'], minlength=len(bodies)))
    np.savez_compressed(os.path.join(G, 'measure_grad.npz'), **out)
    print('measure_grad.npz', os.path.getsize(os.path.join(G, 'measure_grad.npz')), 'bytes')


if __name__ == '__main__':
    which = sys.argv[1:] or ['body', 'smplx', 'head', 'hrnet', 'preprocess', 'b2a', 'p2p', 'v2v', 'smplx_seed5', 'keypoint',
                             'camera']
    torch.set_num_threads(8)
    if 'body' in which:
        body_fixture()
    if 'smplx' in which:
        smplx_fixture()
    if 'head' in which:
        head_fixture()
    if 'hrnet' in which:
        hrnet_fixture()
    if 'preprocess' in which:
        preprocess_fixture()
    if 'b2a' in which:
        b2a_fixture()
    if 'p2p' in which:
        p2p_fixture()
    if 'v2v' in which:
        v2v_fixture()
    if 'smplx_seed5' in which:
        smplx_seed5_fixture()
    if 'keypoint' in which:
        keypoint_fixture()
    if 'camera' in which:
        camera_fixture()
    if 'mmi' in which:
        mmi_fixture()
    if 'measure_grad' in which:
        measure_grad_fixture()
