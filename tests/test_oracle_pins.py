"""Pins oracle/* (the CPU restatements) against the reference's golden vectors and against
outputs of the reference's own code (tests/golden/*, written by tools/make_golden.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import measure_oracle, net_oracle, smplx_oracle
from shapy_b200 import synth


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


@pytest.fixture(scope='module')
def body(golden_dir):
    return dict(np.load(os.path.join(golden_dir, 'img00_body.npz')))


def test_decoder_6d_golden(body):
    # img_00.npz: real SHAPY_A output; decoder must map raw_* -> rotation matrices
    r = smplx_oracle.decode_6d(torch.from_numpy(body['raw_body_pose'])[None])[0].numpy()
    assert np.abs(r - body['body_pose']).max() < 5e-7
    r = smplx_oracle.decode_6d(torch.from_numpy(body['raw_global_rot'])[None])[0].numpy()
    assert np.abs(r - body['global_rot']).max() < 5e-7


def test_camera_golden(body):
    pj = smplx_oracle.weak_persp(torch.from_numpy(body['joints'])[None], torch.from_numpy(body['camera'])[None])
    assert np.abs(pj[0].numpy() - body['proj_joints']).max() < 1e-6


def test_measurements_golden(body):
    m = measure_oracle.measure(body['v_shaped'], body['faces'])
    for name, gold in zip(body['meas_names'], body['meas_values']):
        assert abs(m[str(name)] - gold) / gold < 1e-6, (name, m[str(name)], gold)


def test_smplx_oracle_vs_reference_lbs(golden_dir):
    g = np.load(os.path.join(golden_dir, 'ref_smplx.npz'))
    model = synth.make_smplx()
    raw = torch.from_numpy(g['raw'])
    grot, bpose = smplx_oracle.decode_6d(raw[:, :6]), smplx_oracle.decode_6d(raw[:, 6:])
    assert np.abs(grot.numpy() - g['global_rot']).max() < 1e-6
    out = smplx_oracle.smplx_forward(model, torch.from_numpy(g['betas']), grot, bpose)
    assert _rel(out['vertices'].numpy(), g['vertices']) < 2e-6
    assert _rel(out['joints'].numpy(), g['joints']) < 2e-6
    assert _rel(out['v_shaped'].numpy(), g['v_shaped']) < 1e-6
    # config 1: T-pose, B=1
    eye = torch.eye(3).view(1, 1, 3, 3)
    t = smplx_oracle.smplx_forward(model, torch.from_numpy(g['betas'][:1]), eye, eye.expand(1, 21, 3, 3))
    assert _rel(t['vertices'].numpy(), g['t_vertices']) < 2e-6
    assert _rel(t['joints'].numpy(), g['t_joints']) < 2e-6
    # rotated neck: dynamic contour LUT on both sides of zero
    raw2 = torch.from_numpy(g['raw2'])
    o2 = smplx_oracle.smplx_forward(model, torch.from_numpy(g['betas']), smplx_oracle.decode_6d(raw2[:, :6]),
                                    smplx_oracle.decode_6d(raw2[:, 6:]))
    assert _rel(o2['joints'].numpy(), g['joints2']) < 2e-6
    assert _rel(o2['vertices'][:, ::97].numpy(), g['vertices2_sub']) < 2e-6


def test_head_oracle_vs_reference(golden_dir):
    g = np.load(os.path.join(golden_dir, 'ref_head.npz'))
    sd = synth.make_head_state_dict()
    outs = net_oracle.head_forward(sd, torch.from_numpy(g['feats']))
    for k in range(3):
        assert _rel(outs[k].numpy(), g['params'][k]) < 2e-6


def test_hrnet_oracle_vs_reference(golden_dir):
    import json
    g = np.load(os.path.join(golden_dir, 'ref_hrnet.npz'))
    keys = json.load(open(os.path.join(golden_dir, 'hrnet_keys.json')))
    template = {k: (torch.zeros(s, dtype=torch.long) if k.endswith('num_batches_tracked') else torch.zeros(s))
                for k, s in keys['keys']}
    sd = synth.make_state_dict(template, seed=1)
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    x = torch.randn(1, 3, 64, 96, generator=_gen_after_first())
    with torch.no_grad():
        out = net_oracle.hrnet_forward(sd, x)
    assert _rel(out['concat'].numpy(), g['concat64']) < 2e-5


def _gen_after_first():
    # tools/make_golden.py draws the (2,3,224,224) batch first, then the 64x96 image
    gen = torch.Generator().manual_seed(0)
    torch.randn(2, 3, 224, 224, generator=gen)
    return gen


def test_smplx_oracle_vs_live_reference(golden_dir):
    """Against SMPLX.forward of the reference re-assembled on its verbatim lbs.py (oracle/ref_shim.py) on a second seeded
    batch: tests/golden/ref_smplx_seed5.npz (tools/make_golden.py smplx_seed5) stores every 4th vertex."""
    g = np.load(os.path.join(golden_dir, 'ref_smplx_seed5.npz'))
    model = synth.make_smplx()
    betas, raw = torch.from_numpy(g['betas']), torch.from_numpy(g['raw'])
    grot, bpose = smplx_oracle.decode_6d(raw[:, :6]), smplx_oracle.decode_6d(raw[:, 6:])
    out = smplx_oracle.smplx_forward(model, betas, grot, bpose)
    assert _rel(out['vertices'][:, ::4].numpy(), g['vertices_sub']) < 2e-6
    assert _rel(out['joints'].numpy(), g['joints']) < 2e-6
    assert _rel(out['v_shaped'][:, ::4].numpy(), g['v_shaped_sub']) < 2e-6
