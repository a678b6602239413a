"""Output writers (SURVEY.md 8f rank 4): camera conversion against the reference's own function, .npz contents as
demo.py:338-352 builds them, .ply round trip.  Pure host code."""
import os

import numpy as np
import pytest
import torch

from shapy_b200 import writer


class Target:
    def __init__(self, **fields):
        self.fields = fields

    def has_field(self, k):
        return k in self.fields

    def get_field(self, k, default=None):
        return self.fields.get(k, default)


def make_targets(n, rng):
    return [Target(fname=f'img_{i:02d}.jpg', orig_bbox_size=float(rng.uniform(150, 400)),
                   orig_center=np.float32(rng.uniform(100, 500, 2)), filename='' if i % 2 else f'/data/set{i}/seq/img_{i:02d}.jpg')
            for i in range(n)]


def test_camera_conversion_matches_reference_source(golden_dir):
    """The mirror against the outputs of weak_persp_to_blender of the reference's demo.py on the same targets and camera
    parameters (tests/golden/camera.npz, written by tools/make_golden.py camera)."""
    g = np.load(os.path.join(golden_dir, 'camera.npz'))
    targets = [Target(orig_bbox_size=float(s), orig_center=c) for s, c in zip(g['bbox_size'], g['center'])]
    mine = writer.weak_persp_to_blender(targets, torch.from_numpy(g['scale']), torch.from_numpy(g['transl']), H=720, W=1280,
                                        sensor_width=36, focal_length=5000)
    assert sorted(mine) == sorted(g['keys'].tolist())
    for k in mine:
        assert np.array_equal(np.asarray(mine[k]), g[f'out_{k}']), k


def test_ply_round_trip(tmp_path):
    rng = np.random.default_rng(0)
    v = rng.normal(size=(10475, 3)).astype(np.float32)
    f = rng.integers(0, 10475, (20908, 3)).astype(np.int64)
    p = str(tmp_path / 'a.ply')
    writer.write_ply(p, v, f)
    v2, f2 = writer.read_ply(p)
    assert np.array_equal(v, v2) and np.array_equal(f, f2)
    head = open(p, 'rb').read(300).decode('ascii', 'ignore')
    assert head.startswith('ply\nformat binary_little_endian 1.0') and 'property list uchar int vertex_indices' in head


def test_batch_files_like_the_demo(tmp_path):
    rng = np.random.default_rng(1)
    n = 4
    targets = make_targets(n, rng)
    faces = rng.integers(0, 50, (80, 3)).astype(np.int64)
    stage = {'vertices': torch.randn(n, 50, 3), 'betas': torch.randn(n, 10), 'faces': faces,
             'global_rot': torch.randn(n, 1, 3, 3), 'measurements': {'mass': torch.ones(n)}}
    hd = writer.weak_persp_to_blender(targets, torch.rand(n, 1) + 0.5, torch.randn(n, 2) * 0.1, H=480, W=640)
    with writer.ResultWriter(str(tmp_path), workers=3) as w:
        w.submit(targets, stage, hd)
    for i, t in enumerate(targets):
        d = writer.output_dir(str(tmp_path), t)
        assert (d == str(tmp_path)) == (t.get_field('filename') == '')
        z = np.load(os.path.join(d, f'img_{i:02d}.npz'), allow_pickle=True)
        assert str(z['fname']) == f'img_{i:02d}.jpg'
        assert np.array_equal(z['vertices'], stage['vertices'][i].numpy()) and np.array_equal(z['betas'], stage['betas'][i].numpy())
        assert np.array_equal(z['faces'], faces)                                   # non-tensor entries are stored whole
        assert np.allclose(z['transl'], hd['transl'][i]) and float(z['focal_length_in_px']) == 5000
        v, f = writer.read_ply(os.path.join(d, f'img_{i:02d}.ply'))
        assert np.allclose(v, stage['vertices'][i].numpy() + hd['transl'][i].astype(np.float32), atol=1e-6) and np.array_equal(f, faces)


def test_same_output_name_and_numpy_inputs(tmp_path):
    """Two people in one image share `fname`: the jobs must not corrupt each other's temp files and the later one wins (as
    in the reference's sequential loop); numpy arrays with one row per target are stored per image; a mesh without
    topology is refused up front."""
    rng = np.random.default_rng(3)
    targets = [Target(fname='same.jpg', orig_bbox_size=200.0, orig_center=np.float32([10, 20])) for _ in range(6)]
    verts = rng.normal(size=(6, 50, 3)).astype(np.float32)
    faces = rng.integers(0, 50, (30, 3))
    hd = dict(transl=np.zeros((6, 3), np.float32), focal_length_in_px=np.full(6, 1000.0), center=np.zeros((6, 2)),
              focal_length_in_mm=np.full(6, 50.0), sensor_width=np.full(6, 36.0))
    with writer.ResultWriter(str(tmp_path)) as w:
        for _ in range(3):
            w.submit(targets, {'vertices': torch.from_numpy(verts), 'betas': verts[:, 0, :], 'faces': faces}, hd)
    d = np.load(tmp_path / 'same.npz', allow_pickle=True)
    assert d['betas'].shape == (3,) and np.allclose(d['vertices'], verts[5])        # last target wins, row 5
    v, f = writer.read_ply(str(tmp_path / 'same.ply'))
    assert np.allclose(v, verts[5]) and (f == faces).all()
    assert not [p for p in os.listdir(tmp_path) if 'tmp' in p]
    with pytest.raises(ValueError):
        writer.ResultWriter(str(tmp_path)).submit(targets, {'vertices': torch.from_numpy(verts)}, hd)
