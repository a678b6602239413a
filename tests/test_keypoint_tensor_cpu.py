"""KeypointTensor (the wrapper every `joints` / `proj_joints` entry of the regressor's output comes in): behaviour of
the mirror class, derived from the reference's class (regressor/human_shape/models/body_models/utils.py:123-309):
indexing gives the plain tensor, tensor methods and torch functions give a KeypointTensor that keeps the keypoint
metadata, `numpy()` gives the array, everything else is forwarded to the wrapped tensor."""
import json
import os

import numpy as np
import torch

from shapy_b200.human_shape.models.body_models.utils import KeypointTensor

META = dict(source='smplx', keypoint_names=['pelvis', 'left_hip', 'right_hip'], connections=[(0, 1), (0, 2)],
            part_indices={'body': [0, 1, 2]}, part_connections={'body': [(0, 1)]})


def make(cls=KeypointTensor):
    return cls(torch.arange(18, dtype=torch.float32).view(2, 3, 3), **META)


def check_meta(k, cls=KeypointTensor):
    assert isinstance(k, cls)
    assert k.source == 'smplx' and k.keypoint_names == META['keypoint_names'] and k.connections == META['connections']
    assert k.part_indices == META['part_indices'] and k.part_connections == META['part_connections']


def test_wrapping_and_forwarding():
    k = make()
    check_meta(k)
    assert tuple(k.shape) == (2, 3, 3) and k.dtype == torch.float32 and k.device.type == 'cpu'
    assert torch.is_tensor(k[0]) and not isinstance(k[0], KeypointTensor) and k[0].shape == (3, 3)   # utils.py:263-264
    assert isinstance(k.numpy(), np.ndarray) and k.numpy().shape == (2, 3, 3)                        # utils.py:278-279
    assert repr(k).startswith('KeypointTensor:')
    # re-wrapping unwraps the tensor (no nested wrapper); the metadata is the constructor's, as in the reference
    assert torch.is_tensor(KeypointTensor(k, **META)._t) and not isinstance(KeypointTensor(k, **META)._t, KeypointTensor)
    check_meta(KeypointTensor(k, **META))
    assert KeypointTensor(k).keypoint_names is None and KeypointTensor(k).source == 'smplx'


def test_methods_and_torch_functions_keep_the_metadata():
    k = make()
    for out in (k.view(2, 9), k.detach(), k.clone(), k.contiguous(), k.to(torch.float64), k.reshape(6, 3)):
        check_meta(out)
    assert k.view(2, 9).shape == (2, 9) and k.to(torch.float64).dtype == torch.float64
    for out in (torch.add(k, 1.0), torch.sum(k, dim=1), torch.matmul(k, torch.eye(3)), torch.clamp(k, 0, 5)):
        check_meta(out)                                # __torch_function__, utils.py:296-309
    assert torch.equal(torch.add(k, 1.0)._t, k._t + 1.0)
    assert torch.allclose(k, k._t) is True             # non-tensor results are returned as they are
    check_meta(KeypointTensor.from_obj(torch.zeros(1, 3, 3), k))
    assert KeypointTensor.from_obj(torch.zeros(1, 3, 3), k).shape == (1, 3, 3)


# tensor METHODS only: the reference's instance-level __torch_function__ predates torch 1.7's protocol and returns
# NotImplemented under torch 2.x, so torch.* functions on its class cannot be compared
REFERENCE_OPS = [lambda k: k.view(2, 9), lambda k: k.detach(), lambda k: k.to(torch.float64), lambda k: k.sum(dim=2),
                 lambda k: k.matmul(torch.full((3, 3), 0.5)), lambda k: k.clone().reshape(3, 6), lambda k: k.permute(2, 0, 1)]


def record(k):
    """What is compared with the reference class: result type, wrapped values and keypoint metadata, as JSON values."""
    return dict(type=type(k).__name__, dtype=str(k._t.dtype), shape=list(k._t.shape), values=k._t.reshape(-1).tolist(),
                keypoint_names=k.keypoint_names, source=k.source, connections=[list(c) for c in k.connections],
                part_indices=k.part_indices)


def test_same_results_as_the_reference_class(golden_dir):
    """The mirror against the reference's own class on REFERENCE_OPS: tests/golden/keypoint_tensor.json holds what the
    reference class returned (tools/make_golden.py keypoint)."""
    with open(os.path.join(golden_dir, 'keypoint_tensor.json')) as f:
        ref = json.load(f)
    a = make()
    assert len(ref['ops']) == len(REFERENCE_OPS)
    for f, r in zip(REFERENCE_OPS, ref['ops']):
        assert record(f(a)) == r
    assert a[1].tolist() == ref['index1'] and type(a[1]).__name__ == ref['index1_type']
    assert a.numpy().tolist() == ref['numpy']
