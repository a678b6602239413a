"""ctypes binding of libshapy_b200.so (the C ABI declared in include/shapy_b200.h).

There is NO fallback: if the library is missing or a call fails, a RuntimeError is raised.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('SHAPY_B200_LIB') or os.path.join(_HERE, 'libshapy_b200.so')   # override: build variants

c_void_p, c_int, c_size_t, c_float_p = C.c_void_p, C.c_int, C.c_size_t, C.c_void_p


class SmplxDesc(C.Structure):
    _fields_ = [
        ('num_verts', c_int), ('num_joints', c_int), ('num_betas', c_int), ('num_expr', c_int), ('num_faces', c_int),
        ('v_template', c_void_p), ('shapedirs', c_void_p), ('expr_dirs', c_void_p), ('posedirs', c_void_p),
        ('J_regressor', c_void_p), ('lbs_weights', c_void_p), ('parents', c_void_p), ('faces', c_void_p),
        ('num_static_lmk', c_int), ('lmk_faces_idx', c_void_p), ('lmk_bary_coords', c_void_p),
        ('num_dyn_lmk', c_int), ('num_dyn_rows', c_int), ('dynamic_lmk_faces_idx', c_void_p),
        ('dynamic_lmk_bary_coords', c_void_p), ('neck_chain_len', c_int), ('neck_kin_chain', c_void_p),
        ('num_extra', c_int), ('extra_joint_regressor', c_void_p), ('num_overwrite', c_int),
        ('source_idxs', c_void_p), ('target_idxs', c_void_p),
    ]


class MeasureLandmarks(C.Structure):
    _fields_ = [('face_idx', c_int * 5), ('bc', (C.c_float * 3) * 5)]


class ConvDesc(C.Structure):
    _fields_ = [('cin', c_int), ('cout', c_int), ('ksize', c_int), ('stride', c_int), ('weight', c_void_p),
                ('bias', c_void_p), ('bn_weight', c_void_p), ('bn_bias', c_void_p), ('bn_mean', c_void_p),
                ('bn_var', c_void_p), ('bn_eps', C.c_float)]


class Op(C.Structure):
    _fields_ = [('kind', c_int), ('conv', c_int), ('in_slot', c_int), ('out_slot', c_int), ('out_coff', c_int),
                ('res_slot', c_int), ('relu', c_int), ('n_in', c_int), ('fuse_in', c_int * 4),
                ('fuse_shift', c_int * 4), ('lane', c_int)]


class Slot(C.Structure):
    _fields_ = [('channels', c_int), ('div', c_int)]


class ImageDesc(C.Structure):
    _fields_ = [('offset', C.c_longlong), ('height', c_int), ('width', c_int), ('ul_x', c_int), ('ul_y', c_int),
                ('br_x', c_int), ('br_y', c_int)]


OP_STEM, OP_CONV, OP_FUSE, OP_POOL = 0, 1, 2, 3

_SIGS = {
    'shapy_last_error': (C.c_char_p, []),
    'shapy_version': (c_int, []),
    'shapy_launch_count': (C.c_longlong, []),
    'shapy_smplx_create': (c_int, [C.POINTER(c_void_p), C.POINTER(SmplxDesc)]),
    'shapy_smplx_destroy': (None, [c_void_p]),
    'shapy_smplx_num_keypoints': (c_int, [c_void_p]),
    'shapy_smplx_faces_i32': (c_void_p, [c_void_p]),
    'shapy_smplx_workspace_bytes': (c_size_t, [c_void_p, c_int]),
    'shapy_decode_rot6d': (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    'shapy_smplx_forward': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    'shapy_smplx_forward_shape': (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    'shapy_smplx_shape_backward': (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    'shapy_measure_forward': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, C.POINTER(MeasureLandmarks), c_void_p,
                                      c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    'shapy_measure_forward_tris': (c_int, [c_void_p, c_int, c_int, C.POINTER(MeasureLandmarks), c_void_p, c_void_p,
                                           c_void_p, c_int, c_void_p, c_void_p]),
    'shapy_measure_backward_workspace_bytes': (c_size_t, [c_int, c_int]),
    'shapy_measure_backward': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, C.POINTER(MeasureLandmarks), c_void_p,
                                       c_void_p, c_void_p, c_size_t, c_void_p]),
    'shapy_measure_backward_tris': (c_int, [c_void_p, c_int, c_int, C.POINTER(MeasureLandmarks), c_void_p, c_void_p,
                                            c_void_p]),
    'shapy_mmi_workspace_bytes': (c_size_t, [c_int, c_int, c_int]),
    'shapy_mmi_forward': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                  c_size_t, c_void_p]),
    'shapy_head_workspace_bytes': (c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    'shapy_head_forward': (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_size_t,
                                   c_void_p]),
    'shapy_head_forward_collapsed': (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                             c_void_p, c_void_p, c_size_t, c_void_p]),
    'shapy_hrnet_create': (c_int, [C.POINTER(c_void_p), C.POINTER(ConvDesc), c_int, C.POINTER(Op), c_int,
                                   C.POINTER(Slot), c_int, c_int, c_int, c_int]),
    'shapy_hrnet_destroy': (None, [c_void_p]),
    'shapy_hrnet_workspace_bytes': (c_size_t, [c_void_p, c_int, c_int, c_int]),
    'shapy_hrnet_forward': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    'shapy_hrnet_read_slot': (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    'shapy_hrnet_flops': (C.c_double, [c_void_p, c_int, c_int, c_int]),
    'shapy_preprocess_forward': (c_int, [c_void_p, c_void_p, c_int, c_int, C.POINTER(C.c_float), C.POINTER(C.c_float), c_void_p,
                                         c_void_p]),
    'shapy_b2a_forward': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p,
                                  c_void_p]),
    'shapy_a2b_forward': (c_int, [c_void_p] * 7 + [c_int] * 4 + [c_void_p, c_void_p]),
    'shapy_p2p_workspace_bytes': (c_size_t, [c_int, c_int]),
    'shapy_p2p_error': (c_int, [c_void_p] * 8 + [c_int] * 5 + [c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    'shapy_v2v_error': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    'shapy_conv_test': (c_int, [C.POINTER(ConvDesc), c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                                c_void_p, c_void_p]),
}

EXPORTS = sorted(_SIGS)
_lib = None


def lib():
    """Loads the shared library once.  Raises if it has not been built (python -m shapy_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f'{LIB_PATH} not found: the CUDA extension is not built. Run `python -m shapy_b200.build` '
                '(there is no CPU / PyTorch fallback).')
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)      # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int, what: str = ''):
    if rc != 0:
        msg = lib().shapy_last_error().decode(errors='replace')
        raise RuntimeError(f'shapy_b200 {what} failed (code {rc}): {msg}')


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device / host pointer of a torch tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())
