"""ctypes binding of libspecb200.so (the C ABI in include/specb200.h).

There is no fallback: if the library is missing it is built with nvcc; if that fails, or a
compute call is made without an sm_100 device, a RuntimeError is raised.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libspecb200.so')

OP_CONV, OP_MAXPOOL, OP_UPADD, OP_BILINEAR, OP_COPY = 1, 2, 3, 4, 5
PREC = {'fp32': 0, 'bf16': 1, 'fp16': 2}


class Op(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ('type', 'src', 'src2', 'dst', 'cin', 'cout', 'kh', 'kw', 'stride', 'pad',
                                          'relu', 'dst_coff', 'shift', 'wslot', 'pair')]


_F = C.POINTER(C.c_float)
_I = C.POINTER(C.c_int32)


class HmrParams(C.Structure):
    _fields_ = ([('in_features', C.c_int32), ('use_cam_feats', C.c_int32), ('use_cam', C.c_int32),
                 ('focal_length', C.c_float), ('img_res', C.c_float)] +
                [(n, C.c_void_p) for n in ('fc1_w', 'fc1_b', 'fc2_w', 'fc2_b', 'decpose_w', 'decpose_b', 'decshape_w',
                                           'decshape_b', 'deccam_w', 'deccam_b', 'init_pose', 'init_shape', 'init_cam',
                                           'v_template', 'shapedirs', 'posedirs', 'J_regressor', 'lbs_weights',
                                           'J_regressor_extra', 'parents', 'joint_map', 'vertex_ids')])


OUTPUT_KEYS = ('smpl_vertices', 'smpl_joints3d', 'smpl_joints2d', 'pred_cam_t', 'pred_pose', 'pred_cam',
               'pred_shape', 'pred_pose_6d')


class HmrOutputs(C.Structure):
    _fields_ = [f for k in ('vertices', 'joints3d', 'joints2d', 'cam_t', 'pose', 'cam', 'shape', 'pose_6d')
                for f in ((('smpl_' if k in ('vertices', 'joints3d', 'joints2d') else 'pred_') + k, C.c_void_p),
                          ('ld_' + k, C.c_int64))]


_lib = None

_PROTOS = {
    'specb200_last_error': (C.c_char_p, []),
    'specb200_abi_version': (C.c_int, []),
    'specb200_device_check': (C.c_int, []),
    'specb200_trunk_create': (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(Op), C.c_int32, _I, C.c_int32, C.c_int32,
                                        C.c_int32, C.c_int32]),
    'specb200_trunk_set_conv': (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                          C.c_int32, C.c_int32]),
    'specb200_trunk_set_chunk': (C.c_int, [C.c_void_p, C.c_int32]),
    'specb200_trunk_out_shape': (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, _I, _I, _I]),
    'specb200_trunk_workspace_bytes': (C.c_int64, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32]),
    'specb200_trunk_forward': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                         C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    'specb200_trunk_forward_until': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_int32,
                                               _I, _I, _I, C.c_void_p, C.c_void_p]),
    'specb200_trunk_last_launches': (C.c_int64, [C.c_void_p]),
    'specb200_trunk_num_ops': (C.c_int32, [C.c_void_p]),
    'specb200_trunk_num_fused_bottlenecks': (C.c_int32, [C.c_void_p]),
    'specb200_trunk_fused_group_first_op': (C.c_int32, [C.c_void_p, C.c_int32]),
    'specb200_trunk_profile': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int64,
                                         C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    'specb200_trunk_destroy': (None, [C.c_void_p]),
    'specb200_camtail_create': (C.c_int, [C.POINTER(C.c_void_p), C.c_int32, C.c_int32]),
    'specb200_camtail_add_linear': (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]),
    'specb200_camtail_finalize': (C.c_int, [C.c_void_p]),
    'specb200_camtail_workspace_bytes': (C.c_int64, [C.c_void_p, C.c_int32]),
    'specb200_camtail_forward': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int64,
                                           C.c_void_p, C.c_void_p]),
    'specb200_camcalib_decode': (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'specb200_camtail_destroy': (None, [C.c_void_p]),
    'specb200_hmrtail_create': (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(HmrParams)]),
    'specb200_hmrtail_workspace_bytes': (C.c_int64, [C.c_void_p, C.c_int32]),
    'specb200_hmrtail_x_ld': (C.c_int32, [C.c_void_p]),
    'specb200_hmrtail_forward': (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(HmrOutputs),
                                           C.c_void_p]),
    'specb200_hmrtail_last_launches': (C.c_int64, [C.c_void_p]),
    'specb200_hmrtail_destroy': (None, [C.c_void_p]),
    'specb200_eval_create': (C.c_int, [C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p]),
    'specb200_eval_workspace_bytes': (C.c_int64, [C.c_void_p, C.c_int32]),
    'specb200_eval_forward': (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32,
                                        C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'specb200_eval_create_mapped': (C.c_int, [C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p, C.c_int32]),
    'specb200_eval_forward_ex': (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                           C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    'specb200_eval_joint_errors': (C.c_int, [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'specb200_eval_destroy': (None, [C.c_void_p]),
    'specb200_body_create': (C.c_int, [C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'specb200_body_workspace_bytes': (C.c_int64, [C.c_void_p, C.c_int32]),
    'specb200_body_forward': (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p,
                                        C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]),
    'specb200_body_regress_joints': (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    'specb200_body_destroy': (None, [C.c_void_p]),
    'specb200_preproc_create': (C.c_int, [C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p]),
    'specb200_preproc_crop': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_void_p, C.c_int32,
                                        C.c_double, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    'specb200_preproc_crop_transforms': (C.c_int, [C.c_void_p, C.c_int32, C.c_double, C.c_int32, C.c_void_p, C.c_void_p]),
    'specb200_preproc_resized_shape': (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    'specb200_preproc_resize_workspace_bytes': (C.c_int64, [C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    'specb200_preproc_resize': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
                                          C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    'specb200_preproc_destroy': (None, [C.c_void_p]),
    'specb200_gather_create': (C.c_int, [C.POINTER(C.c_void_p), C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_void_p]),
    'specb200_gather_connect': (C.c_int, [C.c_void_p, C.c_void_p]),
    'specb200_gather_recv_ptr': (C.c_void_p, [C.c_void_p, C.c_int32]),
    'specb200_allgather_outputs': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_uint32, C.c_int32, C.c_void_p]),
    'specb200_gather_set_push_ctas': (C.c_int, [C.c_void_p, C.c_int32]),
    'specb200_gather_destroy': (None, [C.c_void_p]),
    'specb200_linear_f32': (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                                      C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_PROTOS)


def lib():
    """Load (building first if necessary) libspecb200.so.  Raises if it cannot be had."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        from .build import build_library
        build_library()
    l = C.CDLL(LIB_PATH)
    for name, (res, args) in _PROTOS.items():
        fn = getattr(l, name)          # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if l.specb200_abi_version() != 1:
        raise RuntimeError('libspecb200 ABI version mismatch')
    _lib = l
    return l


def check(rc):
    if rc != 0:
        raise RuntimeError('libspecb200: ' + lib().specb200_last_error().decode())


_device_ok = set()


def require_device(t=None):
    """The product has no CPU path: refuse anything but a CUDA sm_100 tensor/device.  The architecture check is made once
    per device (it is a driver query; on the hot path it cost milliseconds per call and blocked behind nvidia-smi pollers)."""
    import torch
    if t is not None and not t.is_cuda:
        raise RuntimeError('spec_b200 has no CPU path: tensors must live on a CUDA sm_100 (B200) device '
                           f'(got {t.device})')
    key = t.device.index if t is not None else -1
    if key in _device_ok:
        return
    if not torch.cuda.is_available():
        raise RuntimeError('spec_b200 has no CPU path: no CUDA device available')
    if t is not None:
        with torch.cuda.device(t.device):
            check(lib().specb200_device_check())
    else:
        check(lib().specb200_device_check())
    _device_ok.add(key)


def refuse_training(module):
    """The library implements the INFERENCE path only (eval-mode BatchNorm folded into the conv weights, dropout = identity,
    no autograd graph).  The reference shares these classes with its trainer (spec/trainer.py:50-56): a ``forward`` in training
    mode with gradients enabled would silently train nothing, so it raises instead."""
    import torch
    if module.training and torch.is_grad_enabled():
        raise RuntimeError(f'{type(module).__name__}: spec_b200 implements the inference path only -- call .eval() and/or run under '
                           'torch.no_grad(); training (spec/trainer.py) is out of scope')


class VersionWatch:
    """In-place version counters of every parameter and buffer of some modules, snapshotted when their packed device copies
    are made: lets the next forward notice in-place updates (optimizer steps, ``param.data.copy_``) that neither
    ``load_state_dict`` nor ``_apply`` report.  Checking costs one attribute read per tensor (~50 us for two ResNet-50s)."""

    def __init__(self, *modules):
        self.tensors = [t for m in modules for t in list(m.parameters()) + list(m.buffers())]
        self.snap = tuple(t._version for t in self.tensors)

    def changed(self):
        return tuple(t._version for t in self.tensors) != self.snap
