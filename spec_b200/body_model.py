"""SMPL body model on the device: the ``smplx.SMPL`` forward the evaluation side calls with ground-truth or predicted
parameters (/root/reference/spec/utils/compute_error.py:115-181: axis-angle pose with smplx's default ``pose2rot=True``;
/root/reference/spec/trainer.py:249-254: the predicted rotation matrices with ``pose2rot=False``).

It runs the HMR tail's SMPL kernels (csrc/tail.cu): one prep kernel (batch_rodrigues or the given rotations, rest joints,
kinematic chain) and the blend-shape + skinning kernel.  Vertices and the 24 posed kinematic joints come back; nothing is
synchronised, so ``forward`` can be captured in a CUDA graph after one warm-up call.
"""
import ctypes as C
from collections import namedtuple

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from .hmr import _load_smpl_data

BodyModelOutput = namedtuple('BodyModelOutput', ['vertices', 'joints'])
BodyModelOutput.__doc__ = """``vertices`` (B,6890,3); ``joints`` (B,24,3) = ``smplx.SMPL(...).joints[:, :24]``, the posed kinematic joints
(not smplx's 45-joint tensor, whose entries 24.. are vertex picks)."""


class BodyModel(nn.Module):
    """Stands in for ``smplx.SMPL(SMPL_MODEL_DIR, gender=..., create_transl=False)`` on the evaluation side.

    Buffers carry smplx's names (``v_template``, ``shapedirs``, ``posedirs``, ``J_regressor``, ``lbs_weights``,
    ``parents``).  Assets load like the HMR's SMPL layer: ``SMPL_{NEUTRAL,MALE,FEMALE}.{npz,pkl}`` under
    ``SPECB200_SMPL_DIR``; ``smpl_data=`` (a dict of those arrays) overrides ``gender``.  There is no CPU path."""

    def __init__(self, smpl_data=None, gender='neutral'):
        super().__init__()
        d = smpl_data if smpl_data is not None else _load_smpl_data(gender, need_extra=False)
        f = lambda k: torch.as_tensor(np.asarray(d[k])).float()
        self.register_buffer('v_template', f('v_template'))          # (6890,3)
        self.register_buffer('shapedirs', f('shapedirs'))            # (6890,3,10)
        self.register_buffer('posedirs', f('posedirs'))              # (207,20670)
        self.register_buffer('J_regressor', f('J_regressor'))        # (24,6890)
        self.register_buffer('lbs_weights', f('lbs_weights'))        # (6890,24)
        self.register_buffer('parents', torch.as_tensor(np.asarray(d['parents'])).long())
        assert self.v_template.shape == (6890, 3) and self.shapedirs.shape == (6890, 3, 10)
        assert self.posedirs.shape == (207, 20670) and self.J_regressor.shape == (24, 6890) and self.lbs_weights.shape == (6890, 24)
        self.gender = gender
        self._handle = None
        self._device = None
        self._watch = None
        self._ws = None

    def __del__(self):
        try:
            self._release()
        except Exception:
            pass

    def _release(self):
        if self._handle is not None:
            _lib.lib().specb200_body_destroy(self._handle)
            self._handle = None

    def _apply(self, fn, *a, **k):
        self._release()
        return super()._apply(fn, *a, **k)

    def _ensure(self, device):
        if self._handle is not None and self._device == device and not self._watch.changed():
            return
        _lib.require_device()
        self._release()
        keep = [self.v_template, self.shapedirs, self.posedirs, self.J_regressor, self.lbs_weights]
        keep = [t.detach().float().contiguous().cpu() for t in keep]
        par = self.parents.detach().to(torch.int32).contiguous().cpu()
        h = C.c_void_p()
        with torch.cuda.device(device):
            _lib.check(_lib.lib().specb200_body_create(C.byref(h), *[t.data_ptr() for t in keep], par.data_ptr()))
        self._handle, self._device = h, device
        self._watch = _lib.VersionWatch(self)

    def _workspace(self, B, device):
        n = _lib.lib().specb200_body_workspace_bytes(self._handle, B)
        if self._ws is None or self._ws.numel() < n or self._ws.device != device:
            self._ws = torch.empty(n, dtype=torch.uint8, device=device)
        return self._ws

    @torch.no_grad()
    def forward(self, betas=None, body_pose=None, global_orient=None, pose2rot=True):
        """smplx's argument names.  ``pose2rot=True``: ``global_orient`` (B,3) and ``body_pose`` (B,69) axis-angle;
        ``pose2rot=False``: rotation matrices, ``global_orient`` (B,1,3,3) and ``body_pose`` (B,23,3,3) (any shape with
        9 floats per joint).  ``betas`` (B,10).  Missing arguments are zeros, as smplx's defaults are.
        Returns ``BodyModelOutput(vertices (B,6890,3), joints (B,24,3))``."""
        ref = next((t for t in (betas, body_pose, global_orient) if t is not None), None)
        if ref is None:
            raise ValueError('BodyModel.forward needs at least one of betas, body_pose, global_orient (for the batch size)')
        _lib.require_device(ref)
        dev, B = ref.device, ref.shape[0]
        if B == 0:
            raise ValueError('empty batch')
        per = 3 if pose2rot else 9

        def part(x, joints):
            if x is None:
                if pose2rot:
                    return torch.zeros(B, joints * 3, dtype=torch.float32, device=dev)
                return torch.eye(3, dtype=torch.float32, device=dev).reshape(1, 1, 9).expand(B, joints, 9).reshape(B, joints * 9)
            _lib.require_device(x)
            x = x.to(dev, torch.float32).reshape(B, -1)
            if x.shape[1] != joints * per:
                raise ValueError(f'expected {joints * per} values per image, got {x.shape[1]}')
            return x
        pose = torch.cat([part(global_orient, 1), part(body_pose, 23)], 1).contiguous()
        if betas is None:
            betas = torch.zeros(B, 10, dtype=torch.float32, device=dev)
        _lib.require_device(betas)
        betas = betas.to(dev, torch.float32).reshape(B, -1)
        if betas.shape[1] != 10:
            raise ValueError(f'betas: expected 10 shape coefficients, got {betas.shape[1]}')
        betas = betas.contiguous()
        self._ensure(dev)
        ws = self._workspace(B, dev)
        verts = torch.empty(B, 6890, 3, dtype=torch.float32, device=dev)
        joints = torch.empty(B, 24, 3, dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().specb200_body_forward(self._handle, B, betas.data_ptr(), pose.data_ptr(), 0 if pose2rot else 1,
                                                        ws.data_ptr(), ws.numel(), verts.data_ptr(), 6890 * 3, joints.data_ptr(), 72,
                                                        torch.cuda.current_stream(dev).cuda_stream))
        return BodyModelOutput(verts, joints)

    @torch.no_grad()
    def regress_joints(self, vertices, rot=None):
        """``einsum('bik,ji->bjk', vertices, J_regressor)`` (compute_error.py:184), optionally followed by the per-image
        rotation ``rot`` (B,3,3): the joints of ``bmm(rot, vertices)``.  ``vertices`` (B,6890,3) may be a strided view (the
        ``smpl_vertices`` of a packed record).  Returns (B,24,3)."""
        _lib.require_device(vertices)
        dev, B = vertices.device, vertices.shape[0]
        vertices = _vertex_view(vertices)
        self._ensure(dev)
        r = _rot(rot, B, dev)
        out = torch.empty(B, 24, 3, dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().specb200_body_regress_joints(self._handle, B, vertices.data_ptr(), vertices.stride(0),
                                                               r.data_ptr() if r is not None else 0, out.data_ptr(),
                                                               torch.cuda.current_stream(dev).cuda_stream))
        return out


def _vertex_view(v):
    """(B,6890,3) fp32 with unit strides inside an image (the per-image stride is free)."""
    if v.dim() != 3 or v.shape[1:] != (6890, 3):
        raise ValueError(f'expected vertices of shape (B,6890,3), got {tuple(v.shape)}')
    if v.dtype != torch.float32 or v.stride(2) != 1 or v.stride(1) != 3:
        v = v.float().contiguous()
    return v


def _rot(r, B, dev):
    if r is None:
        return None
    _lib.require_device(r)
    return r.to(dev, torch.float32).reshape(B, 9).contiguous()
