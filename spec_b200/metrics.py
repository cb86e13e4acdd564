"""Eval-side metrics on the GPU (SURVEY.md section 8f, rank 1).

Replaces what /root/reference/spec/trainer.py:272-316 and /root/reference/spec/utils/compute_error.py:33-86 do per
validation batch -- ``J_regressor_h36m @ vertices`` -> 14 LSP joints (``H36M_TO_J14``) -> pelvis centring -> MPJPE,
Procrustes-aligned MPJPE (``reconstruction_error``: numpy SVD per sample on the host) and per-vertex error
(``compute_error_verts``) -- without copying the 21 MB of vertices per batch to the host.  Units are the inputs' (the
reference multiplies by 1000 afterwards).

``joint_errors`` and ``SPECErrorEval`` add the 24-SMPL-joint and camera-frame protocol of SPEC-SYN / SPEC-MTP
(compute_error.py:33-49,89-223, the 24-joint half of trainer.py:249-344), with :class:`~spec_b200.BodyModel` for the
ground-truth meshes.
"""
import ctypes as C

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from .constants import H36M_TO_J14


class EvalMetrics(nn.Module):
    """``J_regressor`` is the (17, 6890) H36M regressor the reference loads from ``data/J_regressor_h36m.npy`` and
    registers as the buffer ``J_regressor`` (spec/trainer.py:96-99).  ``joint_mapper`` picks the evaluated joints from the
    17: ``H36M_TO_J14`` (14 entries, the default) or ``H36M_TO_J17`` (17 entries, the trainer's ``mpi-inf-3dhp`` branch,
    trainer.py:259-260); any other length raises."""

    def __init__(self, J_regressor_h36m, joint_mapper=H36M_TO_J14):
        super().__init__()
        J = torch.as_tensor(np.asarray(J_regressor_h36m)).float()
        assert J.shape == (17, 6890)
        self.register_buffer('J_regressor', J)
        self.joint_mapper = [int(j) for j in joint_mapper]
        if len(self.joint_mapper) not in (14, 17):
            raise ValueError(f'joint_mapper must have 14 (H36M_TO_J14) or 17 (H36M_TO_J17) entries, got {len(self.joint_mapper)}')
        if not all(0 <= j < 17 for j in self.joint_mapper):
            raise ValueError('joint_mapper entries must index the 17 H36M joints')
        self._handle = None
        self._device = None
        self._ws = None

    def __del__(self):
        try:
            if self._handle is not None:
                _lib.lib().specb200_eval_destroy(self._handle)
        except Exception:
            pass

    def _ensure(self, device):
        if self._handle is not None and self._device == device:
            return
        _lib.require_device()
        J = self.J_regressor.detach().float().contiguous().cpu()
        m = torch.tensor(self.joint_mapper, dtype=torch.int32)
        h = C.c_void_p()
        with torch.cuda.device(device):
            _lib.check(_lib.lib().specb200_eval_create_mapped(C.byref(h), J.data_ptr(), m.data_ptr(), len(self.joint_mapper)))
        self._handle, self._device = h, device

    @torch.no_grad()
    def forward(self, pred_vertices, gt_keypoints_3d=None, gt_vertices=None, center_v2v=False, per_joint=False, pred_rot=None,
                gt_rot=None):
        """pred_vertices (B,6890,3) [may be a strided view of the packed record].  Give either ``gt_keypoints_3d``
        (B,n,3) with n = len(joint_mapper) as the trainer does, or ``gt_vertices`` (B,6890,3) as compute_error.py does (or
        both: keypoints for the joint errors, vertices for v2v).  ``pred_rot`` / ``gt_rot`` (B,3,3): rotate each mesh first
        (the camera-frame metrics, compute_error.py:164,186); ``gt_rot`` also rotates given keypoints.  Returns dict of (B,)
        tensors + ``pred_keypoints_3d`` (B,n,3), and with ``per_joint`` ``mpjpe_per_joint`` / ``pa_mpjpe_per_joint`` (B,n)."""
        _lib.require_device(pred_vertices)
        dev = pred_vertices.device
        B = pred_vertices.shape[0]
        n = len(self.joint_mapper)
        if pred_vertices.stride(2) != 1 or pred_vertices.stride(1) != 3 or pred_vertices.dtype != torch.float32:
            pred_vertices = pred_vertices.float().contiguous()
        if gt_keypoints_3d is None and gt_vertices is None:
            raise ValueError('need gt_keypoints_3d or gt_vertices')
        if gt_keypoints_3d is not None and gt_keypoints_3d.shape[1] != n:
            raise ValueError(f'gt_keypoints_3d has {gt_keypoints_3d.shape[1]} joints, the joint mapper selects {n}')
        if center_v2v and gt_keypoints_3d is not None:
            # the centred vertex error (compute_error.py) subtracts the pelvis regressed from BOTH meshes; with ground-truth
            # keypoints supplied the kernel takes the joint errors from them and never regresses the GT pelvis
            raise ValueError('center_v2v=True needs the joints regressed from gt_vertices: do not pass gt_keypoints_3d with it')
        self._ensure(dev)
        L = _lib.lib()
        kp = gt_keypoints_3d.to(dev, torch.float32).contiguous() if gt_keypoints_3d is not None else None
        gv = gt_vertices.to(dev, torch.float32) if gt_vertices is not None else None
        if gv is not None and (gv.stride(2) != 1 or gv.stride(1) != 3):
            gv = gv.contiguous()
        pr, gr = _rot(pred_rot, B, dev), _rot(gt_rot, B, dev)
        nb = L.specb200_eval_workspace_bytes(self._handle, B)
        if self._ws is None or self._ws.numel() < nb or self._ws.device != dev:
            self._ws = torch.empty(nb, dtype=torch.uint8, device=dev)
        out = {k: torch.empty(B, dtype=torch.float32, device=dev) for k in ('mpjpe', 'pa_mpjpe')}
        v2v = torch.empty(B, dtype=torch.float32, device=dev) if gv is not None else None
        pk = torch.empty(B, n, 3, dtype=torch.float32, device=dev)
        pj = [torch.empty(B, n, dtype=torch.float32, device=dev) for _ in range(2)] if per_joint else [None, None]
        ptr = lambda t: t.data_ptr() if t is not None else 0
        with torch.cuda.device(dev):
            _lib.check(L.specb200_eval_forward_ex(self._handle, B, pred_vertices.data_ptr(), pred_vertices.stride(0), ptr(pr), ptr(kp),
                                                  ptr(gv), gv.stride(0) if gv is not None else 0, ptr(gr), int(bool(center_v2v)),
                                                  self._ws.data_ptr(), self._ws.numel(), out['mpjpe'].data_ptr(),
                                                  out['pa_mpjpe'].data_ptr(), ptr(v2v), pk.data_ptr(), ptr(pj[0]), ptr(pj[1]), n,
                                                  torch.cuda.current_stream(dev).cuda_stream))
        if v2v is not None:
            out['v2v'] = v2v
        out['pred_keypoints_3d'] = pk
        if per_joint:
            out['mpjpe_per_joint'], out['pa_mpjpe_per_joint'] = pj
        return out


def _rot(r, B, dev):
    if r is None:
        return None
    _lib.require_device(r)
    return r.to(dev, torch.float32).reshape(B, 9).contiguous()


@torch.no_grad()
def joint_errors(pred, gt, center=True, per_joint=False, rot_pred=None, rot_gt=None):
    """MPJPE and Procrustes-aligned MPJPE of already-regressed joints ``pred``, ``gt`` (B,n,3), n = 14, 17 or 24, in input
    units.  ``center=True`` subtracts joint 0 on both sides first (compute_error.py:33-49 ``eval_j_24``); ``center=False``
    takes them as given (the trainer's ``error_j_24`` / ``reconstruction_error(pred_joints_24, gt_joints_24)``,
    trainer.py:282-302, after it subtracted the predicted pelvis itself).  ``rot_pred`` / ``rot_gt`` (B,3,3) rotate each side
    before the centring.  Returns a dict of (B,) tensors ``mpjpe``, ``pa_mpjpe`` and with ``per_joint`` the (B,n)
    ``mpjpe_per_joint`` / ``pa_mpjpe_per_joint`` (``reconstruction_error(..., reduction=None)[1]``)."""
    _lib.require_device(pred)
    dev = pred.device
    if pred.dim() != 3 or pred.shape[2] != 3 or pred.shape != gt.shape:
        raise ValueError(f'pred and gt must both be (B,n,3), got {tuple(pred.shape)} and {tuple(gt.shape)}')
    B, n = pred.shape[0], pred.shape[1]
    if n not in (14, 17, 24):
        raise ValueError(f'joint_errors evaluates 14, 17 or 24 joints, got {n}')
    p = pred.to(dev, torch.float32).contiguous()
    g = gt.to(dev, torch.float32).contiguous()
    rp, rg = _rot(rot_pred, B, dev), _rot(rot_gt, B, dev)
    out = {k: torch.empty(B, dtype=torch.float32, device=dev) for k in ('mpjpe', 'pa_mpjpe')}
    pj = [torch.empty(B, n, dtype=torch.float32, device=dev) for _ in range(2)] if per_joint else [None, None]
    ptr = lambda t: t.data_ptr() if t is not None else 0
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().specb200_eval_joint_errors(B, n, p.data_ptr(), g.data_ptr(), ptr(rp), ptr(rg), int(bool(center)),
                                                         out['mpjpe'].data_ptr(), out['pa_mpjpe'].data_ptr(), ptr(pj[0]), ptr(pj[1]),
                                                         torch.cuda.current_stream(dev).cuda_stream))
    if per_joint:
        out['mpjpe_per_joint'], out['pa_mpjpe_per_joint'] = pj
    return out


SPEC_ERROR_KEYS = ('w_mpjpe', 'mpjpe', 'pa_mpjpe', 'w_v2v', 'v2v', 'w_mpjpe_24', 'mpjpe_24', 'pa_mpjpe_24')


class SPECErrorEval(nn.Module):
    """The per-batch body of ``compute_error`` (/root/reference/spec/utils/compute_error.py:142-203) on the device: the
    world-frame and camera-frame errors of SPEC-SYN / SPEC-MTP (14 H36M joints, 24 SMPL joints, vertices).

    ``body_model`` (a :class:`~spec_b200.BodyModel`) supplies the ``J_regressor`` that regresses the 24 predicted joints
    (``body_model_orig.J_regressor``); ``body_model_gt`` (default: ``body_model``) builds the ground-truth meshes."""

    def __init__(self, J_regressor_h36m, body_model, body_model_gt=None):
        super().__init__()
        self.metrics = EvalMetrics(J_regressor_h36m, H36M_TO_J14)
        self.body_model = body_model
        self.body_model_gt = body_model_gt if body_model_gt is not None else body_model

    @torch.no_grad()
    def batch(self, pred_vertices, gt_pose, gt_betas, pred_cam_rotmat, gt_cam_rotmat=None, gt_pose_cam=None):
        """pred_vertices (B,6890,3) (may be the strided ``smpl_vertices`` view of a packed record); gt_pose (B,72) axis-angle;
        gt_betas (B,10); pred_cam_rotmat (B,3,3).  With ``gt_cam_rotmat`` (B,3,3) the ``spec-syn`` branch runs (the GT mesh
        and joints are rotated by it, and so is the prediction); otherwise ``gt_pose_cam`` (B,72) gives the camera-frame GT
        mesh.  Returns a dict of (B,) tensors in input units (compute_error multiplies by 1000): ``w_mpjpe, mpjpe, pa_mpjpe,
        w_v2v, v2v, w_mpjpe_24, mpjpe_24, pa_mpjpe_24``."""
        _lib.require_device(pred_vertices)
        if gt_cam_rotmat is None and gt_pose_cam is None:
            raise ValueError('give gt_cam_rotmat (spec-syn) or gt_pose_cam')
        gt = self.body_model_gt(betas=gt_betas, global_orient=gt_pose[:, :3], body_pose=gt_pose[:, 3:])
        if gt_cam_rotmat is not None:                                   # compute_error.py:162-166
            rot_p = rot_g = gt_cam_rotmat
            gt_cam_vertices, gt_cam_joints = gt.vertices, gt.joints
        else:                                                           # compute_error.py:167-181
            rot_p, rot_g = pred_cam_rotmat, None
            gc = self.body_model_gt(betas=gt_betas, global_orient=gt_pose_cam[:, :3], body_pose=gt_pose_cam[:, 3:])
            gt_cam_vertices, gt_cam_joints = gc.vertices, gc.joints
        w = self.metrics(pred_vertices, gt_vertices=gt.vertices, center_v2v=True)                          # :189
        c = self.metrics(pred_vertices, gt_vertices=gt_cam_vertices, center_v2v=True, pred_rot=rot_p, gt_rot=rot_g)   # :190
        w24 = joint_errors(self.body_model.regress_joints(pred_vertices), gt.joints, center=True)          # :184,192
        c24 = joint_errors(self.body_model.regress_joints(pred_vertices, rot=rot_p), gt_cam_joints, center=True, rot_gt=rot_g)  # :187,193
        return {'w_mpjpe': w['mpjpe'], 'mpjpe': c['mpjpe'], 'pa_mpjpe': w['pa_mpjpe'], 'w_v2v': w['v2v'], 'v2v': c['v2v'],
                'w_mpjpe_24': w24['mpjpe'], 'mpjpe_24': c24['mpjpe'], 'pa_mpjpe_24': w24['pa_mpjpe']}

    @staticmethod
    def summary(per_image, dataset_name):
        """The values compute_error logs (compute_error.py:207-223), in millimetres, from ``batch`` outputs (one dict or a
        list of them, input units = metres).  Reproduced as the reference logs them, quirks included: ``C-MPJPE`` /
        ``C-MPJPE-24`` are the WORLD-frame ``w_mpjpe`` / ``w_mpjpe_24`` and ``C-V2V`` is the world-frame ``w_v2v`` (the
        reference logs ``wmpjpe_error`` and ``wvertex2vertex_error`` under those names)."""
        if isinstance(per_image, dict):
            per_image = [per_image]
        cat = {k: np.concatenate([np.asarray(torch.as_tensor(d[k]).detach().cpu(), dtype=np.float64).reshape(-1) for d in per_image])
               for k in SPEC_ERROR_KEYS}
        mm = {k: float(v.mean() * 1000.0) for k, v in cat.items()}
        if dataset_name == '3dpw-test-cam':          # standard protocol for 3dpw is 14 joint evaluation
            out = {'W-MPJPE': mm['w_mpjpe'], 'C-MPJPE': mm['w_mpjpe'], 'MPJPE': mm['mpjpe'], 'PA-MPJPE': mm['pa_mpjpe']}
        else:                                        # 24 SMPL joints for SPEC-SYN and SPEC-MTP
            out = {'W-MPJPE-24': mm['w_mpjpe_24'], 'C-MPJPE-24': mm['w_mpjpe_24'], 'MPJPE-24': mm['mpjpe_24'],
                   'PA-MPJPE-24': mm['pa_mpjpe_24']}
        out.update({'W-V2V': mm['w_v2v'], 'C-V2V': mm['w_v2v'], 'V2V': mm['v2v']})
        return out
