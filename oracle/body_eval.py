"""CPU oracle of the SPEC evaluation protocol (TEST INFRASTRUCTURE): the axis-angle SMPL forward and the 24-joint /
camera-frame errors of /root/reference/spec/utils/compute_error.py:33-203.

``batch_rodrigues`` and the ``pose2rot=True`` path of ``smplx.lbs`` are [UPSTREAM-RECALLED] (smplx 0.1.28, not installed
offline); the skinning itself is ``oracle.head.lbs``.  ``reconstruction_error_per_joint`` is pare's
``reconstruction_error(..., reduction=None)`` [UPSTREAM-RECALLED: SPIN's utils/pose_utils.py], built on
``oracle.eval_metrics.compute_similarity_transform``.  ``eval_j_24`` and ``compute_error_batch`` restate the reference's
own code (compute_error.py:33-49 and the loop body 142-203); tests/golden/reference_eval.py pins them to its unmodified
``eval_single`` / ``eval_j_24``.  Errors are in input units (the reference multiplies by 1000).
"""
import numpy as np
import torch

from .constants import SMPL_PARENTS
from .eval_metrics import compute_similarity_transform, eval_single
from .head import lbs


def batch_rodrigues(rot_vecs):
    """smplx.lbs.batch_rodrigues: (N,3) axis-angle -> (N,3,3).  angle = |r + 1e-8|, R = I + sin K + (1 - cos) K^2."""
    N, dtype = rot_vecs.shape[0], rot_vecs.dtype
    angle = torch.norm(rot_vecs + 1e-8, dim=1, keepdim=True)
    rot_dir = rot_vecs / angle
    cos = torch.unsqueeze(torch.cos(angle), dim=1)
    sin = torch.unsqueeze(torch.sin(angle), dim=1)
    rx, ry, rz = torch.split(rot_dir, 1, dim=1)
    zeros = torch.zeros((N, 1), dtype=dtype)
    K = torch.cat([zeros, -rz, ry, rz, zeros, -rx, -ry, rx, zeros], dim=1).view((N, 3, 3))
    ident = torch.eye(3, dtype=dtype).unsqueeze(dim=0)
    return ident + sin * K + (1 - cos) * torch.bmm(K, K)


def smpl_forward(smpl, betas, global_orient, body_pose, pose2rot=True):
    """``smplx.SMPL(...)(betas=, global_orient=, body_pose=, pose2rot=)`` without translation: returns (vertices (B,6890,3),
    joints (B,24,3) = ``.joints[:, :24]``, the posed kinematic joints).  ``smpl``: dict / module with smplx's buffer names.
    Computes in the dtype of ``betas``."""
    get = (lambda k: smpl[k]) if isinstance(smpl, dict) else (lambda k: getattr(smpl, k))
    dt = betas.dtype
    c = lambda k: torch.as_tensor(np.asarray(get(k)) if isinstance(smpl, dict) else get(k)).to(dt)
    B = betas.shape[0]
    if pose2rot:
        full = torch.cat([global_orient.reshape(B, 3), body_pose.reshape(B, 69)], 1).to(dt)
        rotmats = batch_rodrigues(full.reshape(-1, 3)).view(B, 24, 3, 3)
    else:
        rotmats = torch.cat([global_orient.reshape(B, 1, 3, 3), body_pose.reshape(B, 23, 3, 3)], 1).to(dt)
    return lbs(betas, rotmats, c('v_template'), c('shapedirs'), c('posedirs'), c('J_regressor'), SMPL_PARENTS, c('lbs_weights'))


def reconstruction_error_per_joint(S1, S2):
    """pare ``reconstruction_error(S1, S2, reduction=None)``: (per-image mean, per-joint distances) after one similarity
    alignment per image."""
    S1_hat = np.stack([compute_similarity_transform(a, b) for a, b in zip(S1, S2)])
    re_per_joint = np.sqrt(((S1_hat - S2) ** 2).sum(axis=-1))
    return re_per_joint.mean(axis=-1), re_per_joint


def eval_j_24(pred_joints, gt_joints):
    """compute_error.py:33-49: both sides centred on joint 0; returns (mpjpe, pa_mpjpe) per image."""
    pred_joints = pred_joints - pred_joints[:, [0], :].clone()
    gt_joints = gt_joints - gt_joints[:, [0], :].clone()
    pa, _ = reconstruction_error_per_joint(pred_joints.numpy(), gt_joints.numpy())
    mpjpe = torch.sqrt(((pred_joints - gt_joints) ** 2).sum(dim=-1)).mean(dim=-1).numpy()
    return mpjpe, pa


def compute_error_batch(pred_verts, gt_pose, gt_betas, pred_cam_rotmat, J_regressor_h36m, smpl, gt_cam_rotmat=None,
                        gt_pose_cam=None):
    """One batch of the compute_error loop (compute_error.py:142-203).  ``gt_cam_rotmat`` given: the ``spec-syn`` branch;
    otherwise ``gt_pose_cam``.  ``smpl`` serves as both ``body_model`` and ``body_model_orig`` (one SMPL model dir).
    Returns a dict of (B,) arrays (input units)."""
    gt_vertices, gt_joints = smpl_forward(smpl, gt_betas, gt_pose[:, :3], gt_pose[:, 3:])
    if gt_cam_rotmat is not None:
        gt_cam_vertices = torch.bmm(gt_cam_rotmat, gt_vertices.transpose(2, 1)).transpose(2, 1)
        gt_cam_joints = torch.bmm(gt_cam_rotmat, gt_joints.transpose(2, 1)).transpose(2, 1)
        pred_cam_rotmat = gt_cam_rotmat
    else:
        gt_cam_vertices, gt_cam_joints = smpl_forward(smpl, gt_betas, gt_pose_cam[:, :3], gt_pose_cam[:, 3:])
    Jr = torch.as_tensor(np.asarray(smpl['J_regressor'] if isinstance(smpl, dict) else smpl.J_regressor)).to(pred_verts.dtype)
    pred_joints = torch.einsum('bik,ji->bjk', [pred_verts, Jr])
    pred_vertices_gt_cam = torch.bmm(pred_cam_rotmat, pred_verts.transpose(2, 1)).transpose(2, 1)
    pred_cam_joints = torch.einsum('bik,ji->bjk', [pred_vertices_gt_cam, Jr])
    J = torch.as_tensor(np.asarray(J_regressor_h36m)).to(pred_verts.dtype)
    wmpjpe, pampjpe, wv2v = eval_single(pred_verts, gt_vertices, J)
    mpjpe, _, v2v = eval_single(pred_vertices_gt_cam, gt_cam_vertices, J)
    wmpjpe_24, pampjpe_24 = eval_j_24(pred_joints, gt_joints)
    mpjpe_24, _ = eval_j_24(pred_cam_joints, gt_cam_joints)
    return {'w_mpjpe': wmpjpe, 'mpjpe': mpjpe, 'pa_mpjpe': pampjpe, 'w_v2v': wv2v, 'v2v': v2v,
            'w_mpjpe_24': wmpjpe_24, 'mpjpe_24': mpjpe_24, 'pa_mpjpe_24': pampjpe_24}
