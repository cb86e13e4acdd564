"""Geometry helpers of the hot path, restated for the CPU oracle.

All of these live upstream in ``pare.utils.geometry`` / ``pare.models.layers``
([UPSTREAM-RECALLED], SURVEY.md Appendix A.3, A.5-A.8); the reference call
sites that constrain them are cited per function.
"""
import numpy as np
import torch
import torch.nn.functional as F


def rotmat_to_rot6d(R):
    """(B,3,3) -> (B,6): first two columns, row-major (A.3).  Used by HMRHead on
    ``cam_rotmat`` (call site /root/reference/spec/models/hmr.py:96)."""
    return R[:, :, :2].reshape(R.shape[0], 6)


def rot6d_to_rotmat(x):
    """(B,144)->(B*24,3,3) Gram-Schmidt (A.3); output consumed as (B,24,3,3) at
    /root/reference/spec/trainer.py:250-252."""
    x = x.reshape(-1, 3, 2)
    a1, a2 = x[:, :, 0], x[:, :, 1]
    b1 = F.normalize(a1, dim=1, eps=1e-12)
    b2 = F.normalize(a2 - torch.einsum('bi,bi->b', b1, a2).unsqueeze(-1) * b1, dim=1, eps=1e-12)
    b3 = torch.cross(b1, b2, dim=1)
    return torch.stack((b1, b2, b3), dim=-1)


def softargmax1d(heatmaps, temperature=1.0, normalize_keypoints=True):
    """(B,C,D) -> ((B,C), probs) (A.7); call site /root/reference/camcalib/cam_utils.py:114-118."""
    D = heatmaps.shape[-1]
    p = torch.softmax(heatmaps * temperature, dim=-1)
    idx = torch.arange(D, dtype=heatmaps.dtype, device=heatmaps.device)
    k = (p * idx).sum(-1)
    if normalize_keypoints:
        k = k / float(D - 1) * 2 - 1
    return k, p


def batch_euler2matrix(r):
    """(B,3) euler (x,y,z) -> (B,3,3) via quaternion (A.8); call site
    /root/reference/spec/utils/cam_params.py:37 with r=(pitch,0,roll)."""
    h = r * 0.5
    cx, cy, cz = torch.cos(h[:, 0]), torch.cos(h[:, 1]), torch.cos(h[:, 2])
    sx, sy, sz = torch.sin(h[:, 0]), torch.sin(h[:, 1]), torch.sin(h[:, 2])
    qw = cx * cy * cz - sx * sy * sz
    qx = cx * sy * sz + cy * cz * sx
    qy = cx * cz * sy - sx * cy * sz
    qz = cx * cy * sz + sx * cz * sy
    q = torch.stack([qw, qx, qy, qz], 1)
    q = q / q.norm(p=2, dim=1, keepdim=True)
    w, x, y, z = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    w2, x2, y2, z2 = w * w, x * x, y * y, z * z
    wx, wy, wz, xy, xz, yz = w * x, w * y, w * z, x * y, x * z, y * z
    R = torch.stack([
        w2 + x2 - y2 - z2, 2 * xy - 2 * wz, 2 * wy + 2 * xz,
        2 * wz + 2 * xy, w2 - x2 + y2 - z2, 2 * yz - 2 * wx,
        2 * xz - 2 * wy, 2 * wx + 2 * yz, w2 - x2 - y2 + z2], dim=1).view(-1, 3, 3)
    return R


def convert_pare_to_full_img_cam(pare_cam, bbox_height, bbox_center, img_w, img_h, focal_length, crop_res=224):
    """Crop weak-perspective (s,tx,ty) -> full-image translation (A.5); args evidenced at
    /root/reference/spec/models/hmr.py:104-110, the *200 convention at spec/tester.py:127."""
    s, tx, ty = pare_cam[:, 0], pare_cam[:, 1], pare_cam[:, 2]
    res = crop_res
    r = bbox_height / res
    tz = 2 * focal_length / (r * res * s)
    cx = 2 * (bbox_center[:, 0] - (img_w / 2.)) / (s * bbox_height)
    cy = 2 * (bbox_center[:, 1] - (img_h / 2.)) / (s * bbox_height)
    return torch.stack([tx + cx, ty + cy, tz], dim=-1)


def perspective_projection(points, rotation, translation, cam_intrinsics):
    """(A.6) p = R X + t ; p /= p_z ; uv = (K p)[:2].  K[2,2] may be 0
    (/root/reference/spec/utils/cam_params.py:39-46) -- the last row is dropped."""
    K = cam_intrinsics
    points = torch.einsum('bij,bkj->bki', rotation, points)
    points = points + translation.unsqueeze(1)
    projected = points / points[:, :, -1].unsqueeze(-1)
    projected = torch.einsum('bij,bkj->bki', K, projected.float())
    return projected[:, :, :-1]


# ---- CamCalib decode (these ARE in /root/reference) ---------------------------------------
VFOV_MIN, VFOV_MAX = 0.2617, 2.1      # camcalib/cam_utils.py:55  np.linspace(0.2617, 2.1, 255)
PITCH_MIN, PITCH_MAX = -0.6, 0.6      # camcalib/cam_utils.py:39
ROLL_MIN, ROLL_MAX = -0.6, 0.6        # camcalib/cam_utils.py:133


def soft_idx_to_angle(soft_idx, min, max):
    """camcalib/cam_utils.py:110-111"""
    return (max - min) * ((soft_idx + 1) / 2) + min


def get_softargmax(pred):
    """camcalib/cam_utils.py:114-118"""
    pred = pred.unsqueeze(1)
    k, _ = softargmax1d(pred, normalize_keypoints=True)
    return k.reshape(-1)


def convert_preds_to_angles(pred_vfov, pred_pitch, pred_roll):
    """camcalib/cam_utils.py:121-145, the ``softargmax_l2`` branch (default loss of
    scripts/camcalib_demo.py:227), legacy=False."""
    # np.min/np.max of the float64 linspace bins are exactly the end points
    vfov = soft_idx_to_angle(get_softargmax(pred_vfov), min=np.float64(VFOV_MIN), max=np.float64(VFOV_MAX))
    pitch = soft_idx_to_angle(get_softargmax(pred_pitch), min=np.float64(PITCH_MIN), max=np.float64(PITCH_MAX))
    roll = soft_idx_to_angle(get_softargmax(pred_roll), min=ROLL_MIN, max=ROLL_MAX)
    return vfov.float(), pitch.float(), roll.float()


def cam_params_from_angles(vfov, pitch, roll, img_h, img_w):
    """The CamCalib -> SPEC glue: f_pix (scripts/camcalib_demo.py:127-129) and
    read_cam_params (spec/utils/cam_params.py:24-50), batched and without the pkl round trip.
    Returns cam_rotmat (B,3,3), cam_intrinsics (B,3,3) [K[2,2] left 0], f_pix (B,)."""
    B = vfov.shape[0]
    img_h = torch.as_tensor(img_h, dtype=torch.float32).expand(B) if not torch.is_tensor(img_h) else img_h.float()
    img_w = torch.as_tensor(img_w, dtype=torch.float32).expand(B) if not torch.is_tensor(img_w) else img_w.float()
    # scripts/camcalib_demo.py:127 computes this in NumPy from a float32 0-d array and Python floats: float64 under the
    # NumPy 1.x promotion rules the reference pins; read_cam_params then stores it into a float32 tensor (cam_params.py:43).
    # Checked bit for bit against the unmodified reference code by tests/golden/reference_wrappers.py.
    f_pix = (img_h.double() / 2. / torch.tan(vfov.double() / 2.)).float()
    eul = torch.stack([pitch, torch.zeros_like(pitch), roll], 1).float()
    R = batch_euler2matrix(eul)
    K = torch.zeros(B, 3, 3)
    K[:, 0, 0] = f_pix
    K[:, 1, 1] = f_pix
    K[:, 0, 2] = img_w / 2.
    K[:, 1, 2] = img_h / 2.
    return R, K, f_pix
