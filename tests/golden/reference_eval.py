"""Runs the UNMODIFIED evaluation functions of the original SPEC repository -- ``eval_single`` and ``eval_j_24`` of
spec/utils/compute_error.py -- on seeded synthetic inputs and writes what they returned to tests/golden/reference_eval.npz.

compute_error.py imports ``smplx``, ``pare.models``, ``pare.core.constants``, ``pare.utils.eval_utils`` and (relatively)
``spec.config``; none of the first four is installable offline.  ``install_stubs`` puts stand-ins for exactly those names
into ``sys.modules`` -- backed by the oracle (oracle/body_eval.py, oracle/eval_metrics.py) -- and the file is then executed
from where it lies as ``spec.utils.compute_error`` (importlib, by path; nothing is copied).  ``compute_error()`` itself
hard-codes ``device='cuda'`` and reads dataset files, so its loop body is restated in ``oracle.body_eval.compute_error_batch``;
this fixture pins the two functions that loop body calls.

    python -m tests.golden.reference_eval <path to a SPEC checkout>          # regenerate the fixture

The inputs are regenerated from seeds by ``make_inputs`` (tests/test_eval_protocol.py and tests/test_gpu_eval_protocol.py
call it); only the reference's outputs are committed.
"""
import importlib.util
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.dirname(os.path.abspath(__file__))
FIXTURE = os.path.join(GOLDEN, 'reference_eval.npz')
SEED, BATCH = 7, 8
_STUB_NAMES = ['smplx', 'pare', 'pare.models', 'pare.core', 'pare.core.constants', 'pare.utils', 'pare.utils.eval_utils',
               'spec', 'spec.config', 'spec.utils']


def _rotations(g, n, scale):
    from oracle.body_eval import batch_rodrigues
    return batch_rodrigues(torch.from_numpy(g.randn(n, 3) * scale)).float()


def make_inputs(seed=SEED, batch=BATCH):
    """Seeded protocol inputs (float32 CPU tensors): SMPL meshes from random axis-angle poses (the synthetic SMPL constants of
    spec_b200.synthetic, computed in float64), predictions that are rotated, scaled, shifted, noisy and -- for every third
    image -- reflected versions of them, a non-trivial camera rotation per image and a seeded H36M-like regressor."""
    from oracle.body_eval import smpl_forward
    from spec_b200.synthetic import synthetic_smpl_data
    g = np.random.RandomState(seed)
    smpl = synthetic_smpl_data(0)
    J = g.rand(17, 6890) ** 8
    J_h36m = (J / J.sum(1, keepdims=True)).astype(np.float32)
    gt_pose = (g.randn(batch, 72) * 0.4).astype(np.float32)
    gt_pose_cam = gt_pose.copy()
    gt_pose_cam[:, :3] = (g.randn(batch, 3) * 0.8).astype(np.float32)
    gt_betas = (g.randn(batch, 10) * 1.0).astype(np.float32)
    s64 = {k: torch.as_tensor(np.asarray(v)).double() for k, v in smpl.items() if k != 'parents'}
    gv, gj = smpl_forward(s64, torch.from_numpy(gt_betas).double(), torch.from_numpy(gt_pose[:, :3]).double(),
                          torch.from_numpy(gt_pose[:, 3:]).double())
    gt_vertices, gt_joints = gv.float(), gj.float()
    R = _rotations(g, batch, 0.3)
    scale = torch.from_numpy(1.0 + 0.1 * g.randn(batch, 1, 1)).float()
    shift = torch.from_numpy(0.05 * g.randn(batch, 1, 3)).float()
    noise = torch.from_numpy(0.01 * g.randn(batch, 6890, 3)).float()
    pred = scale * torch.bmm(gt_vertices, R.transpose(1, 2)) + shift + noise
    refl = torch.ones(batch, 1, 3)
    refl[::3, 0, 0] = -1.0
    pred_vertices = (pred * refl).contiguous()
    cam_rotmat = _rotations(g, batch, 0.6)
    pred_cam_rotmat = torch.bmm(_rotations(g, batch, 0.05), cam_rotmat)
    return {'smpl': smpl, 'J_h36m': J_h36m, 'gt_pose': torch.from_numpy(gt_pose), 'gt_pose_cam': torch.from_numpy(gt_pose_cam),
            'gt_betas': torch.from_numpy(gt_betas), 'gt_vertices': gt_vertices, 'gt_joints': gt_joints,
            'pred_vertices': pred_vertices, 'cam_rotmat': cam_rotmat, 'pred_cam_rotmat': pred_cam_rotmat}


def install_stubs():
    """sys.modules stand-ins for the names compute_error.py imports (and nothing else); returns what they replaced."""
    from oracle import eval_metrics as oe, body_eval as ob
    from oracle.constants import H36M_TO_J14
    from spec_b200.synthetic import synthetic_smpl_data
    saved = {n: sys.modules.get(n) for n in _STUB_NAMES}
    mods = {n: types.ModuleType(n) for n in _STUB_NAMES}
    for n in _STUB_NAMES:
        if '.' in n:
            parent, child = n.rsplit('.', 1)
            setattr(mods[parent], child, mods[n])
        mods[n].__path__ = []

    class SMPL(torch.nn.Module):                          # smplx.SMPL / pare.models.SMPL as compute_error.py:115-127 builds them
        def __init__(self, model_path=None, batch_size=1, create_transl=False, create_global_orient=True, **kw):
            super().__init__()
            d = synthetic_smpl_data(0)
            for k in ('v_template', 'shapedirs', 'posedirs', 'J_regressor', 'lbs_weights'):
                self.register_buffer(k, torch.as_tensor(d[k]).float())

        def forward(self, betas=None, body_pose=None, global_orient=None, pose2rot=True, **kw):
            v, j = ob.smpl_forward(self, betas, global_orient, body_pose, pose2rot=pose2rot)
            return types.SimpleNamespace(vertices=v, joints=j)

    def reconstruction_error(S1, S2, reduction='mean'):  # [UPSTREAM-RECALLED] pare.utils.eval_utils
        re, re_per_joint = ob.reconstruction_error_per_joint(S1, S2)
        if reduction == 'mean':
            re = re.mean()
        elif reduction == 'sum':
            re = re.sum()
        return re, re_per_joint

    mods['smplx'].SMPL = SMPL
    mods['pare.models'].SMPL = SMPL
    mods['pare.core.constants'].H36M_TO_J14 = H36M_TO_J14
    mods['pare.utils.eval_utils'].compute_error_verts = oe.compute_error_verts
    mods['pare.utils.eval_utils'].reconstruction_error = reconstruction_error
    mods['spec.config'].DATASET_FILES = [{}]
    mods['spec.config'].SMPL_MODEL_DIR = 'data/body_models/smpl'
    sys.modules.update(mods)
    return saved


def load_compute_error(ref_root):
    saved = install_stubs()
    try:
        spec = importlib.util.spec_from_file_location('spec.utils.compute_error', os.path.join(ref_root, 'spec/utils/compute_error.py'))
        mod = importlib.util.module_from_spec(spec)
        sys.modules['spec.utils.compute_error'] = mod
        spec.loader.exec_module(mod)
        return mod, saved
    except BaseException:
        _restore(saved)
        raise


def _restore(saved):
    sys.modules.pop('spec.utils.compute_error', None)
    for n, m in saved.items():
        if m is None:
            sys.modules.pop(n, None)
        else:
            sys.modules[n] = m


def run_reference(ref_root, seed=SEED, batch=BATCH):
    """The reference's eval_single / eval_j_24 on make_inputs(seed): world frame, camera frame (the spec-syn rotation of
    both meshes) and the 24-joint errors; returns the arrays written to FIXTURE (millimetres, as the reference returns)."""
    ce, saved = load_compute_error(ref_root)
    try:
        x = make_inputs(seed, batch)
        Jb = torch.from_numpy(x['J_h36m'])[None].expand(1, -1, -1)
        Jr = torch.as_tensor(x['smpl']['J_regressor']).float()
        pv, gv, R = x['pred_vertices'], x['gt_vertices'], x['cam_rotmat']
        rot = lambda M, v: torch.bmm(M, v.transpose(2, 1)).transpose(2, 1)
        out = {}
        out['w_mpjpe'], out['pa_mpjpe'], out['w_v2v'] = ce.eval_single(pv, gv, Jb)
        out['c_mpjpe'], out['c_pa_mpjpe'], out['c_v2v'] = ce.eval_single(rot(R, pv), rot(R, gv), Jb)
        pj = torch.einsum('bik,ji->bjk', [pv, Jr])
        out['w_mpjpe_24'], out['pa_mpjpe_24'] = ce.eval_j_24(pj, x['gt_joints'])
        out['c_mpjpe_24'], _ = ce.eval_j_24(torch.einsum('bik,ji->bjk', [rot(R, pv), Jr]), rot(R, x['gt_joints']))
        # the per-joint distances eval_j_24's reconstruction_error(reduction=None) computed (it returns only the mean)
        p0 = pj - pj[:, [0]]
        g0 = x['gt_joints'] - x['gt_joints'][:, [0]]
        out['pa_per_joint_24'] = sys.modules['pare.utils.eval_utils'].reconstruction_error(p0.numpy(), g0.numpy(), reduction=None)[1] * 1000
        return {k: np.asarray(v, dtype=np.float64) for k, v in out.items()}
    finally:
        _restore(saved)


if __name__ == '__main__':
    if len(sys.argv) != 2:
        sys.exit('usage: python -m tests.golden.reference_eval <path to a SPEC checkout>')
    res = run_reference(sys.argv[1])
    np.savez(FIXTURE, seed=np.int64(SEED), batch=np.int64(BATCH), **res)
    for k, v in res.items():
        print(f'{k:16s} {np.array2string(v.reshape(-1)[:4], precision=4)}')
    print('wrote', FIXTURE)
