"""CPU tests of the SPEC evaluation protocol: the oracle's axis-angle SMPL and 24-joint / camera-frame errors against
scipy and against the committed outputs of the reference's own compute_error.py (tests/golden/reference_eval.npz), and the
CPU-checkable parts of spec_b200.BodyModel / EvalMetrics / SPECErrorEval."""
import numpy as np
import pytest
import torch
from scipy.spatial.transform import Rotation

import spec_b200 as sb
from oracle import body_eval as ob
from oracle import eval_metrics as oe
from oracle.constants import H36M_TO_J14, H36M_TO_J17
from spec_b200.synthetic import synthetic_smpl_data
from tests.golden.reference_eval import FIXTURE, make_inputs


def test_batch_rodrigues_matches_scipy():
    g = np.random.RandomState(0)
    rv = [np.zeros(3), np.array([np.pi - 1e-4, 0, 0]), np.array([0, 0, -np.pi + 1e-3]),
          (np.pi - 1e-3) * np.array([1.0, 2.0, -2.0]) / 3.0]
    rv = np.concatenate([np.stack(rv), g.randn(64, 3) * 1.5])
    got = ob.batch_rodrigues(torch.from_numpy(rv)).numpy()
    ref = Rotation.from_rotvec(rv).as_matrix()
    np.testing.assert_allclose(got, ref, atol=1e-7)
    np.testing.assert_array_equal(ob.batch_rodrigues(torch.zeros(1, 3)).numpy()[0], np.eye(3, dtype=np.float32))


def test_identity_pose_gives_the_shaped_template():
    d = synthetic_smpl_data(0)
    s64 = {k: torch.as_tensor(np.asarray(v)).double() for k, v in d.items() if k != 'parents'}
    betas = torch.from_numpy(np.random.RandomState(1).randn(3, 10))
    v, j = ob.smpl_forward(s64, betas, torch.zeros(3, 3, dtype=torch.float64), torch.zeros(3, 69, dtype=torch.float64))
    shaped = s64['v_template'][None] + torch.einsum('bl,mkl->bmk', betas, s64['shapedirs'])
    # the float32 skinning weights of a vertex sum to 1 within float32 rounding only
    torch.testing.assert_close(v, shaped, atol=1e-7, rtol=0)
    torch.testing.assert_close(j, torch.einsum('bik,ji->bjk', shaped, s64['J_regressor']), atol=1e-12, rtol=0)
    # rotation matrices (pose2rot=False) of the same pose give the same mesh
    R = ob.batch_rodrigues(torch.zeros(72, 3, dtype=torch.float64)).view(3, 24, 3, 3)
    v2, _ = ob.smpl_forward(s64, betas, R[:, :1], R[:, 1:], pose2rot=False)
    torch.testing.assert_close(v2, v, atol=1e-12, rtol=0)


def test_oracle_matches_reference_eval_fixture():
    fx = np.load(FIXTURE)
    x = make_inputs(int(fx['seed']), int(fx['batch']))
    J = torch.from_numpy(x['J_h36m'])
    Jr = torch.as_tensor(x['smpl']['J_regressor']).float()
    pv, gv, R = x['pred_vertices'], x['gt_vertices'], x['cam_rotmat']
    rot = lambda M, v: torch.bmm(M, v.transpose(2, 1)).transpose(2, 1)
    tol = dict(rtol=1e-5, atol=1e-4)                    # millimetres; the reference ran the same float32 ops
    mp, pa, v2v = oe.eval_single(pv, gv, J)
    for k, v in (('w_mpjpe', mp), ('pa_mpjpe', pa), ('w_v2v', v2v)):
        np.testing.assert_allclose(v * 1000, fx[k], err_msg=k, **tol)
    mp, pa, v2v = oe.eval_single(rot(R, pv), rot(R, gv), J)
    for k, v in (('c_mpjpe', mp), ('c_pa_mpjpe', pa), ('c_v2v', v2v)):
        np.testing.assert_allclose(v * 1000, fx[k], err_msg=k, **tol)
    pj = torch.einsum('bik,ji->bjk', [pv, Jr])
    mp, pa = ob.eval_j_24(pj, x['gt_joints'])
    np.testing.assert_allclose(mp * 1000, fx['w_mpjpe_24'], **tol)
    np.testing.assert_allclose(pa * 1000, fx['pa_mpjpe_24'], **tol)
    mp, _ = ob.eval_j_24(torch.einsum('bik,ji->bjk', [rot(R, pv), Jr]), rot(R, x['gt_joints']))
    np.testing.assert_allclose(mp * 1000, fx['c_mpjpe_24'], **tol)
    re, per_joint = ob.reconstruction_error_per_joint((pj - pj[:, [0]]).numpy(), (x['gt_joints'] - x['gt_joints'][:, [0]]).numpy())
    np.testing.assert_allclose(per_joint * 1000, fx['pa_per_joint_24'], **tol)
    np.testing.assert_allclose(re, per_joint.mean(-1))
    # the restated loop body (spec-syn branch) reproduces the same numbers
    out = ob.compute_error_batch(pv, x['gt_pose'], x['gt_betas'], x['pred_cam_rotmat'], x['J_h36m'], x['smpl'], gt_cam_rotmat=R)
    for ours, theirs in (('w_mpjpe', 'w_mpjpe'), ('pa_mpjpe', 'pa_mpjpe'), ('w_v2v', 'w_v2v'), ('mpjpe', 'c_mpjpe'), ('v2v', 'c_v2v'),
                         ('w_mpjpe_24', 'w_mpjpe_24'), ('pa_mpjpe_24', 'pa_mpjpe_24'), ('mpjpe_24', 'c_mpjpe_24')):
        np.testing.assert_allclose(out[ours] * 1000, fx[theirs], err_msg=ours, rtol=1e-4, atol=1e-2)


def test_body_model_buffers_follow_smplx():
    m = sb.BodyModel(smpl_data=synthetic_smpl_data(0))
    shapes = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    assert shapes == {'v_template': (6890, 3), 'shapedirs': (6890, 3, 10), 'posedirs': (207, 20670), 'J_regressor': (24, 6890),
                      'lbs_weights': (6890, 24), 'parents': (24,)}
    assert sb.BodyModel(gender='female').v_template.shape == (6890, 3)          # synthetic stand-in of SMPL_FEMALE
    with pytest.raises(ValueError):
        sb.BodyModel(gender='other')


@pytest.mark.skipif(torch.cuda.is_available(), reason='CPU-only check')
def test_body_model_has_no_cpu_path():
    m = sb.BodyModel(smpl_data=synthetic_smpl_data(0))
    with pytest.raises(RuntimeError, match='no CPU path'):
        m(betas=torch.zeros(1, 10))
    with pytest.raises(RuntimeError, match='no CPU path'):
        sb.joint_errors(torch.zeros(1, 24, 3), torch.zeros(1, 24, 3))


def test_eval_metrics_mapper_length():
    J = np.full((17, 6890), 1.0 / 6890, np.float32)
    assert len(sb.EvalMetrics(J).joint_mapper) == 14
    assert len(sb.EvalMetrics(J, joint_mapper=H36M_TO_J17).joint_mapper) == 17
    for bad in (H36M_TO_J14[:13], H36M_TO_J17 + [0], list(range(24))):
        with pytest.raises(ValueError, match='14.*17'):
            sb.EvalMetrics(J, joint_mapper=bad)


def test_summary_reproduces_the_reference_log_values():
    d = {k: torch.full((4,), float(i + 1) / 1000) for i, k in enumerate(sb.metrics.SPEC_ERROR_KEYS)}
    # w_mpjpe 1, mpjpe 2, pa_mpjpe 3, w_v2v 4, v2v 5, w_mpjpe_24 6, mpjpe_24 7, pa_mpjpe_24 8 (mm)
    s = sb.SPECErrorEval.summary([d, d], 'spec-syn')
    assert list(s) == ['W-MPJPE-24', 'C-MPJPE-24', 'MPJPE-24', 'PA-MPJPE-24', 'W-V2V', 'C-V2V', 'V2V']
    assert [round(v, 6) for v in s.values()] == [6, 6, 7, 8, 4, 4, 5]              # C-* repeat the world-frame values
    s = sb.SPECErrorEval.summary(d, '3dpw-test-cam')
    assert [round(v, 6) for v in s.values()] == [1, 1, 2, 3, 4, 4, 5]
