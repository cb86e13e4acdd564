"""GPU tests of the SPEC evaluation protocol (``pytest -m gpu`` on a B200): spec_b200.BodyModel, EvalMetrics (J17 mapper,
per-joint outputs, rotations), joint_errors and SPECErrorEval against the CPU oracle (oracle/body_eval.py) and against
the committed outputs of the reference's own compute_error.py (tests/golden/reference_eval.npz)."""
import numpy as np
import pytest
import torch

import spec_b200 as sb
from oracle import body_eval as ob
from oracle import eval_metrics as oe
from oracle.constants import H36M_TO_J14, H36M_TO_J17
from spec_b200.synthetic import synthetic_smpl_data, synthetic_batch, synthetic_camera
from tests.conftest import make_pair
from tests.golden.reference_eval import FIXTURE, make_inputs

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
# the existing eval tolerances (tests/test_gpu_parity.py::test_eval_metrics_match_oracle)
TOL = {'mpjpe': (1e-5, 1e-4), 'pa': (2e-5, 1e-3), 'v2v': (1e-5, 1e-4)}
KIND = {'w_mpjpe': 'mpjpe', 'mpjpe': 'mpjpe', 'pa_mpjpe': 'pa', 'w_v2v': 'v2v', 'v2v': 'v2v', 'w_mpjpe_24': 'mpjpe',
        'mpjpe_24': 'mpjpe', 'pa_mpjpe_24': 'pa'}


def _close(name, got, ref, atol, rtol=0.0):
    got = torch.as_tensor(got).detach().double().cpu()
    ref = torch.as_tensor(np.asarray(ref)).double()
    assert got.shape == ref.shape, (name, got.shape, ref.shape)
    assert torch.isfinite(got).all(), f'{name}: non-finite output'
    err = (got - ref).abs()
    bad = err > atol + rtol * ref.abs()
    assert not bad.any(), f'{name}: max err {err.max().item():.3e} (tol {atol:g}+{rtol:g}*|ref|), {int(bad.sum())}/{bad.numel()} bad'


def _s64(d):
    return {k: torch.as_tensor(np.asarray(v)).double() for k, v in d.items() if k != 'parents'}


def _params(B, seed):
    g = np.random.RandomState(seed)
    pose = torch.from_numpy(g.randn(B, 72) * 0.5).float()
    betas = torch.from_numpy(g.randn(B, 10)).float()
    return pose, betas


# --------------------------------------------------------------------------------------- body model
@pytest.mark.parametrize('B', [1, 37, 257])
@pytest.mark.parametrize('pose2rot', [True, False])
def test_body_model_matches_oracle(B, pose2rot):
    d = synthetic_smpl_data(0)
    m = sb.BodyModel(smpl_data=d).to(DEV)
    pose, betas = _params(B, 100 + B)
    if pose2rot:
        got = m(betas=betas.to(DEV), global_orient=pose[:, :3].to(DEV), body_pose=pose[:, 3:].to(DEV))
        rv, rj = ob.smpl_forward(_s64(d), betas.double(), pose[:, :3].double(), pose[:, 3:].double())
    else:
        R = ob.batch_rodrigues(pose.reshape(-1, 3)).reshape(B, 24, 3, 3)
        got = m(betas=betas.to(DEV), global_orient=R[:, :1].to(DEV), body_pose=R[:, 1:].to(DEV), pose2rot=False)
        rv, rj = ob.smpl_forward(_s64(d), betas.double(), R[:, :1].double(), R[:, 1:].double(), pose2rot=False)
    assert got.vertices.shape == (B, 6890, 3) and got.joints.shape == (B, 24, 3)
    _close('vertices', got.vertices, rv, 1e-5)
    _close('joints24', got.joints, rj, 1e-5)


def test_body_model_reproduces_the_hmr_tail_and_leaves_it_alone():
    """BodyModel(pose2rot=False) on an HMR forward's pred_pose / pred_shape gives its smpl_vertices bit for bit (same kernels);
    creating body handles does not disturb the live HMR handle (its joint-map / vertex-id tables)."""
    hmr, _ = make_pair('resnet50', seed=0)
    hmr.backbone.set_precision('fp32')
    hmr.to(DEV)
    b = synthetic_batch(5, seed=3, device=DEV)
    from oracle import geometry as og
    vfov, pitch, roll = synthetic_camera(5, seed=3)
    R, K, _ = og.cam_params_from_angles(vfov, pitch, roll, b['img_h'].cpu(), b['img_w'].cpu())
    run = lambda: hmr(b['images'], R.to(DEV), K.to(DEV), b['bbox_scale'], b['bbox_center'], b['img_w'], b['img_h'])
    out = run()
    m = sb.BodyModel(smpl_data=synthetic_smpl_data(0)).to(DEV)
    f = sb.BodyModel(smpl_data=synthetic_smpl_data(5)).to(DEV)
    got = m(betas=out['pred_shape'], global_orient=out['pred_pose'][:, :1], body_pose=out['pred_pose'][:, 1:], pose2rot=False)
    f(betas=out['pred_shape'], global_orient=out['pred_pose'][:, :1], body_pose=out['pred_pose'][:, 1:], pose2rot=False)
    assert torch.equal(got.vertices, out['smpl_vertices'])
    again = run()
    for k in out:
        assert torch.equal(out[k], again[k]), k


def test_coexisting_body_handles():
    dn, dfem = synthetic_smpl_data(0), synthetic_smpl_data(2)
    neutral, female = sb.BodyModel(smpl_data=dn).to(DEV), sb.BodyModel(smpl_data=dfem, gender='female').to(DEV)
    pose, betas = _params(19, 7)
    args = dict(betas=betas.to(DEV), global_orient=pose[:, :3].to(DEV), body_pose=pose[:, 3:].to(DEV))
    a1 = neutral(**args)
    b1 = female(**args)
    a2 = neutral(**args)
    assert torch.equal(a1.vertices, a2.vertices)
    assert (a1.vertices - b1.vertices).abs().max() > 1e-2
    for out, d in ((a1, dn), (b1, dfem)):
        rv, rj = ob.smpl_forward(_s64(d), betas.double(), pose[:, :3].double(), pose[:, 3:].double())
        _close('vertices', out.vertices, rv, 1e-5)
        _close('joints24', out.joints, rj, 1e-5)


# --------------------------------------------------------------------------------------- SPECErrorEval
def _evaluator(x):
    bm = sb.BodyModel(smpl_data=x['smpl']).to(DEV)
    return sb.SPECErrorEval(x['J_h36m'], bm).to(DEV)


def _run(ev, x, branch, pred=None):
    pred = x['pred_vertices'].to(DEV) if pred is None else pred
    common = (pred, x['gt_pose'].to(DEV), x['gt_betas'].to(DEV), x['pred_cam_rotmat'].to(DEV))
    if branch == 'spec-syn':
        return ev.batch(*common, gt_cam_rotmat=x['cam_rotmat'].to(DEV))
    return ev.batch(*common, gt_pose_cam=x['gt_pose_cam'].to(DEV))


@pytest.mark.parametrize('branch', ['spec-syn', 'pose_cam'])
def test_spec_error_eval_matches_oracle(branch):
    x = make_inputs(seed=11, batch=37)
    got = _run(_evaluator(x), x, branch)
    kw = dict(gt_cam_rotmat=x['cam_rotmat']) if branch == 'spec-syn' else dict(gt_pose_cam=x['gt_pose_cam'])
    ref = ob.compute_error_batch(x['pred_vertices'], x['gt_pose'], x['gt_betas'], x['pred_cam_rotmat'], x['J_h36m'], x['smpl'], **kw)
    assert set(got) == set(sb.metrics.SPEC_ERROR_KEYS)
    for k in sb.metrics.SPEC_ERROR_KEYS:
        _close(f'{branch}:{k}', got[k], ref[k], *TOL[KIND[k]])


def test_spec_error_eval_matches_reference_fixture():
    fx = np.load(FIXTURE)
    x = make_inputs(int(fx['seed']), int(fx['batch']))
    got = _run(_evaluator(x), x, 'spec-syn')
    for ours, theirs in (('w_mpjpe', 'w_mpjpe'), ('pa_mpjpe', 'pa_mpjpe'), ('w_v2v', 'w_v2v'), ('mpjpe', 'c_mpjpe'), ('v2v', 'c_v2v'),
                         ('w_mpjpe_24', 'w_mpjpe_24'), ('pa_mpjpe_24', 'pa_mpjpe_24'), ('mpjpe_24', 'c_mpjpe_24')):
        atol, rtol = TOL[KIND[ours]]
        _close(ours, got[ours], fx[theirs] / 1000.0, atol, rtol)
    s = sb.SPECErrorEval.summary(got, 'spec-syn')
    assert abs(s['PA-MPJPE-24'] - fx['pa_mpjpe_24'].mean()) < 1e-2


def test_determinism_graph_capture_and_packed_input():
    x = make_inputs(seed=12, batch=33)
    ev = _evaluator(x)
    a = _run(ev, x, 'pose_cam')
    b = _run(ev, x, 'pose_cam')
    for k in a:
        assert torch.equal(a[k], b[k]), k
    # a packed per-image record (the multi-GPU all-gather buffer): the strided smpl_vertices view goes in as it is
    rec = torch.zeros(33, sb.pipeline.RECORD_FLOATS, device=DEV)
    view = sb.unpack_record(rec)['smpl_vertices']
    view.copy_(x['pred_vertices'].to(DEV))
    assert view.stride(0) != 6890 * 3
    c = _run(ev, x, 'pose_cam', pred=view)
    for k in a:
        assert torch.equal(a[k], c[k]), k
    # CUDA-graph capture after the warm-up above: replay equals eager
    st = {k: x[k].to(DEV) for k in ('pred_vertices', 'gt_pose', 'gt_betas', 'pred_cam_rotmat', 'cam_rotmat')}
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        outs = ev.batch(st['pred_vertices'], st['gt_pose'], st['gt_betas'], st['pred_cam_rotmat'], gt_cam_rotmat=st['cam_rotmat'])
    eager = _run(ev, x, 'spec-syn')
    g.replay()
    torch.cuda.synchronize()
    for k in eager:
        assert torch.equal(outs[k], eager[k]), k


# --------------------------------------------------------------------------------------- per-joint, J17, reflection
def _meshes(B, seed):
    x = make_inputs(seed=seed, batch=B)
    return x, torch.from_numpy(x['J_h36m'])


def test_per_joint_and_j17_match_oracle():
    B = 29
    x, J = _meshes(B, 13)
    pv, gv = x['pred_vertices'], x['gt_vertices']             # every third prediction is reflected: det < 0 branch
    Jb = J[None].expand(B, -1, -1)
    for mapper in (H36M_TO_J14, H36M_TO_J17):
        n = len(mapper)
        pk = torch.matmul(Jb, pv)
        pk = pk[:, mapper] - pk[:, [0]]
        gk = torch.matmul(Jb, gv)
        gk = gk[:, mapper] - gk[:, [0]]
        m = sb.EvalMetrics(x['J_h36m'], joint_mapper=mapper).to(DEV)
        got = m(pv.to(DEV), gt_keypoints_3d=gk.to(DEV), gt_vertices=gv.to(DEV), per_joint=True)
        re, re_pj = ob.reconstruction_error_per_joint(pk.numpy(), gk.numpy())
        mp_pj = torch.sqrt(((pk - gk) ** 2).sum(-1))
        _close(f'J{n} mpjpe', got['mpjpe'], mp_pj.mean(-1), *TOL['mpjpe'])
        _close(f'J{n} mpjpe_pj', got['mpjpe_per_joint'], mp_pj, *TOL['mpjpe'])
        _close(f'J{n} pa', got['pa_mpjpe'], re, *TOL['pa'])
        _close(f'J{n} pa_pj', got['pa_mpjpe_per_joint'], re_pj, *TOL['pa'])
        _close(f'J{n} v2v', got['v2v'], oe.compute_error_verts(pv.numpy(), gv.numpy()), *TOL['v2v'])
        _close(f'J{n} pred_kp', got['pred_keypoints_3d'], pk, 1e-5)
        if n == 17:
            with pytest.raises(ValueError):
                m(pv.to(DEV), gt_keypoints_3d=gk[:, :14].to(DEV))
    # the 14-joint results are unchanged by per_joint=True
    m14 = sb.EvalMetrics(x['J_h36m']).to(DEV)
    a = m14(pv.to(DEV), gt_vertices=gv.to(DEV), center_v2v=True)
    b = m14(pv.to(DEV), gt_vertices=gv.to(DEV), center_v2v=True, per_joint=True)
    for k in ('mpjpe', 'pa_mpjpe', 'v2v', 'pred_keypoints_3d'):
        assert torch.equal(a[k], b[k]), k


@pytest.mark.parametrize('center', [True, False])
def test_joint_errors_24_match_oracle(center):
    B = 41
    x, _ = _meshes(B, 14)
    Jr = torch.as_tensor(x['smpl']['J_regressor']).float()
    pj = torch.einsum('bik,ji->bjk', [x['pred_vertices'], Jr])
    gj = x['gt_joints']
    R = x['cam_rotmat']
    got = sb.joint_errors(pj.to(DEV), gj.to(DEV), center=center, per_joint=True, rot_pred=R.to(DEV), rot_gt=R.to(DEV))
    rp = torch.bmm(R, pj.transpose(1, 2)).transpose(1, 2)
    rg = torch.bmm(R, gj.transpose(1, 2)).transpose(1, 2)
    if center:
        rp, rg = rp - rp[:, [0]], rg - rg[:, [0]]
    re, re_pj = ob.reconstruction_error_per_joint(rp.numpy(), rg.numpy())
    mp_pj = torch.sqrt(((rp - rg) ** 2).sum(-1))
    _close('mpjpe', got['mpjpe'], mp_pj.mean(-1), *TOL['mpjpe'])
    _close('mpjpe_pj', got['mpjpe_per_joint'], mp_pj, *TOL['mpjpe'])
    _close('pa', got['pa_mpjpe'], re, *TOL['pa'])
    _close('pa_pj', got['pa_mpjpe_per_joint'], re_pj, *TOL['pa'])
    # regression of the 24 joints (with and without a rotation) on the device
    bm = sb.BodyModel(smpl_data=x['smpl']).to(DEV)
    _close('regress', bm.regress_joints(x['pred_vertices'].to(DEV)), pj, 1e-5)
    _close('regress rot', bm.regress_joints(x['pred_vertices'].to(DEV), rot=R.to(DEV)), rp if not center else
           torch.bmm(R, pj.transpose(1, 2)).transpose(1, 2), 1e-5)
