"""CPU tests of the oracle itself: pinned parts against torchvision, restated tables against the
reference's name tables, domain invariants (SURVEY.md section 4) and the committed golden vectors."""
import os

import numpy as np
import pytest
import torch

from oracle import constants as oc
from oracle import geometry as og
from oracle import models as om
from oracle.head import lbs, SMPL49
from oracle.resnet import resnet50, resnet34
from spec_b200.synthetic import synthetic_smpl_data, synthetic_mean_params
from spec_b200 import constants as pc

GOLD = os.path.join(os.path.dirname(__file__), 'golden')


@pytest.mark.parametrize('name', ['resnet50', 'resnet34'])
def test_resnet_trunk_matches_torchvision(name):
    import torchvision
    torch.manual_seed(0)
    tv = getattr(torchvision.models, name)(weights=None).eval()
    mine = {'resnet50': resnet50, 'resnet34': resnet34}[name]().eval()
    sd = {k: v for k, v in tv.state_dict().items() if not k.startswith('fc.')}
    mine.load_state_dict(sd, strict=True)            # identical key set minus fc
    x = torch.randn(2, 3, 96, 128)
    with torch.no_grad():
        y = tv.layer4(tv.layer3(tv.layer2(tv.layer1(tv.maxpool(tv.relu(tv.bn1(tv.conv1(x))))))))
        z = mine(x)
    assert z.shape == y.shape and torch.equal(z, y)


def test_joint_map_tables():
    # resolved table == [JOINT_MAP[n] for n in JOINT_NAMES] (spec/constants.py:29-105), bit exact
    assert oc.JOINT_MAP_49 == [oc.JOINT_MAP[n] for n in oc.JOINT_NAMES]
    assert len(oc.JOINT_MAP_49) == 49 and max(oc.JOINT_MAP_49) == 53 and min(oc.JOINT_MAP_49) == 0
    assert pc.JOINT_MAP_49 == oc.JOINT_MAP_49                 # product table == oracle table
    assert pc.SMPL_VERTEX_IDS_21 == oc.SMPL_VERTEX_IDS_21 and pc.SMPL_PARENTS == oc.SMPL_PARENTS
    # candidates 35..44 (finger tips) are never selected
    assert not set(range(35, 45)) & set(oc.JOINT_MAP_49)
    assert pc.RECORD_FLOATS == 21294


def test_reference_name_tables_agree():
    """The restated tables equal the reference's own (spec/constants.py), as recorded in tests/golden/reference_tables.json."""
    import json
    with open(os.path.join(GOLD, 'reference_tables.json')) as fh:
        ref = json.load(fh)
    assert ref['JOINT_NAMES'] == oc.JOINT_NAMES and ref['JOINT_MAP'] == oc.JOINT_MAP
    assert ref['H36M_TO_J14'] == oc.H36M_TO_J14 and ref['IMG_NORM_MEAN'] == oc.IMG_NORM_MEAN


def test_rot6d_orthonormal():
    torch.manual_seed(0)
    R = og.rot6d_to_rotmat(torch.randn(16, 144))
    eye = torch.eye(3).expand_as(R)
    assert torch.allclose(R.transpose(1, 2) @ R, eye, atol=1e-5)
    assert torch.allclose(torch.linalg.det(R), torch.ones(R.shape[0]), atol=1e-5)
    # identity 6d -> identity
    I6 = torch.tensor([1., 0, 0, 1, 0, 0]).repeat(1, 24)
    assert torch.allclose(og.rot6d_to_rotmat(I6), torch.eye(3).expand(24, 3, 3))


def test_identity_pose_lbs_returns_shaped_template():
    d = {k: torch.as_tensor(v) for k, v in synthetic_smpl_data(0).items()}
    betas = torch.randn(3, 10)
    R = torch.eye(3).expand(3, 24, 3, 3).contiguous()
    v, J = lbs(betas, R, d['v_template'], d['shapedirs'], d['posedirs'], d['J_regressor'], d['parents'].tolist(), d['lbs_weights'])
    v_shaped = d['v_template'][None] + torch.einsum('bl,mkl->bmk', betas, d['shapedirs'])
    assert torch.allclose(v, v_shaped, atol=2e-6)
    assert torch.allclose(J, torch.einsum('bik,ji->bjk', v_shaped, d['J_regressor']), atol=2e-6)


def _random_rotmats(n, seed):
    g = torch.Generator().manual_seed(seed)
    return og.rot6d_to_rotmat(torch.randn(n, 6, generator=g)).reshape(n, 3, 3)


def test_lbs_root_rotation_is_rigid_about_the_root_joint():
    """Size-independent LBS property (smplx.lbs, A.4): the pose blendshapes only see joints 1..23, so pre-multiplying the
    ROOT rotation by Q moves every vertex and joint rigidly about the rest root joint: v' = Q (v - J0) + J0."""
    d = {k: torch.as_tensor(v) for k, v in synthetic_smpl_data(0).items()}
    B = 3
    betas = torch.randn(B, 10, generator=torch.Generator().manual_seed(1))
    R = _random_rotmats(B * 24, 2).reshape(B, 24, 3, 3)
    Q = _random_rotmats(B, 3)
    args = (d['v_template'], d['shapedirs'], d['posedirs'], d['J_regressor'], d['parents'].tolist(), d['lbs_weights'])
    v, J = lbs(betas, R, *args)
    R2 = R.clone()
    R2[:, 0] = Q @ R[:, 0]
    v2, J2 = lbs(betas, R2, *args)
    v_shaped = d['v_template'][None] + torch.einsum('bl,mkl->bmk', betas, d['shapedirs'])
    J0 = torch.einsum('bik,i->bk', v_shaped, d['J_regressor'][0])[:, None]
    assert torch.allclose(v2, (v - J0) @ Q.transpose(1, 2) + J0, atol=5e-6)
    assert torch.allclose(J2, (J - J0) @ Q.transpose(1, 2) + J0, atol=5e-6)
    assert torch.allclose(J[:, 0], J0[:, 0], atol=2e-6)               # the root joint itself does not move


def test_lbs_against_an_independent_float64_forward_kinematics():
    """The vectorised restatement (oracle/head.py::lbs) against a per-vertex, per-joint float64 loop written from the
    definition: G_j = G_parent(j) [R_j | J_j - J_parent(j)], v = sum_j w_vj G_j [R|t] applied to (v_posed - J_j)."""
    d = {k: np.asarray(v, dtype=np.float64) for k, v in synthetic_smpl_data(0).items() if k != 'parents'}
    parents = [int(p) for p in synthetic_smpl_data(0)['parents']]
    betas = torch.randn(2, 10, generator=torch.Generator().manual_seed(4))
    R = _random_rotmats(2 * 24, 5).reshape(2, 24, 3, 3)
    dt = {k: torch.as_tensor(v).float() for k, v in d.items()}
    v, J = lbs(betas, R, dt['v_template'], dt['shapedirs'], dt['posedirs'], dt['J_regressor'], parents, dt['lbs_weights'])
    vidx = [0, 17, 1234, 3456, 6889]
    for b in range(2):
        be, Rb = betas[b].double().numpy(), R[b].double().numpy()
        v_shaped = d['v_template'] + d['shapedirs'] @ be                      # (6890,3)
        Jr = d['J_regressor'] @ v_shaped                                       # (24,3)
        pf = (Rb[1:] - np.eye(3)).reshape(-1)
        v_posed = v_shaped + (pf @ d['posedirs']).reshape(-1, 3)
        Grot, Gt = [None] * 24, [None] * 24                                    # world rotation / translation of each joint
        for j in range(24):
            if j == 0:
                Grot[j], Gt[j] = Rb[0], Jr[0]
            else:
                pa = parents[j]
                Grot[j] = Grot[pa] @ Rb[j]
                Gt[j] = Grot[pa] @ (Jr[j] - Jr[pa]) + Gt[pa]
        for k in range(24):
            assert np.allclose(J[b, k].numpy(), Gt[k], atol=5e-6)
        for vi in vidx:
            out = np.zeros(3)
            for j in range(24):
                out += d['lbs_weights'][vi, j] * (Grot[j] @ (v_posed[vi] - Jr[j]) + Gt[j])
            assert np.allclose(v[b, vi].numpy(), out, atol=5e-6), (b, vi)


def test_projection_optical_axis_and_k22():
    B = 4
    K = torch.zeros(B, 3, 3); K[:, 0, 0] = K[:, 1, 1] = 1000.; K[:, 0, 2] = 960.; K[:, 1, 2] = 540.   # K[2,2]=0 as cam_params.py
    pts = torch.tensor([[[0., 0., 5.]]]).expand(B, 1, 3)
    uv = og.perspective_projection(pts, torch.eye(3).expand(B, 3, 3), torch.zeros(B, 3), K)
    assert torch.allclose(uv, torch.tensor([960., 540.]).expand(B, 1, 2))


def test_softargmax_uniform_is_midrange():
    z = torch.zeros(2, 256)
    vfov, pitch, roll = og.convert_preds_to_angles(z, z, z)
    assert torch.allclose(vfov, torch.full((2,), (0.2617 + 2.1) / 2), atol=1e-6)
    assert torch.allclose(pitch, torch.zeros(2), atol=1e-6) and torch.allclose(roll, torch.zeros(2), atol=1e-6)


def test_euler_is_rx_rz():
    p, r = torch.tensor([0.3, -0.5]), torch.tensor([-0.2, 0.4])
    R = og.batch_euler2matrix(torch.stack([p, torch.zeros(2), r], 1))
    def rx(a): return torch.tensor([[1, 0, 0], [0, np.cos(a), -np.sin(a)], [0, np.sin(a), np.cos(a)]], dtype=torch.float32)
    def rz(a): return torch.tensor([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]], dtype=torch.float32)
    for i in range(2):
        assert torch.allclose(R[i], rx(float(p[i])) @ rz(float(r[i])), atol=1e-6)


def test_full_img_cam_formula():
    cam = torch.tensor([[0.8, 0.1, -0.2]])
    t = og.convert_pare_to_full_img_cam(cam, torch.tensor([400.]), torch.tensor([[1000., 600.]]),
                                        torch.tensor([1920.]), torch.tensor([1080.]), torch.tensor([1500.]))
    assert torch.allclose(t, torch.tensor([[0.1 + 2 * 40 / (0.8 * 400), -0.2 + 2 * 60 / (0.8 * 400), 2 * 1500 / (400 * 0.8)]]), atol=1e-5)


def test_golden_vectors_reproduce():
    """The committed golden outputs (tests/golden/make_golden.py) are reproduced by the oracle."""
    from tests.golden.make_golden import build_case
    g = np.load(os.path.join(GOLD, 'spec_resnet50_b2.npz'))
    out = build_case()
    for k in g.files:
        np.testing.assert_allclose(out[k], g[k], rtol=0, atol=1e-5, err_msg=k)


def test_procrustes_oracle_invariants():
    """reconstruction_error is invariant to a similarity transform of the prediction (and zero for an exact one)."""
    from oracle.eval_metrics import reconstruction_error
    rng = np.random.RandomState(0)
    S2 = rng.randn(5, 14, 3).astype(np.float32)
    q, _ = np.linalg.qr(rng.randn(3, 3))
    if np.linalg.det(q) < 0:
        q[:, 0] *= -1
    S1 = (1.7 * S2 @ q.T + np.array([0.3, -2.0, 1.0])).astype(np.float32)
    assert reconstruction_error(S1, S2).max() < 1e-5
    noisy = S1 + 0.05 * rng.randn(*S1.shape).astype(np.float32)
    e = reconstruction_error(noisy, S2)
    assert (e > 1e-3).all() and (e < 0.2).all()
