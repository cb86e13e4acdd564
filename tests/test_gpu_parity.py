"""GPU parity tests (run on a B200 with ``pytest -m gpu``): the CUDA path, called through the C ABI, against
the CPU oracle on the same seeded inputs.

Tolerances (north star, BASELINE.json): fp32 mode -- vertices <= 1e-3, camera parameters <= 1e-5, joint
index tables bit-exact.  16-bit tensor-core modes are compared with the precision-matched oracle
(oracle/lowp.py), tolerance stated per test.
"""
import numpy as np
import pytest
import torch

import spec_b200 as sb
from spec_b200.backbone import Trunk
from spec_b200.synthetic import synthetic_batch, synthetic_camera, randomize_module_
from spec_b200.constants import JOINT_MAP_49, SMPL_VERTEX_IDS_21
from oracle import geometry as og
from oracle import lowp
from oracle.models import spec_full_forward
from tests.conftest import make_pair, make_camcalib_pair

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
TORCH_DT = {'fp32': torch.float32, 'bf16': torch.bfloat16, 'fp16': torch.float16}


def _assert_close(name, got, ref, atol, rtol=0.0):
    got, ref = got.detach().float().cpu(), ref.detach().float().cpu()
    assert got.shape == ref.shape, (name, got.shape, ref.shape)
    assert torch.isfinite(got).all(), f'{name}: non-finite output'
    err = (got - ref).abs()
    tol = atol + rtol * ref.abs()
    bad = err > tol
    assert not bad.any(), f'{name}: max err {err.max().item():.3e} (tol {atol:g}+{rtol:g}*|ref|), {int(bad.sum())}/{bad.numel()} bad, ref scale {ref.abs().mean().item():.3e}'


# --------------------------------------------------------------------------------------- building blocks
def test_linear_f32_matches_torch():
    import ctypes
    from spec_b200 import _lib
    torch.manual_seed(0)
    for (M, N, K) in [(256, 1024, 2048), (7, 157, 1024), (33, 768, 512), (1, 64, 164)]:
        a = torch.randn(M, K, device=DEV)
        w = torch.randn(N, K, device=DEV) / K ** 0.5
        b = torch.randn(N, device=DEV)
        out = torch.empty(M, N, device=DEV)
        _lib.check(_lib.lib().specb200_linear_f32(a.data_ptr(), K, w.data_ptr(), K, b.data_ptr(), out.data_ptr(), N, M, N, K,
                                                  torch.cuda.current_stream().cuda_stream))
        ref = (a.double() @ w.double().t() + b.double()).float()
        _assert_close(f'linear {M}x{N}x{K}', out, ref, atol=2e-5, rtol=1e-5)


def _mini(cmid, cout, k, stride, pad, res, precision):
    def builder(root, P):
        a = P.conv(root, 0, 3, cmid, 3, 1, 1, 'c0', 'b0', True)
        r = P.conv(root, a, cmid, cout, k, stride, pad, 'cr', 'br', False) if res else None
        b = P.conv(root, a, cmid, cout, k, stride, pad, 'c1', 'b1', True, res=r)
        return b, cout
    t = Trunk('custom', builder=builder, precision=precision)
    randomize_module_(t, 3)
    return t


def _mini_ref(t, x, dtype, res):
    a = lowp.conv_bn_act(lowp._rnd(x, dtype), t.c0, t.b0, dtype, True)
    r = lowp.conv_bn_act(a, t.cr, t.br, dtype, False) if res else None
    return lowp.conv_bn_act(a, t.c1, t.b1, dtype, True, res=r)


CONV_CASES = [
    # cmid, cout, k, stride, pad, res, H, W, B      what it exercises
    (64, 64, 1, 1, 0, False, 16, 16, 2),            # 1x1: tiled TMA A, 1 k-block, BLOCK_N=64, persistent kernel
    (256, 128, 1, 1, 0, True, 12, 20, 3),           # 1x1 tiled TMA A, 4 k-blocks, BLOCK_N=128, persistent kernel, residual, ragged M
    (64, 64, 3, 1, 1, False, 14, 14, 2),            # halo kernel, 8x14 tiles, padding
    (128, 128, 3, 2, 1, False, 15, 17, 2),          # 3x3 stride 2, odd sizes: TMA im2col A, one-tile kernel
    (64, 256, 1, 2, 0, False, 14, 14, 2),           # strided 1x1 (downsample): TMA im2col A, persistent kernel, BLOCK_N=128 (K=64)
    (32, 32, 3, 1, 1, True, 10, 10, 2),             # Cin=32 (HRNet), even width: pixel-pair view as a 64->64 conv, too narrow for the halo kernel -> im2col one-tile kernel
    (64, 512, 1, 1, 0, False, 7, 7, 5),             # persistent kernel, 4 N tiles
    (64, 64, 3, 1, 1, True, 9, 23, 3),              # halo kernel, ragged 4x30 tiles, residual
    (128, 128, 3, 1, 1, True, 20, 30, 2),           # 3x3 TMA im2col A, one-tile kernel, BLOCK_N=128, residual
    (256, 256, 3, 1, 1, False, 16, 17, 1),          # CTA-pair kernel, im2col A, N=256, 3 m-tiles: the second pair tile is half outside M
    (256, 512, 1, 1, 0, True, 9, 9, 3),             # CTA-pair kernel, tiled A, N=256 tiles, residual, ragged M
    (32, 32, 3, 1, 1, True, 9, 11, 2),              # Cin=32 on an ODD width: the pixel-pair view does not apply -> gather-kernel fallback
    (512, 512, 3, 1, 1, False, 14, 14, 56),         # CTA-pair kernel, im2col A, K=4608: 43 pair-tiles x 2 n-tiles = 86 tiles on 74 clusters (multi-tile loop)
    (1024, 2048, 1, 1, 0, True, 7, 7, 200),         # CTA-pair kernel, 1x1: 39 pair-tiles x 8 n-tiles = 312 tiles on 74 clusters: the multi-tile loop + TMEM phase flips
]


@pytest.mark.parametrize('precision', ['bf16', 'fp16', 'fp32'])
@pytest.mark.parametrize('case', CONV_CASES, ids=[f'c{c[0]}-{c[1]}k{c[2]}s{c[3]}h{c[6]}' for c in CONV_CASES])
def test_conv_kernels(case, precision):
    cmid, cout, k, stride, pad, res, H, W, B = case
    t = _mini(cmid, cout, k, stride, pad, res, precision)
    torch.manual_seed(1)
    x = torch.randn(B, 3, H, W)
    ref = _mini_ref(t, x, TORCH_DT[precision], res)
    got = t.to(DEV)(x.to(DEV))
    scale = ref.abs().mean().item()
    if precision == 'fp32':
        _assert_close('conv fp32', got, ref, atol=1e-4 * max(scale, 1.0), rtol=1e-4)
    else:
        # one 16-bit ulp (2^-8 bf16 / 2^-11 fp16) of slack for rounding-boundary flips from summation order ...
        _assert_close(f'conv {precision}', got, ref, atol=0.02 * scale, rtol=0.02)
        # ... which are RARE on identical inputs: on average the kernel agrees with the emulation to ~1e-6 (a wrong rounding
        # point, a missing bias or a mis-addressed tap would be >= 1e-2)
        rel = ((got.cpu() - ref).abs().mean() / scale).item()
        assert rel < 2e-4, rel


BNECK_CASES = [
    # H, W, B                what it exercises
    (56, 56, 8),           # the layer1 geometry: 7 x 4 tiles per image, 224 tiles on 148 persistent CTAs (multi-tile loop, x ring wrap)
    (37, 45, 3),           # ragged tiles: clipped right / bottom borders, out-of-image halo rows zeroed
    (8, 14, 1),            # exactly one tile
    (5, 9, 2),             # smaller than a tile
]


@pytest.mark.parametrize('precision', ['bf16', 'fp16'])
@pytest.mark.parametrize('case', BNECK_CASES, ids=[f'h{c[0]}w{c[1]}b{c[2]}' for c in BNECK_CASES])
def test_fused_bottleneck_kernel(case, precision):
    """bottleneck64_kernel (conv_bneck.cu): a downsample block (64 -> 256) followed by two identity blocks (256 -> 256), each ONE
    launch, against the precision-matched oracle that rounds after every conv exactly where the un-fused kernels do."""
    from spec_b200.backbone import _bottleneck
    from spec_b200 import _lib
    H, W, B = case

    def builder(root, P):
        x = P.conv(root, 0, 3, 64, 3, 1, 1, 'c0', 'b0', True)
        x = _bottleneck(P, root, x, 'blk0.', 64, 64, 1, True)
        x = _bottleneck(P, root, x, 'blk1.', 256, 64, 1, False)
        x = _bottleneck(P, root, x, 'blk2.', 256, 64, 1, False)
        return x, 256
    t = Trunk('custom', builder=builder, precision=precision)
    randomize_module_(t, 7)
    dt = TORCH_DT[precision]
    torch.manual_seed(2)
    x = torch.randn(B, 3, H, W)

    def block(pre, a, ds):
        g = lambda n: getattr(getattr(t, pre), n)
        # the downsample conv shares conv3's fp32 accumulator inside the fused kernel: its output is not rounded on its own
        idt = lowp.conv_bn_act(a, g('downsample')._modules['0'], g('downsample')._modules['1'], dt, False, keep_fp32=True) if ds else a
        u = lowp.conv_bn_act(a, g('conv1'), g('bn1'), dt, True)
        u = lowp.conv_bn_act(u, g('conv2'), g('bn2'), dt, True)
        return lowp.conv_bn_act(u, g('conv3'), g('bn3'), dt, True, res=idt)
    a = lowp.conv_bn_act(lowp._rnd(x, dt), t.c0, t.b0, dt, True)
    ref = block('blk2', block('blk1', block('blk0', a, True), False), False)
    got = t.to(DEV)(x.to(DEV))
    assert _lib.lib().specb200_trunk_num_fused_bottlenecks(t._handle) == 3          # the fused kernel really ran
    assert t.last_launches() == 2 + 3 + 1                                              # image conversion, stem conv, 3 blocks, layout
    scale = ref.abs().mean().item()
    err = (got.cpu() - ref).abs()
    # three chained blocks: a rounding-boundary flip in block 0 is amplified by blocks 1-2 (test_layerwise_lowp_profile), so a
    # handful of elements may sit a few ulps off; the bulk must agree to ~1e-5
    assert (err > 0.02 * scale + 0.02 * ref.abs()).float().mean().item() < 1e-5
    assert err.max().item() < 0.25 * max(scale, ref.abs().max().item() * 0.05), err.max().item()
    rel = (err.mean() / scale).item()
    assert rel < 2e-3, rel


def test_stem_conv7x7_and_maxpool():
    for precision, (H, W) in (('bf16', (64, 96)), ('bf16', (70, 100)), ('fp16', (37, 53)), ('fp32', (64, 96))):
        def builder(root, P):
            x = P.conv(root, 0, 3, 64, 7, 2, 3, 'conv1', 'bn1', True)
            y = P.op(2, x, P.new(64))
            return y, 64
        t = Trunk('custom', builder=builder, precision=precision)
        randomize_module_(t, 5)
        x = torch.randn(3, 3, H, W)          # odd sizes: partial 8x16 tiles of the dedicated stem kernel
        dt = TORCH_DT[precision]
        ref = torch.nn.functional.max_pool2d(lowp.conv_bn_act(lowp._rnd(x, dt), t.conv1, t.bn1, dt, True), 3, 2, 1)
        got = t.to(DEV)(x.to(DEV))
        s = ref.abs().mean().item()
        _assert_close('stem ' + precision, got, ref, atol=(1e-4 if precision == 'fp32' else 0.02) * s, rtol=1e-4 if precision == 'fp32' else 0.02)


# --------------------------------------------------------------------------------------- full path, fp32 parity mode
def _run_product(cc, hmr, b, precision, graph=False):
    cc.backbone.set_precision(precision)
    hmr.backbone.set_precision(precision)
    cc.to(DEV), hmr.to(DEV)
    pipe = sb.SPECPipeline(cc, hmr, use_graph=graph)
    bd = {k: v.to(DEV) for k, v in b.items()}
    out = pipe(bd['images'], bd['bbox_scale'], bd['bbox_center'], bd['img_w'], bd['img_h'])
    torch.cuda.synchronize()
    return {k: v.clone() for k, v in out.items()}


@pytest.fixture(scope='module')
def models():
    hmr, hmr_ref = make_pair('resnet50', seed=0)
    cc, cc_ref = make_camcalib_pair('resnet50', seed=1)
    return cc, cc_ref, hmr, hmr_ref


def test_full_forward_fp32_parity(models):
    cc, cc_ref, hmr, hmr_ref = models
    b = synthetic_batch(4, seed=0)
    ref = spec_full_forward(cc_ref, hmr_ref, b['images'], b['bbox_scale'], b['bbox_center'], b['img_w'], b['img_h'])
    got = _run_product(cc, hmr, b, 'fp32')
    # camera parameters <= 1e-5 (north star)
    ang_ref = torch.stack([ref['cam_vfov'], ref['cam_pitch'], ref['cam_roll']], 1)
    _assert_close('cam angles', got['cam_angles'], ang_ref, atol=1e-5)
    _assert_close('pred_cam', got['pred_cam'], ref['pred_cam'], atol=1e-5, rtol=1e-5)
    # vertices <= 1e-3 (north star); the rest at comparable relative accuracy
    _assert_close('smpl_vertices', got['smpl_vertices'], ref['smpl_vertices'], atol=1e-3)
    _assert_close('smpl_joints3d', got['smpl_joints3d'], ref['smpl_joints3d'], atol=1e-3)
    _assert_close('pred_pose', got['pred_pose'], ref['pred_pose'], atol=1e-4)
    _assert_close('pred_pose_6d', got['pred_pose_6d'], ref['pred_pose_6d'], atol=1e-4, rtol=1e-4)
    _assert_close('pred_shape', got['pred_shape'], ref['pred_shape'], atol=1e-4, rtol=1e-4)
    _assert_close('pred_cam_t', got['pred_cam_t'], ref['pred_cam_t'], atol=1e-4, rtol=1e-4)
    _assert_close('smpl_joints2d', got['smpl_joints2d'], ref['smpl_joints2d'], atol=0.05, rtol=1e-4)   # pixels


def test_against_committed_golden(models):
    """CUDA fp32 path vs tests/golden/spec_resnet50_b2.npz (oracle-made; see make_golden.py)."""
    import os
    from tests.golden.make_golden import build_models
    g = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'spec_resnet50_b2.npz'))
    cc_ref, hmr_ref = build_models(0)
    cc = sb.CameraRegressorNetwork('resnet50'); cc.load_state_dict(cc_ref.state_dict())
    hmr = sb.HMR('resnet50', use_cam=True, use_cam_feats=True); hmr.load_state_dict(hmr_ref.state_dict())
    got = _run_product(cc, hmr, synthetic_batch(2, 0), 'fp32')
    T = lambda k: torch.from_numpy(g[k])
    _assert_close('golden vfov', got['cam_angles'][:, 0], T('cam_vfov'), atol=1e-5)
    _assert_close('golden pitch', got['cam_angles'][:, 1], T('cam_pitch'), atol=1e-5)
    _assert_close('golden roll', got['cam_angles'][:, 2], T('cam_roll'), atol=1e-5)
    _assert_close('golden pred_cam', got['pred_cam'], T('pred_cam'), atol=1e-5, rtol=1e-5)
    _assert_close('golden verts', got['smpl_vertices'][:, :64], T('smpl_vertices_first64'), atol=1e-3)
    _assert_close('golden vert mean', got['smpl_vertices'].mean(1), T('smpl_vertices_mean'), atol=1e-4)
    _assert_close('golden joints3d', got['smpl_joints3d'], T('smpl_joints3d'), atol=1e-3)
    _assert_close('golden joints2d', got['smpl_joints2d'], T('smpl_joints2d'), atol=0.05, rtol=1e-4)


def test_joint_gather_bit_exact(models):
    """Integer tables are applied exactly: duplicated map entries are bit-identical, vertex-picked joints equal
    the vertices they select, rotations are orthonormal."""
    cc, _, hmr, _ = models
    got = _run_product(cc, hmr, synthetic_batch(3, seed=2), 'fp32')
    j3, v = got['smpl_joints3d'], got['smpl_vertices']
    jm = JOINT_MAP_49
    for a in range(49):
        for c in range(a + 1, 49):
            if jm[a] == jm[c]:
                assert torch.equal(j3[:, a], j3[:, c]), (a, c)
        if 24 <= jm[a] < 45:
            assert torch.equal(j3[:, a], v[:, SMPL_VERTEX_IDS_21[jm[a] - 24]]), a
    R = got['pred_pose'].reshape(-1, 3, 3)
    assert torch.allclose(R.transpose(1, 2) @ R, torch.eye(3, device=R.device).expand_as(R), atol=1e-5)
    assert torch.allclose(torch.linalg.det(R), torch.ones(R.shape[0], device=R.device), atol=1e-5)


def test_smpl_kernels_isolated_from_trunk(models):
    """smpl_prep / smpl_verts / smpl_joints alone: the oracle's SMPL49 (oracle/head.py::lbs, restating smplx.lbs A.4) is fed the
    pose / shape THE PRODUCT predicted, so backbone and head deviations drop out and the fp32 LBS kernels are held to fp32
    round-off (1e-5 absolute; measured error is printed by the assert on failure) instead of the 1e-3 vertex tolerance of the full path.  B = 70 spans two 64-image tiles of the
    vertex kernel, the second one ragged with idle warps."""
    cc, _, hmr, hmr_ref = models
    b = synthetic_batch(70, seed=11)
    got = _run_product(cc, hmr, b, 'bf16')
    verts, j49 = hmr_ref.smpl.smpl(got['pred_pose'].cpu().reshape(-1, 24, 3, 3), got['pred_shape'].cpu())
    _assert_close('verts | product pose', got['smpl_vertices'], verts, atol=1e-5, rtol=1e-5)
    _assert_close('joints3d | product pose', got['smpl_joints3d'], j49, atol=1e-5, rtol=1e-5)


# --------------------------------------------------------------------------------------- 16-bit tensor-core modes
@pytest.mark.parametrize('precision', ['bf16', 'fp16'])
def test_full_forward_lowp_parity(models, precision):
    cc, cc_ref, hmr, hmr_ref = models
    dt = TORCH_DT[precision]
    b = synthetic_batch(4, seed=0)
    lg = lowp.camcalib_lowp(cc_ref, b['images'], dt)
    vfov, pitch, roll = og.convert_preds_to_angles(*lg)
    R, K, _ = og.cam_params_from_angles(vfov, pitch, roll, b['img_h'], b['img_w'])
    ref = lowp.hmr_lowp(hmr_ref, b['images'], R, K, b['bbox_scale'], b['bbox_center'], b['img_w'], b['img_h'], dt)
    got = _run_product(cc, hmr, b, precision)
    # tolerance: the emulation rounds at the same points; what is left is fp32 summation order, which can flip a
    # 16-bit rounding (1 ulp = 2^-8 bf16) on isolated activations -> ~1e-3 relative on pooled features.
    _assert_close('cam angles', got['cam_angles'], torch.stack([vfov, pitch, roll], 1), atol=2e-3)
    _assert_close('pred_cam', got['pred_cam'], ref['pred_cam'], atol=5e-3, rtol=5e-3)
    _assert_close('smpl_vertices', got['smpl_vertices'], ref['smpl_vertices'], atol=1e-2)
    _assert_close('pred_pose', got['pred_pose'], ref['pred_pose'], atol=1e-2)


def test_lowp_vs_fp32_oracle_deviation_is_small(models):
    """Sanity: bf16 stays near the fp32 oracle (reported, loose bound: SURVEY.md 7.2 measured ~3% of feature std)."""
    cc, cc_ref, hmr, hmr_ref = models
    b = synthetic_batch(2, seed=3)
    ref = spec_full_forward(cc_ref, hmr_ref, b['images'], b['bbox_scale'], b['bbox_center'], b['img_w'], b['img_h'])
    got = _run_product(cc, hmr, b, 'bf16')
    err = (got['smpl_vertices'].cpu() - ref['smpl_vertices']).abs().max().item()
    assert err < 0.15, err


# --------------------------------------------------------------------------------------- other backbones
@pytest.mark.parametrize('backbone', ['hrnet_w32-conv', 'hrnet_w32-interp', 'resnet34'])
def test_other_backbones_fp32(backbone):
    # un-normalised random-init HRNet features are large; keep the decoders at their xavier(0.01) scale so the
    # regressed body stays metre-sized and the absolute 1e-3 vertex bound of the north star is meaningful
    hmr, ref = make_pair(backbone, seed=4, amplify=False)
    b = synthetic_batch(2, seed=4)
    vfov, pitch, roll = synthetic_camera(2, seed=4)
    R, K, _ = og.cam_params_from_angles(vfov, pitch, roll, b['img_h'], b['img_w'])
    with torch.no_grad():
        want = ref(b['images'], R, K, b['bbox_scale'], b['bbox_center'], b['img_w'], b['img_h'])
        feat_ref = ref.backbone(b['images'])
    hmr.backbone.set_precision('fp32')
    hmr.to(DEV)
    feat = hmr.backbone(b['images'].to(DEV))
    _assert_close('features', feat, feat_ref, atol=1e-3 * feat_ref.abs().mean().item(), rtol=1e-3)
    got = hmr(b['images'].to(DEV), R.to(DEV), K.to(DEV), b['bbox_scale'].to(DEV), b['bbox_center'].to(DEV),
              b['img_w'].to(DEV), b['img_h'].to(DEV))
    _assert_close('smpl_vertices', got['smpl_vertices'], want['smpl_vertices'], atol=1e-3)
    _assert_close('pred_cam', got['pred_cam'], want['pred_cam'], atol=1e-5, rtol=1e-5)


# fp16 is not run for HRNet: with un-normalised random weights its activations grow past 65504 (features ~3e3 x a 20x stage-4
# dynamic range), so the fp16 emulation AND the kernels overflow to inf -- a property of the synthetic weights, not of the path
@pytest.mark.parametrize('backbone,precision', [('hrnet_w32-conv', 'bf16'), ('hrnet_w32-interp', 'bf16')])
def test_hrnet_lowp_parity(backbone, precision):
    """HRNet tensor-core path against the PRECISION-MATCHED oracle (oracle/lowp.py::hrnet_trunk_lowp rounds to 16 bits after
    every op the CUDA path materialises).  What is left is fp32 summation order flipping isolated 16-bit roundings -- and
    with these un-normalised random weights the network AMPLIFIES such a flip: test_layerwise_lowp_profile (measured on
    B200) shows the CUDA/oracle difference starting at 1e-7..1e-9 mean-relative on the first convs (bit-identical up to
    single-ulp flips), growing smoothly ~3-10x per block with no jump at any kernel, and saturating after ~25 convs at the
    level of two independent 16-bit realisations (6e-3..8e-3 mean-relative, isolated elements up to 0.2 x scale) for ResNet-50
    and HRNet alike.  The end-of-trunk bound therefore is the bf16 noise floor (3e-2 mean, 0.6 x scale max); the tight
    per-kernel statement is test_conv_kernels / test_fused_bottleneck_kernel (identical inputs: mean-relative < 2e-4)."""
    hmr, ref = make_pair(backbone, seed=4, amplify=False)
    dt = TORCH_DT[precision]
    b = synthetic_batch(2, seed=4)
    feat_ref = lowp.hrnet_trunk_lowp(ref.backbone, b['images'], dt)
    hmr.backbone.set_precision(precision)
    feat = hmr.to(DEV).backbone(b['images'].to(DEV)).cpu()
    scale = feat_ref.abs().mean().item()
    ulp = 2.0 ** -8 if precision == 'bf16' else 2.0 ** -11
    rel = ((feat - feat_ref).abs().mean() / scale).item()
    print(f'{backbone} {precision}: mean rel err {rel:.3e}, max err / scale {((feat - feat_ref).abs().max() / scale).item():.3e}')
    assert rel < 3e-2, rel
    _assert_close(f'{backbone} features', feat, feat_ref, atol=0.6 * scale, rtol=0.0)
    # (the head / SMPL tail on HRNet features is checked in fp32 by test_other_backbones_fp32: with un-normalised random weights
    # the features are ~3e3 and the regressed vertices inherit the 16-bit noise floor at a scale where an absolute bound says nothing)


def _layerwise_profile(prod_trunk, ref_trunk, images, dt, emulate):
    """(conv name, mean rel err, max err / scale) of every conv op of the compiled program whose destination is a plain
    activation buffer, CUDA path vs the traced precision-matched oracle."""
    lowp.TRACE = {}
    try:
        emulate(ref_trunk, images, dt)
        trace = dict(lowp.TRACE)
    finally:
        lowp.TRACE = None
    mods = dict(ref_trunk.named_modules())
    rows = []
    P = prod_trunk._program
    for i, o in enumerate(P.ops):
        if o['type'] != 1 or o['dst_coff'] != 0 or P.buf_ch[o['dst']] != o['cout']:
            continue
        name = P.convs[o['wslot']][0]
        want = trace.get(mods[name])
        if want is None:
            continue
        got = prod_trunk.activation_after(images.to(DEV), i).cpu()
        assert got.shape == want.shape, (name, got.shape, want.shape)
        want = lowp._rnd(want, dt)          # (a fused block's downsample branch is fp32 in the trace; its un-fused debug read-out is 16 bit)
        scale = want.abs().mean().item() + 1e-30
        rows.append((name, ((got - want).abs().mean() / scale).item(), ((got - want).abs().max() / scale).item()))
    return rows


@pytest.mark.parametrize('backbone', ['resnet50', 'hrnet_w32-conv'])
def test_layerwise_lowp_profile(backbone):
    """EVERY intermediate conv output of the bf16 tensor-core path against the precision-matched oracle, layer by layer
    (specb200_trunk_forward_until reads the activation buffers).  A kernel that rounds at a different point, drops a
    bias or mis-handles a border shows up as a jump at ITS layer; what accumulates smoothly is rounding-boundary flips."""
    hmr, ref = make_pair(backbone, seed=4, amplify=False)
    x = synthetic_batch(2, seed=4)['images']
    hmr.backbone.set_precision('bf16')
    hmr.to(DEV)
    rows = _layerwise_profile(hmr.backbone, ref.backbone, x, torch.bfloat16, lowp.trunk_lowp)
    assert len(rows) > 40
    runmax = 0.0
    for i, (name, mean_rel, max_rel) in enumerate(rows):
        print(f'{name:40s} mean rel {mean_rel:.3e}  max/scale {max_rel:.3e}')
        # (a) the first convs agree up to single-ulp flips of isolated elements
        if i < 4:
            assert mean_rel < 2e-5 and max_rel < 0.1, (name, mean_rel, max_rel)
        # (b) no kernel introduces an error of its own: the difference grows smoothly (flips being amplified by the random
        #     network, measured <= 14x from one conv to the next) up to the 16-bit noise floor; a kernel that mis-rounds, drops a
        #     bias or mangles a border would jump to >= 1e-1 at ITS layer
        assert mean_rel <= max(30 * runmax, 1e-5), (name, mean_rel, runmax)
        assert mean_rel < 3e-2 and max_rel < 0.6, (name, mean_rel, max_rel)          # 16-bit noise floor (measured <= 2.1e-2 / 0.19)
        runmax = max(runmax, mean_rel)


def test_hrnet_w48_runs_on_gpu():
    """The W48 program (f4 ctor variant) on the device: fp32 parity of the trunk features, finite bf16 features of the same
    shape within the lowp bound."""
    hmr, ref = make_pair('hrnet_w48-conv', seed=8, amplify=False)
    x = synthetic_batch(1, seed=8)['images']
    with torch.no_grad():
        feat_ref = ref.backbone(x)
    hmr.backbone.set_precision('fp32')
    feat = hmr.to(DEV).backbone(x.to(DEV))
    assert feat.shape == (1, 720, 7, 7)
    _assert_close('w48 features fp32', feat, feat_ref, atol=1e-3 * feat_ref.abs().mean().item(), rtol=1e-3)
    hmr.backbone.set_precision('bf16')
    f16 = hmr.backbone(x.to(DEV)).cpu()
    want = lowp.hrnet_trunk_lowp(ref.backbone, x, torch.bfloat16)
    s = want.abs().mean().item()
    assert ((f16 - want).abs().mean() / s).item() < 3e-2                         # bf16 noise floor, see test_hrnet_lowp_parity
    _assert_close('w48 features bf16', f16, want, atol=0.6 * s, rtol=0.0)


def test_camcalib_module_forward_and_variable_size():
    """CameraRegressorNetwork.forward returns three (B,256) logit tensors; non-224 inputs work (the demo feeds
    min-side-600 images, camcalib_demo.py:95-102)."""
    cc, ref = make_camcalib_pair('resnet50', seed=1)
    cc.backbone.set_precision('fp32')
    cc.to(DEV)
    x = torch.randn(1, 3, 192, 256)
    with torch.no_grad():
        want = ref(x)
    got = cc(x.to(DEV))
    assert isinstance(got, list) and len(got) == 3 and all(g.shape == (1, 256) for g in got)
    for g, w in zip(got, want):
        _assert_close('logits', g, w, atol=2e-5, rtol=1e-4)
    a = sb.convert_preds_to_angles(*got, loss_type='softargmax_l2')
    wa = og.convert_preds_to_angles(*want)
    for g, w in zip(a, wa):
        _assert_close('angles', g, w, atol=1e-5)
    # multi-layer FC variant (model.py:54-70)
    cc3, ref3 = make_camcalib_pair('resnet34', seed=2, num_fc_layers=3)
    cc3.backbone.set_precision('fp32')
    x = torch.randn(2, 3, 224, 224)
    with torch.no_grad():
        want = ref3(x)
    got = cc3.to(DEV)(x.to(DEV))
    for g, w in zip(got, want):
        _assert_close('logits3', g, w, atol=1e-4, rtol=1e-3)


# --------------------------------------------------------------------------------------- consumer contract / properties
def test_consumer_shim_contract(models):
    """Replays what spec/tester.py:143-167 and spec/trainer.py:235-254,348-353 do with the outputs."""
    _, _, hmr, _ = models
    hmr.backbone.set_precision('bf16')
    hmr.to(DEV)
    b = synthetic_batch(3, seed=5, device=DEV)
    vfov, pitch, roll = synthetic_camera(3, seed=5)
    R, K, _ = og.cam_params_from_angles(vfov, pitch, roll, b['img_h'].cpu(), b['img_w'].cpu())
    img_h_int = b['img_h'].long()                       # trainer.py:239-240 passes integer tensors
    img_w_int = b['img_w'].long()
    out = hmr(b['images'], R.to(DEV), K.to(DEV), b['bbox_scale'], b['bbox_center'], img_w_int, img_h_int)   # positional
    assert list(out.keys()) == ['smpl_vertices', 'smpl_joints3d', 'smpl_joints2d', 'pred_cam_t', 'pred_pose',
                                'pred_cam', 'pred_shape', 'pred_pose_6d']
    shapes = {'smpl_vertices': (3, 6890, 3), 'smpl_joints3d': (3, 49, 3), 'smpl_joints2d': (3, 49, 2), 'pred_cam_t': (3, 3),
              'pred_pose': (3, 24, 3, 3), 'pred_cam': (3, 3), 'pred_shape': (3, 10), 'pred_pose_6d': (3, 144)}
    for k, v in out.items():
        assert isinstance(v, torch.Tensor) and v.dtype == torch.float32 and v.device.type == 'cuda'
        assert tuple(v.shape) == shapes[k]
        assert np.isfinite(v.cpu().numpy()).all()                       # tester.py:153-154
    out['smpl_joints2d'][:, :, 0] /= 224.                               # losses.py:191 in-place write
    _ = out['pred_pose'][:, 1:].contiguous(), out['pred_pose'][:, 0].unsqueeze(1).contiguous()   # trainer.py:251-252
    _ = out['smpl_joints3d'][:, 25:]                                    # losses.py:335


def test_graph_equals_eager_and_is_deterministic(models):
    cc, _, hmr, _ = models
    b = synthetic_batch(8, seed=6)
    e = _run_product(cc, hmr, b, 'bf16', graph=False)
    g1 = _run_product(cc, hmr, b, 'bf16', graph=True)
    g2 = _run_product(cc, hmr, b, 'bf16', graph=True)
    for k in e:
        assert torch.equal(e[k], g1[k]), k
        assert torch.equal(g1[k], g2[k]), k


def test_batch_composition_invariance_at_full_size(models):
    """Size-independent property at BASELINE's B=256: an image's result does not depend on its position in the
    batch or on the batch size (every image is independent through the whole path, SURVEY.md 8e)."""
    cc, _, hmr, _ = models
    big = synthetic_batch(256, seed=7)
    out_big = _run_product(cc, hmr, big, 'bf16')
    idx = [0, 127, 128, 255]
    small = {k: v[idx] for k, v in big.items()}
    out_small = _run_product(cc, hmr, small, 'bf16')
    for k in out_big:
        assert torch.equal(out_big[k][idx], out_small[k]), k
    R = out_big['pred_pose'].reshape(-1, 3, 3)
    assert torch.allclose(R.transpose(1, 2) @ R, torch.eye(3, device=R.device).expand_as(R), atol=1e-5)
    assert torch.isfinite(out_big['smpl_vertices']).all()


def _lowp_reference(cc_ref, hmr_ref, b, idx, dt):
    """Precision-matched oracle of the full SPEC step for the images ``idx`` of batch ``b``."""
    sub = {k: v[idx] for k, v in b.items()}
    lg = lowp.camcalib_lowp(cc_ref, sub['images'], dt)
    vfov, pitch, roll = og.convert_preds_to_angles(*lg)
    R, K, _ = og.cam_params_from_angles(vfov, pitch, roll, sub['img_h'], sub['img_w'])
    ref = lowp.hmr_lowp(hmr_ref, sub['images'], R, K, sub['bbox_scale'], sub['bbox_center'], sub['img_w'], sub['img_h'], dt)
    ref['cam_angles'] = torch.stack([vfov, pitch, roll], 1)
    return ref


@pytest.mark.parametrize('precision,B,n_oracle', [('bf16', 256, 32), ('fp16', 64, 16)], ids=['C3-bf16-b256', 'C2-fp16-b64'])
def test_bench_config_under_oracle(models, precision, B, n_oracle):
    """The BENCHMARKED configurations (BASELINE.json configs[2] = bf16 batch 256, configs[1] = fp16 batch 64), run exactly as
    bench.py runs them (SPECPipeline CUDA-graph replay), with EVERY image checked: (a) image by image bit-equal to B=4
    eager runs of the same images (B/4 runs) -- at B=256 the persistent / CTA-pair kernels loop over several tiles per
    CTA (TMEM double-buffer phase flips, remote tempty arrives), at B=4 they do not; (b) ``n_oracle`` images spread over the
    batch against the precision-matched CPU oracle (oracle/lowp.py), same tolerances as test_full_forward_lowp_parity."""
    cc, cc_ref, hmr, hmr_ref = models
    dt = TORCH_DT[precision]
    b = synthetic_batch(B, seed=31)
    big = _run_product(cc, hmr, b, precision, graph=True)
    big2 = _run_product(cc, hmr, b, precision, graph=True)
    for k in big:
        assert torch.isfinite(big[k]).all(), k
        assert torch.equal(big[k], big2[k]), k                           # replay is deterministic
    for i0 in range(0, B, 4):
        small = _run_product(cc, hmr, {k: v[i0:i0 + 4] for k, v in b.items()}, precision, graph=False)
        for k in big:
            assert torch.equal(big[k][i0:i0 + 4], small[k]), (k, i0)
    idx = list(range(0, B, B // n_oracle))
    ref = _lowp_reference(cc_ref, hmr_ref, b, idx, dt)
    _assert_close('cam angles', big['cam_angles'][idx], ref['cam_angles'], atol=2e-3)
    _assert_close('pred_cam', big['pred_cam'][idx], ref['pred_cam'], atol=5e-3, rtol=5e-3)
    _assert_close('smpl_vertices', big['smpl_vertices'][idx], ref['smpl_vertices'], atol=1e-2)
    _assert_close('smpl_joints3d', big['smpl_joints3d'][idx], ref['smpl_joints3d'], atol=1e-2)
    _assert_close('pred_pose', big['pred_pose'][idx], ref['pred_pose'], atol=1e-2)
    _assert_close('pred_shape', big['pred_shape'][idx], ref['pred_shape'], atol=5e-3, rtol=5e-3)


def test_c4_eval_loop_batch_under_oracle(models):
    """BASELINE.json configs[3] (SPEC-SYN-shaped eval loop; /root/reference/spec/trainer.py:235-245): CamCalib is bypassed --
    the dataset supplies pre-computed cam_rotmat / cam_int -- and ``img_h`` / ``img_w`` are the int64 columns of
    ``batch['orig_shape']``; batch 128 per GPU, bf16.  Checked like the bench config: bit-equal to B=4 runs, 16 images
    against the precision-matched oracle."""
    _, _, hmr, hmr_ref = models
    B = 128
    b = synthetic_batch(B, seed=41)
    vfov, pitch, roll = synthetic_camera(B, seed=41)
    R, K, _ = og.cam_params_from_angles(vfov, pitch, roll, b['img_h'], b['img_w'])
    orig_shape = torch.stack([b['img_h'], b['img_w']], 1).long()          # cam_dataset.py:350,486
    hmr.backbone.set_precision('bf16')
    hmr.to(DEV)
    def run(sl):
        o = hmr(b['images'][sl].to(DEV), R[sl].to(DEV), K[sl].to(DEV), b['bbox_scale'][sl].to(DEV), b['bbox_center'][sl].to(DEV),
                orig_shape[sl, 1].to(DEV), orig_shape[sl, 0].to(DEV))
        torch.cuda.synchronize()
        return o
    big = run(slice(0, B))
    for i0 in range(0, B, 4):
        small = run(slice(i0, i0 + 4))
        for k in big:
            assert torch.equal(big[k][i0:i0 + 4], small[k]), (k, i0)
    idx = list(range(0, B, 8))
    ref = lowp.hmr_lowp(hmr_ref, b['images'][idx], R[idx], K[idx], b['bbox_scale'][idx], b['bbox_center'][idx],
                        orig_shape[idx, 1], orig_shape[idx, 0], torch.bfloat16)
    _assert_close('pred_cam', big['pred_cam'][idx], ref['pred_cam'], atol=5e-3, rtol=5e-3)
    _assert_close('smpl_vertices', big['smpl_vertices'][idx], ref['smpl_vertices'], atol=1e-2)
    _assert_close('pred_pose', big['pred_pose'][idx], ref['pred_pose'], atol=1e-2)
    _assert_close('pred_cam_t', big['pred_cam_t'][idx], ref['pred_cam_t'], atol=2e-2, rtol=1e-2)


@pytest.mark.parametrize('case', ['spec_resnet50', 'spec_hrnet_w32_conv', 'hmr_resnet34_nocam'])
def test_against_reference_wrapper_fixture(case):
    """CUDA fp32 path vs tests/golden/reference_wrappers.npz -- outputs of the reference's OWN wrapper code
    (camcalib/model.py, spec/models/hmr.py, cam_utils.py, cam_params.py executed unmodified, pare stubbed;
    tests/golden/reference_wrappers.py).  North-star tolerances: vertices 1e-3, camera parameters 1e-5."""
    from tests.golden import reference_wrappers as rw
    fx = np.load(rw.FIXTURE)
    T = lambda k: torch.from_numpy(fx[f'{case}/{k}'])
    cfg = rw.CASES[case]
    seed = 40 + list(rw.CASES).index(case)
    cc_o, hmr_o = rw.oracle_models(cfg, seed)
    b = rw.case_inputs(cfg, seed)
    hmr = sb.HMR(cfg['hmr'], use_cam=cfg['use_cam'], use_cam_feats=cfg['use_cam_feats'])
    hmr.load_state_dict(hmr_o.state_dict(), strict=True)
    hmr.backbone.set_precision('fp32')
    hmr.to(DEV)
    if cfg['camcalib']:
        cc = sb.CameraRegressorNetwork(cfg['camcalib'], num_fc_layers=cfg['fc_layers'])
        cc.load_state_dict(cc_o.state_dict(), strict=True)
        cc.backbone.set_precision('fp32')
        cc.to(DEV)
        logits = cc(b['images'].to(DEV))
        for n, l in zip(('vfov', 'pitch', 'roll'), logits):       # fp32 GEMM chains (3 layers deep in one case): 1e-5 of the logit scale
            _assert_close('logits ' + n, l, T('logits_' + n), atol=1e-5 * T('logits_' + n).abs().mean().item() + 5e-5, rtol=1e-4)
        ang, R, K, _ = cc.predict_camera(b['images'].to(DEV), b['img_h'].to(DEV), b['img_w'].to(DEV))
        _assert_close('angles', ang, torch.stack([T('cam_vfov'), T('cam_pitch'), T('cam_roll')], 1), atol=1e-5)
        _assert_close('R', R, T('cam_rotmat'), atol=1e-5)
        _assert_close('K', K, T('cam_intrinsics'), atol=1e-2, rtol=1e-5)
        assert (K[:, 2, 2] == 0).all()
        got = hmr(b['images'].to(DEV), R, K, b['bbox_scale'].to(DEV), b['bbox_center'].to(DEV), b['img_w'].to(DEV), b['img_h'].to(DEV))
    else:
        got = hmr(b['images'].to(DEV))
    assert list(got.keys()) == list(fx[f'{case}/keys'])
    _assert_close('smpl_vertices', got['smpl_vertices'], T('hmr_smpl_vertices'), atol=1e-3)
    _assert_close('smpl_joints3d', got['smpl_joints3d'], T('hmr_smpl_joints3d'), atol=1e-3)
    _assert_close('pred_cam', got['pred_cam'], T('hmr_pred_cam'), atol=1e-5, rtol=1e-5)
    _assert_close('pred_shape', got['pred_shape'], T('hmr_pred_shape'), atol=1e-4, rtol=1e-4)
    _assert_close('pred_pose', got['pred_pose'], T('hmr_pred_pose'), atol=1e-4)
    _assert_close('pred_cam_t', got['pred_cam_t'], T('hmr_pred_cam_t'), atol=1e-3, rtol=1e-4)
    _assert_close('smpl_joints2d', got['smpl_joints2d'], T('hmr_smpl_joints2d'), atol=0.05, rtol=1e-3)


# --------------------------------------------------------------------------------------- edge cases
@pytest.mark.parametrize('batch', [1, 33, 257])
def test_ragged_batches_bf16(models, batch):
    """Batch sizes that are not multiples of any tile (128-row GEMM tiles, 32-image SMPL tiles): image i of a ragged
    batch equals image i of a padded batch bit for bit, and everything is finite."""
    cc, _, hmr, _ = models
    b = synthetic_batch(batch, seed=11)
    got = _run_product(cc, hmr, b, 'bf16')
    pad = 4 - batch % 4 if batch % 4 else 4
    bp = {k: torch.cat([v, v[:pad]], 0) for k, v in b.items()}
    ref = _run_product(cc, hmr, bp, 'bf16')
    for k in got:
        assert torch.isfinite(got[k]).all(), k
        assert torch.equal(got[k], ref[k][:batch]), k


def test_empty_batch_and_bad_inputs(models):
    _, _, hmr, _ = models
    hmr.to(DEV)
    z = torch.zeros(0, 3, 224, 224, device=DEV)
    with pytest.raises(ValueError):
        hmr(z, torch.zeros(0, 3, 3, device=DEV), torch.zeros(0, 3, 3, device=DEV), torch.zeros(0, device=DEV),
            torch.zeros(0, 2, device=DEV), torch.zeros(0, device=DEV), torch.zeros(0, device=DEV))
    x = torch.randn(2, 3, 224, 224, device=DEV)
    with pytest.raises(ValueError):
        hmr(x)                                              # camera inputs are required with use_cam / use_cam_feats
    with pytest.raises(ValueError):
        hmr.backbone(torch.randn(2, 4, 224, 224, device=DEV))
    with pytest.raises(RuntimeError, match='no CPU path'):
        hmr.backbone(torch.randn(1, 3, 224, 224))


def test_input_dtype_and_layout_are_normalised(models):
    """fp16 / non-contiguous images are accepted like any nn.Module input and give the same result as fp32 contiguous."""
    _, _, hmr, _ = models
    hmr.backbone.set_precision('bf16')
    hmr.to(DEV)
    x = torch.randn(2, 224, 224, 3, device=DEV).half().float()      # values exactly representable in fp16
    a = hmr.backbone.pooled_features(x.permute(0, 3, 1, 2).contiguous())
    b = hmr.backbone.pooled_features(x.permute(0, 3, 1, 2))            # non-contiguous view
    c = hmr.backbone.pooled_features(x.permute(0, 3, 1, 2).half())      # fp16 input
    assert torch.equal(a, b) and torch.equal(a, c)


def test_camcalib_full_resolution_fp32():
    """The demo feeds CamCalib whole images at min-side 600 (camcalib_demo.py:95-102, pano_dataset.py:156-162)."""
    cc, ref = make_camcalib_pair('resnet50', seed=1)
    x = torch.randn(1, 3, 600, 800)
    with torch.no_grad():
        want = ref(x)
    cc.backbone.set_precision('fp32')
    got = cc.to(DEV)(x.to(DEV))
    for g, w in zip(got, want):
        _assert_close('logits 600x800', g, w, atol=5e-5, rtol=1e-4)
    ang, R, K, f = cc.predict_camera(x.to(DEV), 600, 800)
    wa = og.convert_preds_to_angles(*want)
    _assert_close('angles', ang, torch.stack(wa, 1), atol=1e-5)
    Rw, Kw, fw = og.cam_params_from_angles(*wa, 600, 800)
    _assert_close('R', R, Rw, atol=1e-5)
    _assert_close('K', K, Kw, atol=1e-2, rtol=1e-5)
    assert float(K[0, 2, 2]) == 0.0                                      # cam_params.py:39-46 leaves K[2,2] = 0
    cc.backbone.set_precision('bf16')
    got16 = cc(x.to(DEV))
    assert all(torch.isfinite(g).all() for g in got16)


def test_use_cam_false_branch_fp32():
    """HMR(use_cam=False): SMPLHead with fixed focal length and crop-normalised joints2d (hmr.py:70-74,114-121)."""
    hmr, ref = make_pair('resnet34', seed=6, use_cam=False, use_cam_feats=False)
    x = synthetic_batch(3, seed=6)['images']
    with torch.no_grad():
        want = ref(x)
    hmr.backbone.set_precision('fp32')
    got = hmr.to(DEV)(x.to(DEV))
    assert list(got.keys()) == list(want.keys())
    _assert_close('verts', got['smpl_vertices'], want['smpl_vertices'], atol=1e-3, rtol=1e-4)
    _assert_close('pred_cam', got['pred_cam'], want['pred_cam'], atol=1e-5, rtol=1e-5)
    _assert_close('cam_t', got['pred_cam_t'], want['pred_cam_t'], atol=1e-3, rtol=1e-4)
    _assert_close('joints2d', got['smpl_joints2d'], want['smpl_joints2d'], atol=1e-3, rtol=1e-3)


def test_reload_state_dict_repacks(models):
    """load_state_dict after a forward marks the handles dirty: the next forward uses the new weights."""
    cc, cc_ref, _, _ = models
    cc.backbone.set_precision('fp32')
    cc.to(DEV)
    x = torch.randn(2, 3, 224, 224)
    a = torch.cat(cc(x.to(DEV)), 1).clone()
    sd = {k: v.clone() for k, v in cc.state_dict().items()}
    sd2 = dict(sd)
    sd2['fc_vfov.weight'] = sd['fc_vfov.weight'] * 0.5
    sd2['backbone.layer4.2.bn3.weight'] = sd['backbone.layer4.2.bn3.weight'] * 1.5
    cc.load_state_dict(sd2)
    bnew = torch.cat(cc(x.to(DEV)), 1).clone()
    assert not torch.allclose(a, bnew)
    cc.load_state_dict(sd)
    c = torch.cat(cc(x.to(DEV)), 1)
    assert torch.equal(a, c)


# --------------------------------------------------------------------------------------- eval metrics (SURVEY 8f-1)
def test_eval_metrics_match_oracle():
    from oracle import eval_metrics as oe
    from spec_b200.metrics import EvalMetrics
    rng = np.random.RandomState(3)
    J = rng.rand(17, 6890).astype(np.float64) ** 8
    J = (J / J.sum(1, keepdims=True)).astype(np.float32)
    Jt = torch.from_numpy(J)
    B = 37
    gt_v = torch.from_numpy((rng.randn(B, 6890, 3) * 0.3).astype(np.float32))
    # prediction = rotated / scaled / shifted / noisy ground truth, so Procrustes has real work to do
    ang = 0.4
    Rz = torch.tensor([[np.cos(ang), -np.sin(ang), 0], [np.sin(ang), np.cos(ang), 0], [0, 0, 1]], dtype=torch.float32)
    pred_v = (1.1 * gt_v @ Rz.T + torch.tensor([0.05, -0.02, 0.1]) + 0.01 * torch.randn(B, 6890, 3, generator=torch.Generator().manual_seed(0)))
    gt_kp = (torch.matmul(Jt[None].expand(B, -1, -1), gt_v))
    gt_kp = gt_kp[:, oe.H36M_TO_J14] - gt_kp[:, [0]]
    m = EvalMetrics(J).to(DEV)
    # trainer style: gt keypoints given, raw v2v
    got = m(pred_v.to(DEV), gt_keypoints_3d=gt_kp.to(DEV), gt_vertices=gt_v.to(DEV))
    mp, pa, v2v, pk = oe.trainer_metrics(pred_v, gt_kp, Jt, gt_v)
    _assert_close('mpjpe', got['mpjpe'], torch.from_numpy(mp), atol=1e-5, rtol=1e-4)
    _assert_close('pa_mpjpe', got['pa_mpjpe'], torch.from_numpy(pa), atol=2e-5, rtol=1e-3)
    _assert_close('v2v', got['v2v'], torch.from_numpy(v2v), atol=1e-5, rtol=1e-4)
    _assert_close('pred_kp', got['pred_keypoints_3d'], pk, atol=1e-5)
    # compute_error.py style: joints regressed from both meshes, centred v2v
    got = m(pred_v.to(DEV), gt_vertices=gt_v.to(DEV), center_v2v=True)
    mp, pa, v2v = oe.eval_single(pred_v, gt_v, Jt)
    _assert_close('mpjpe2', got['mpjpe'], torch.from_numpy(mp), atol=1e-5, rtol=1e-4)
    _assert_close('pa_mpjpe2', got['pa_mpjpe'], torch.from_numpy(pa), atol=2e-5, rtol=1e-3)
    _assert_close('v2v2', got['v2v'], torch.from_numpy(v2v), atol=1e-5, rtol=1e-4)
    # a reflected prediction exercises the det(U V^T) < 0 branch
    refl = pred_v * torch.tensor([-1.0, 1.0, 1.0])
    got = m(refl.to(DEV), gt_keypoints_3d=gt_kp.to(DEV))
    _, pa, _, _ = oe.trainer_metrics(refl, gt_kp, Jt)
    _assert_close('pa_mpjpe reflected', got['pa_mpjpe'], torch.from_numpy(pa), atol=5e-5, rtol=2e-3)
    # works straight on the strided vertices view of a packed record buffer
    rec = torch.zeros(B, sb.pipeline.RECORD_FLOATS, device=DEV)
    sb.unpack_record(rec)['smpl_vertices'].copy_(pred_v.to(DEV))
    got2 = m(sb.unpack_record(rec)['smpl_vertices'], gt_keypoints_3d=gt_kp.to(DEV))
    assert torch.equal(got2['mpjpe'], m(pred_v.to(DEV), gt_keypoints_3d=gt_kp.to(DEV))['mpjpe'])


def test_module_graph_cache_survives_shape_changes(models):
    """HMR.forward replays a cached CUDA graph for small batches; interleaving other shapes (which re-allocates the
    eager workspaces) and re-loading weights must not corrupt or stale the cached graphs."""
    _, _, hmr, hmr_ref = models
    hmr.backbone.set_precision('bf16')
    hmr.to(DEV)
    def run(B, seed):
        b = synthetic_batch(B, seed=seed, device=DEV)
        vfov, pitch, roll = synthetic_camera(B, seed=seed)
        R, K, _ = og.cam_params_from_angles(vfov, pitch, roll, b['img_h'].cpu(), b['img_w'].cpu())
        return hmr(b['images'], R.to(DEV), K.to(DEV), b['bbox_scale'], b['bbox_center'], b['img_w'], b['img_h'])
    a1 = run(2, 21)
    _ = run(5, 22)                      # another cached shape
    _ = run(40, 23)                     # eager path (B > graph_max_batch) re-allocates the workspaces
    a2 = run(2, 21)
    for k in a1:
        assert torch.equal(a1[k], a2[k]), k
        assert a1[k].data_ptr() != a2[k].data_ptr()                    # fresh tensors per call
    import os
    os.environ['SPECB200_MODULE_GRAPH'] = '0'
    try:
        hmr._module_graph = False
        e = run(2, 21)
    finally:
        hmr._module_graph = True
        os.environ.pop('SPECB200_MODULE_GRAPH', None)
    for k in a1:
        assert torch.equal(a1[k], e[k]), k                             # graph replay == eager launches, bit for bit
    sd = {k: v.clone() for k, v in hmr.state_dict().items()}
    sd2 = dict(sd); sd2['head.decshape.bias'] = sd['head.decshape.bias'] + 0.5
    hmr.load_state_dict(sd2)
    c = run(2, 21)
    assert not torch.equal(c['pred_shape'], a1['pred_shape'])           # stale graphs were dropped
    hmr.load_state_dict(sd)
    d = run(2, 21)
    assert torch.equal(d['pred_shape'], a1['pred_shape'])
