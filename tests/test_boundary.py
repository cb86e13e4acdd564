"""CPU tests of the drop-in boundary: constructor / forward signatures and state_dict names equal the
reference's (model.py:25-31,72; hmr.py:29-41,82-91), the C-ABI library loads and exports every symbol
include/specb200.h declares, and the product refuses to compute without a GPU (no CPU fallback)."""
import inspect
import os
import re

import numpy as np
import pytest
import torch

import spec_b200 as sb
from spec_b200 import _lib
from tests.conftest import make_pair, make_camcalib_pair, ROOT


def test_library_loads_and_exports_header_symbols():
    hdr = open(os.path.join(ROOT, 'include', 'specb200.h')).read()
    declared = set(re.findall(r'\b(specb200_[a-z0-9_]+)\s*\(', hdr))
    assert len(declared) >= 20
    import ctypes
    l = ctypes.CDLL(_lib.LIB_PATH) if os.path.exists(_lib.LIB_PATH) else _lib.lib()
    for name in sorted(declared):
        assert hasattr(l, name), f'{name} declared in specb200.h but not exported'
    assert declared == set(_lib.EXPORTED_SYMBOLS), declared ^ set(_lib.EXPORTED_SYMBOLS)
    assert _lib.lib().specb200_abi_version() == 1


def test_struct_layouts_match_header():
    import ctypes
    assert ctypes.sizeof(_lib.Op) == 15 * 4
    assert ctypes.sizeof(_lib.HmrOutputs) == 8 * 16
    assert ctypes.sizeof(_lib.HmrParams) == 24 + 22 * 8


def test_signatures_match_reference():
    sig = inspect.signature(sb.CameraRegressorNetwork.__init__)
    assert list(sig.parameters)[1:] == ['backbone', 'num_fc_layers', 'num_fc_channels', 'num_out_channels']
    assert [p.default for p in list(sig.parameters.values())[1:]] == ['resnet50', 1, 1024, 256]
    sig = inspect.signature(sb.HMR.__init__)
    names = list(sig.parameters)[1:11]
    assert names == ['backbone', 'focal_length', 'img_res', 'pretrained', 'use_cam', 'p', 'estimate_var',
                     'use_separate_var_branch', 'uncertainty_activation', 'use_cam_feats']
    fsig = inspect.signature(sb.HMR.forward)
    assert list(fsig.parameters)[1:8] == ['images', 'cam_rotmat', 'cam_intrinsics', 'bbox_scale', 'bbox_center',
                                          'img_w', 'img_h']        # positional order used at trainer.py:139
    assert list(inspect.signature(sb.CameraRegressorNetwork.forward).parameters)[1:] == ['images']


def test_reference_signatures_if_mounted():
    """Argument lists of the reference's drop-in classes, parsed from its sources into tests/golden/reference_tables.json
    (tests/golden/reference_wrappers.py), equal the product's literally."""
    import json
    with open(os.path.join(ROOT, 'tests', 'golden', 'reference_tables.json')) as fh:
        ref = json.load(fh)['signatures']
    assert ref['HMR.forward'] == list(inspect.signature(sb.HMR.forward).parameters)[1:8]
    assert ref['HMR.__init__'] == list(inspect.signature(sb.HMR.__init__).parameters)[1:11]
    assert ref['CameraRegressorNetwork.__init__'] == list(inspect.signature(sb.CameraRegressorNetwork.__init__).parameters)[1:]
    assert ref['CameraRegressorNetwork.forward'] == list(inspect.signature(sb.CameraRegressorNetwork.forward).parameters)[1:]


@pytest.mark.parametrize('backbone', ['resnet50', 'resnet34', 'hrnet_w32-conv', 'hrnet_w32-interp'])
def test_state_dict_roundtrip_with_oracle(backbone):
    prod, ref = make_pair(backbone)              # strict load inside
    a, b = prod.state_dict(), ref.state_dict()
    assert list(a.keys()) == list(b.keys()) or set(a) == set(b)
    for k in ('head.init_pose', 'head.fc1.weight', 'backbone.conv1.weight', 'smpl.smpl.posedirs'):
        assert k in a and a[k].shape == b[k].shape
    exp_c = {'resnet50': 2048, 'resnet34': 512, 'hrnet_w32-conv': 480, 'hrnet_w32-interp': 480}[backbone]
    assert a['head.fc1.weight'].shape == (1024, exp_c + 164)
    if backbone == 'resnet50':
        import torchvision
        tv = set(k for k in torchvision.models.resnet50(weights=None).state_dict() if not k.startswith('fc.'))
        assert tv == set(k[len('backbone.'):] for k in a if k.startswith('backbone.'))


def test_camcalib_state_dict_and_multilayer():
    prod, ref = make_camcalib_pair('resnet50')
    assert set(prod.state_dict()) == set(ref.state_dict())
    prod3, ref3 = make_camcalib_pair('resnet34', num_fc_layers=3)
    assert set(prod3.state_dict()) == set(ref3.state_dict())
    assert 'fc_vfov.2.weight' in prod3.state_dict()


def test_flop_counts():
    assert sb.resnet50().conv_flops_per_image() == 2 * 4087136256          # SURVEY.md B.1
    assert sb.hrnet_w32().conv_flops_per_image() == 2 * 7917220864         # SURVEY.md B.3


@pytest.mark.skipif(torch.cuda.is_available(), reason='CPU-only check')
def test_no_cpu_fallback():
    prod, _ = make_camcalib_pair('resnet34')
    with pytest.raises(RuntimeError, match='no CPU path'):
        prod(torch.randn(1, 3, 64, 64))
    h = sb.HMR('resnet34', use_cam=True, use_cam_feats=True)
    with pytest.raises(RuntimeError, match='no CPU path'):
        h(torch.randn(1, 3, 224, 224), torch.eye(3)[None], torch.eye(3)[None], torch.ones(1), torch.zeros(1, 2),
          torch.ones(1), torch.ones(1))
    with pytest.raises(RuntimeError, match='no CPU path'):
        sb.decode_logits(torch.zeros(1, 768))


def test_product_does_not_import_oracle():
    """The product package must never route through the oracle (test infrastructure)."""
    pkg = os.path.join(ROOT, 'spec_b200')
    for fn in os.listdir(pkg):
        if fn.endswith('.py'):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r'^\s*(from|import)\s+oracle\b', src, re.M), fn
            assert 'from oracle' not in src and 'import oracle' not in src, fn


def test_record_layout_views():
    rec = torch.arange(3 * sb.pipeline.RECORD_FLOATS, dtype=torch.float32).view(3, -1)
    d = sb.unpack_record(rec)
    assert d['smpl_vertices'].shape == (3, 6890, 3) and d['pred_pose'].shape == (3, 24, 3, 3)
    assert d['smpl_vertices'].data_ptr() == rec.data_ptr()              # views, not copies
    assert float(d['smpl_joints3d'][1, 0, 0]) == float(rec[1, 20670])
    assert sum(v[0].numel() for v in d.values()) == sb.pipeline.RECORD_FLOATS
    d['smpl_joints2d'][0, 0, 0] = -1.0                                  # writable (losses.py:191 mutates in place)
    assert float(rec[0, 20670 + 147]) == -1.0


# --------------------------------------------------------------------------------------- op-program compiler (host logic)
@pytest.mark.parametrize('arch,kw', [('resnet50', {}), ('resnet34', {}), ('hrnet_w32', {'use_conv': True}),
                                     ('hrnet_w32', {'use_conv': False}), ('hrnet_w48', {'use_conv': True})])
def test_program_buffer_liveness(arch, kw):
    """The compiled op program reuses activation buffers; replay it symbolically and check that no op reads a buffer
    whose value has been overwritten since the reader's producer wrote it, that residual/src never alias dst for convs,
    and that channel widths line up."""
    from spec_b200.backbone import Trunk
    from spec_b200._lib import OP_CONV, OP_MAXPOOL, OP_UPADD, OP_BILINEAR, OP_COPY
    t = Trunk(arch, **kw)
    P = t._program
    version = {0: 0}                       # buffer -> version counter
    expect = {}                            # buffer -> version its consumers were promised
    ch = list(P.buf_ch)
    ch[0] = 4
    for i, o in enumerate(P.ops):
        srcs = [o['src']] + ([o['src2']] if o['src2'] >= 0 else [])
        for b in srcs:
            assert b in version, f'op {i} reads undefined buffer {b}'
        if o['type'] == OP_CONV:
            assert o['dst'] not in srcs, f'op {i}: conv writes a buffer it reads'
            assert (4 if o['src'] == 0 else o['cin']) == ch[o['src']]
            assert o['dst_coff'] + o['cout'] <= ch[o['dst']]
            if o['src2'] >= 0:
                assert ch[o['src2']] == o['cout']
        if o['type'] in (OP_UPADD,):
            assert o['dst'] in version and ch[o['src']] == ch[o['dst']]
        if o['type'] == OP_CONV and o['dst_coff'] == 0 and o['cout'] == ch[o['dst']] or o['type'] in (OP_MAXPOOL,):
            version[o['dst']] = version.get(o['dst'], 0) + 1
        else:
            version.setdefault(o['dst'], 0)
    assert t._out_buf in version
    # every conv has exactly one weight slot and parameters under the reference's names
    slots = [o['wslot'] for o in P.ops if o['type'] == OP_CONV]
    assert sorted(slots) == list(range(len(P.convs)))
    names = dict(t.named_modules())
    for conv_path, bn_path, cout, cin, k in P.convs:
        assert tuple(names[conv_path].weight.shape) == (cout, cin, k, k)
        assert names[bn_path].running_var.shape == (cout,)


def test_program_matches_oracle_op_counts():
    """conv counts of the compiled programs equal the oracle modules' (53 / 311 / 305 convs, SURVEY B.1, B.3)."""
    import torch.nn as nn
    from oracle import resnet as orn, hrnet as ohr
    from spec_b200.backbone import Trunk
    for arch, ref in (('resnet50', orn.resnet50()), ('hrnet_w32', ohr.hrnet_w32(use_conv=True))):
        n_ref = sum(isinstance(m, nn.Conv2d) for m in ref.modules())
        assert len(Trunk(arch)._program.convs) == n_ref
    assert len(Trunk('hrnet_w32', use_conv=False)._program.convs) == 305


def test_camcalib_wire_format_roundtrip(tmp_path):
    """The CamCalib -> SPEC hand-off file (scripts/camcalib_demo.py:135-140,174; README.md:97-104) can still be written
    and read back by read_cam_params-style code when the fused in-process path is used."""
    import joblib
    import numpy as np
    from spec_b200.cam_utils import save_camcalib_pkl, load_camcalib_pkl
    ang = torch.tensor([[0.9, 0.1, -0.05], [1.2, -0.2, 0.3]])
    f = torch.tensor([1100.0, 700.0])
    paths = save_camcalib_pkl(str(tmp_path), ['a.jpg', 'sub/b.png'], ang, f)
    d = joblib.load(paths[1])
    assert set(d) == {'vfov', 'f_pix', 'pitch', 'roll'} and abs(float(d['pitch']) + 0.2) < 1e-6
    R, K, vfov, pitch, roll, fl = load_camcalib_pkl(str(tmp_path), 'b.png', (1080, 1920))
    assert K[0, 2] == 960 and K[1, 2] == 540 and K[2, 2] == 0 and abs(fl - 700.0) < 1e-6
    assert R.shape == (3, 3) and abs(float(torch.linalg.det(R)) - 1) < 1e-5


@pytest.mark.parametrize('backbone', ['resnet50', 'resnet34', 'hrnet_w32-conv', 'hrnet_w32-interp'])
def test_compiled_program_equals_oracle_on_cpu(backbone):
    """Interpret the compiled op program with torch on the CPU (tests/program_interp.py) and compare with the oracle
    trunk: validates the architecture compilation, buffer reuse, BN folding, fuse order and concat offsets -- the whole
    host side of the trunk -- without a GPU."""
    from tests.program_interp import run_program
    prod, ref = make_pair(backbone, seed=9, amplify=False)
    torch.manual_seed(0)
    x = torch.randn(2, 3, 64, 96)
    with torch.no_grad():
        want = ref.backbone(x)
    got = run_program(prod.backbone, x)
    assert got.shape == want.shape
    err = (got - want).abs().max().item()
    assert err < 2e-3 * max(1.0, want.abs().max().item()), err


def test_header_is_plain_c_and_links(tmp_path):
    """include/specb200.h must be consumable from C (extern "C", plain pointers and sizes, no C++ or torch types): compile a C
    translation unit that references every declared entry point with gcc -std=c99 -pedantic, link it against libspecb200.so and
    run it (host-only calls: ABI version, an error path, the crop-transform arithmetic)."""
    import re
    import shutil
    import subprocess
    from spec_b200 import _lib
    if shutil.which('gcc') is None:
        pytest.skip('gcc not available')
    _lib.lib()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(root, 'include', 'specb200.h')).read()
    names = sorted(set(re.findall(r'\b(specb200_[a-z0-9_]+)\s*\(', hdr)))
    assert set(names) == set(_lib.EXPORTED_SYMBOLS)
    src = ['#include "specb200.h"', '#include <stdio.h>', '#include <math.h>', 'typedef void (*fn_t)(void);', 'int main(void) {', '    fn_t syms[] = {']
    src += [f'        (fn_t)&{n},' for n in names]
    src += ['    };',
            '    double box[4] = {100.0, 60.0, 64.0, 64.0}, trans[6], inv[6];',
            '    if (specb200_abi_version() != 1) return 2;',
            '    if (specb200_preproc_crop_transforms(box, 1, 1.0, 64, trans, inv) != 0) return 3;',
            '    if (fabs(trans[0] - 1.0) > 1e-9 || fabs(trans[2] - (32.0 - 100.0)) > 1e-9 || fabs(inv[5] - (60.0 - 32.0)) > 1e-9) return 4;',
            '    if (specb200_preproc_crop_transforms(0, 1, 1.0, 64, trans, inv) == 0) return 5;     /* error path */',
            '    if (specb200_last_error()[0] == 0) return 6;',
            '    printf("%d symbols\\n", (int)(sizeof(syms) / sizeof(syms[0])));',
            '    return 0;', '}']
    c = tmp_path / 'use_abi.c'
    c.write_text('\n'.join(src))
    exe = tmp_path / 'use_abi'
    libdir = os.path.dirname(_lib.LIB_PATH)
    r = subprocess.run(['gcc', '-std=c99', '-pedantic', '-Wall', '-Werror', '-I', os.path.join(root, 'include'), str(c), '-o', str(exe),
                        '-L', libdir, '-l:libspecb200.so', f'-Wl,-rpath,{libdir}', '-lm'], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    assert r.stdout.strip() == f'{len(names)} symbols'


# ------------------------------------------------------------------------------------------- round-2 behaviours (ADVICE r1)
def test_missing_assets_raise(monkeypatch, tmp_path):
    """Without an explicit opt-in a missing SMPL model / mean-parameter file raises like the reference does; the synthetic
    stand-ins need SPECB200_SYNTHETIC_ASSETS=1 (or explicit smpl_data= / mean_params=)."""
    from spec_b200 import hmr as H
    monkeypatch.setenv('SPECB200_SYNTHETIC_ASSETS', '0')
    monkeypatch.setattr(H, 'SMPL_MODEL_DIR', str(tmp_path / 'nope'))
    monkeypatch.setattr(H, 'SMPL_MEAN_PARAMS', str(tmp_path / 'nope.npz'))
    with pytest.raises(FileNotFoundError, match='SMPL'):
        H.SMPL()
    with pytest.raises(FileNotFoundError, match='SYNTHETIC_ASSETS'):
        H.HMRHead(512)
    with pytest.raises(FileNotFoundError):
        sb.HMR('resnet34', use_cam=True, use_cam_feats=True)
    from spec_b200.synthetic import synthetic_smpl_data, synthetic_mean_params
    sb.HMR('resnet34', use_cam=True, use_cam_feats=True, smpl_data=synthetic_smpl_data(0), mean_params=synthetic_mean_params(0))   # explicit data: fine


def test_smpl_pkl_and_npz_are_accepted(monkeypatch, tmp_path):
    """A standard SPEC data directory ships SMPL_NEUTRAL.pkl (smplx); an .npz export works too (scipy-sparse J_regressor,
    (6890,3,207) posedirs and 300 shape components are normalised to the smplx buffer shapes)."""
    import pickle
    import scipy.sparse as sp
    from spec_b200 import hmr as H
    from spec_b200.synthetic import synthetic_smpl_data
    d = synthetic_smpl_data(3)
    raw = {'v_template': d['v_template'].astype(np.float64), 'shapedirs': np.concatenate([d['shapedirs'], np.zeros((6890, 3, 2), np.float32)], 2),
           'posedirs': d['posedirs'].T.reshape(6890, 3, 207), 'J_regressor': sp.csc_matrix(d['J_regressor']), 'weights': d['lbs_weights']}
    mdir = tmp_path / 'smpl'
    mdir.mkdir()
    with open(mdir / 'SMPL_NEUTRAL.pkl', 'wb') as fh:
        pickle.dump(raw, fh)
    np.save(tmp_path / 'jx.npy', d['J_regressor_extra'])
    monkeypatch.setenv('SPECB200_SYNTHETIC_ASSETS', '0')
    monkeypatch.setattr(H, 'SMPL_MODEL_DIR', str(mdir))
    monkeypatch.setattr(H, 'JOINT_REGRESSOR_TRAIN_EXTRA', str(tmp_path / 'jx.npy'))
    got = H.SMPL()
    for k in ('v_template', 'shapedirs', 'posedirs', 'J_regressor', 'lbs_weights', 'J_regressor_extra'):
        assert torch.equal(getattr(got, k), torch.as_tensor(d[k]).float()), k


def test_training_mode_forward_raises():
    """Inference only: a forward in training mode with autograd enabled raises instead of silently training nothing."""
    from spec_b200 import _lib
    m = sb.CameraRegressorNetwork('resnet34')
    with torch.enable_grad():
        m.train()
        with pytest.raises(RuntimeError, match='inference path only'):
            _lib.refuse_training(m)
        m.eval()
        _lib.refuse_training(m)                          # eval mode: fine
    m.train()
    with torch.no_grad():
        _lib.refuse_training(m)                          # no autograd: fine


def test_checkpoint_loading_aliases_and_reports(tmp_path):
    """HMR.load_pretrained is non-strict like the reference's (hmr.py:124-135) but REPORTS unfilled tensors; the HRNet tail is
    accepted under both spellings (``downsample_layers.{i}`` here / ``downsample_stage_{i+1}`` believed upstream)."""
    from spec_b200.synthetic import synthetic_smpl_data, synthetic_mean_params
    kw = dict(use_cam=True, use_cam_feats=True, smpl_data=synthetic_smpl_data(0), mean_params=synthetic_mean_params(0))
    src = sb.HMR('hrnet_w32-conv', **kw)
    with torch.no_grad():
        for p in src.backbone.parameters():
            p.add_(1.0)
    flat = {}
    for k, v in list(src.backbone.state_dict().items()) + list(src.head.state_dict().items()):
        for i in range(3):
            k = k.replace(f'downsample_layers.{i}.', f'downsample_stage_{i + 1}.')
        flat[k] = v.clone()
    path = tmp_path / 'ckpt.pt'
    torch.save({'model': flat}, path)
    dst = sb.HMR('hrnet_w32-conv', **kw)
    assert dst.load_pretrained(str(path)) == []
    for (k, a), (_, b) in zip(src.backbone.state_dict().items(), dst.backbone.state_dict().items()):
        assert torch.equal(a, b), k
    # a checkpoint that lacks the tail: loud, not silent
    torch.save({'model': {k: v for k, v in flat.items() if 'downsample_stage' not in k}}, path)
    with pytest.raises(RuntimeError, match='downsample_layers'):
        sb.HMR('hrnet_w32-conv', **kw).load_pretrained(str(path))
    with pytest.warns(UserWarning, match='random'):
        missing = sb.HMR('hrnet_w32-conv', **kw).load_pretrained(str(path), strict_report=False)
    assert len(missing) == 6 * 5 and all('downsample_layers' in m for m in missing)


def test_inplace_parameter_updates_are_noticed():
    """Packed device copies are keyed on the tensors' in-place version counters (optimizer steps / param.data.copy_)."""
    t = sb.backbone.resnet18()
    assert t._weights_changed()                          # nothing packed yet
    t._watch = sb._lib.VersionWatch(t)
    assert not t._weights_changed()
    with torch.no_grad():
        t.layer1._modules['0'].conv1.weight.mul_(2.0)
    assert t._weights_changed()


def test_dependent_launch_rule_holds_for_every_kernel():
    """Source lint for the programmatic-dependent-launch rule (csrc/common.cuh): a kernel that is launched through
    ``launch_dep`` may start before its stream predecessor has finished, so it must execute ``griddep_wait()`` before it
    touches activations.  Every ``__global__`` kernel of the library that is NOT launched with ``<<<...>>>`` somewhere is
    launched through ``launch_dep`` (directly or through a function-pointer alias) and has to contain the wait; and no
    kernel may be launched both ways."""
    csrc = os.path.join(ROOT, 'spec_b200', 'csrc')
    text = {f: open(os.path.join(csrc, f)).read() for f in sorted(os.listdir(csrc)) if f.endswith(('.cu', '.cuh'))}
    kernels = {}
    for f, s in text.items():
        for m in re.finditer(r'__global__\s+void\s+(?:__\w+__\s*\([^)]*\)\s*)*(\w+)\s*\(', s):
            i = s.index('{', m.end())
            depth, j = 0, i
            while True:                                            # brace-match the kernel body
                depth += {'{': 1, '}': -1}.get(s[j], 0)
                j += 1
                if depth == 0:
                    break
            kernels[m.group(1)] = (f, s[i:j])
    assert len(kernels) > 25, sorted(kernels)
    allsrc = '\n'.join(text.values())
    plain = {k for k in kernels if re.search(r'\b' + k + r'\b\s*(<[^;()]*?>)?\s*<<<', allsrc)}
    dep = {k for k in kernels if re.search(r'launch_dep\(\s*' + k + r'\b', allsrc)}
    aliased = {k for k in kernels if re.search(r'auto\s+\w+\s*=\s*' + k + r'\b', allsrc)}     # k0 = conv_tcp_kernel<...>; launched via launch_dep(k0, ...)
    assert dep and aliased
    assert not (plain & (dep | aliased)), sorted(plain & (dep | aliased))
    assert (dep | aliased | plain) == set(kernels), sorted(set(kernels) - (dep | aliased | plain))
    for k in sorted(dep | aliased):
        f, body = kernels[k]
        assert 'griddep_wait()' in body, f'{f}: {k} is launched with programmatic dependent launch but never calls griddep_wait()'
        first_ret = body.find('return;')
        assert first_ret < 0 or body.find('griddep_wait()') < first_ret, f'{f}: {k} can return before griddep_wait()'
