"""Runs the UNMODIFIED reference wrapper code of the hot path -- camcalib/model.py (CameraRegressorNetwork),
spec/models/hmr.py (HMR), camcalib/cam_utils.py (convert_preds_to_angles) and spec/utils/cam_params.py (read_cam_params) of a
checkout of the original SPEC repository -- and writes what it produced to tests/golden/reference_wrappers.npz and
tests/golden/reference_wrappers_alt_seeds.npz, plus the reference's own name tables, soft-argmax bin ranges and public
signatures to tests/golden/reference_tables.json.

Those four files import the un-vendored ``pare`` package (requirements.txt:28, no commit pinned; not installable offline).
``install_pare_stubs`` puts stand-ins for exactly the names they import into ``sys.modules`` -- backed by the oracle's
restatements of the pare / smplx internals (oracle/resnet.py, hrnet.py, head.py, geometry.py) -- and ``load_reference`` then
executes the reference files from where they lie (importlib, by path; nothing is copied).  So everything that IS in
the reference for this path -- constructor wiring, the eval()-by-name backbone selection, the forward glue, the cam_vfov
formula, the soft-argmax bin ranges built from scipy/np.linspace, the pkl hand-off and K assembly -- is the reference's own
code producing the fixtures; what stays recalled is pare's / smplx's internals behind the stubs (oracle/__init__.py).

    python -m tests.golden.reference_wrappers <path to a SPEC checkout>          # regenerate the fixtures

tests/test_reference_wrappers.py, tests/test_oracle.py and tests/test_boundary.py compare oracle/models.py, oracle/geometry.py,
oracle/constants.py and the product's signatures with these committed fixtures; the tests never read the reference itself.
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
FIXTURE = os.path.join(GOLDEN, 'reference_wrappers.npz')
ALT_FIXTURE = os.path.join(GOLDEN, 'reference_wrappers_alt_seeds.npz')
TABLES = os.path.join(GOLDEN, 'reference_tables.json')
_STUB_NAMES = ['pare', 'pare.models', 'pare.models.backbone', 'pare.models.backbone.utils', 'pare.models.backbone.hrnet',
               'pare.models.head', 'pare.models.layers', 'pare.models.layers.softargmax', 'pare.utils', 'pare.utils.geometry',
               'pare.utils.train_utils']


def install_pare_stubs():
    """sys.modules stand-ins for the pare names the four reference files import (and nothing else)."""
    from oracle import resnet as o_resnet, hrnet as o_hrnet, head as o_head, geometry as o_geo, models as o_models
    from spec_b200.synthetic import synthetic_smpl_data, synthetic_mean_params
    smpl, mean = synthetic_smpl_data(0), synthetic_mean_params(0)
    mods = {n: types.ModuleType(n) for n in _STUB_NAMES}
    for n in _STUB_NAMES:
        if '.' in n:
            parent, child = n.rsplit('.', 1)
            setattr(mods[parent], child, mods[n])
        mods[n].__path__ = []

    # pare.models.backbone: ``from pare.models.backbone import *`` + ``eval(backbone)(pretrained=True)`` (model.py:20,33; hmr.py:21,53)
    bb = mods['pare.models.backbone']
    for name in ('resnet18', 'resnet34', 'resnet50', 'resnet101'):
        setattr(bb, name, (lambda ctor: (lambda pretrained=False, **kw: ctor()))(getattr(o_resnet, name)))
    bb.__all__ = ['resnet18', 'resnet34', 'resnet50', 'resnet101']
    mods['pare.models.backbone.utils'].get_backbone_info = lambda b: {'n_output_channels': o_models.get_backbone_info(b)}
    mods['pare.models.backbone.hrnet'].hrnet_w32 = o_hrnet.hrnet_w32
    mods['pare.models.backbone.hrnet'].hrnet_w48 = o_hrnet.hrnet_w48

    class HMRHead(o_head.HMRHead):                       # ctor as called at hmr.py:57-64
        def __init__(self, num_input_features, estimate_var=False, use_separate_var_branch=False, uncertainty_activation='',
                     backbone='resnet50', use_cam_feats=False):
            assert not (estimate_var or use_separate_var_branch or uncertainty_activation)
            super().__init__(num_input_features, use_cam_feats=use_cam_feats, mean_params=mean)

    class SMPLCamHead(o_head.SMPLCamHead):               # hmr.py:69
        def __init__(self, img_res=224):
            super().__init__(smpl, img_res=img_res)

    class SMPLHead(o_head.SMPLHead):                     # hmr.py:71-74
        def __init__(self, focal_length=5000., img_res=224):
            super().__init__(smpl, focal_length=focal_length, img_res=img_res)

    hd = mods['pare.models.head']
    hd.HMRHead, hd.SMPLCamHead, hd.SMPLHead = HMRHead, SMPLCamHead, SMPLHead
    mods['pare.models.layers.softargmax'].softargmax1d = o_geo.softargmax1d
    mods['pare.utils.geometry'].batch_euler2matrix = o_geo.batch_euler2matrix

    def load_pretrained_model(model, state_dict, strict=False, overwrite_shape_mismatch=True):     # hmr.py:131 (not on the forward path)
        own = model.state_dict()
        model.load_state_dict({k: v for k, v in state_dict.items() if k in own and own[k].shape == v.shape}, strict=False)
    mods['pare.utils.train_utils'].load_pretrained_model = load_pretrained_model
    saved = {n: sys.modules.get(n) for n in _STUB_NAMES}
    sys.modules.update(mods)
    return saved


def remove_pare_stubs(saved):
    for n, m in saved.items():
        if m is None:
            sys.modules.pop(n, None)
        else:
            sys.modules[n] = m


def _load_by_path(ref_root, name, rel):
    spec = importlib.util.spec_from_file_location(name, os.path.join(ref_root, rel))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def load_reference(ref_root):
    """Executes the four reference files (unmodified, from the SPEC checkout at ``ref_root``) with the pare stubs in place."""
    saved = install_pare_stubs()
    try:
        return {'model': _load_by_path(ref_root, '_specref_camcalib_model', 'camcalib/model.py'),
                'hmr': _load_by_path(ref_root, '_specref_spec_models_hmr', 'spec/models/hmr.py'),
                'cam_utils': _load_by_path(ref_root, '_specref_camcalib_cam_utils', 'camcalib/cam_utils.py'),
                'cam_params': _load_by_path(ref_root, '_specref_spec_utils_cam_params', 'spec/utils/cam_params.py')}
    finally:
        remove_pare_stubs(saved)


# ------------------------------------------------------------------------------------------------------- the cases
# small shapes: the CPU suite must stay fast; the wrappers do not depend on the spatial size
CASES = {
    'spec_resnet50': dict(hmr='resnet50', camcalib='resnet50', fc_layers=1, batch=2, size=96, use_cam=True, use_cam_feats=True),
    'spec_hrnet_w32_conv': dict(hmr='hrnet_w32-conv', camcalib='resnet34', fc_layers=3, batch=2, size=64, use_cam=True, use_cam_feats=True),
    'hmr_resnet34_nocam': dict(hmr='resnet34', camcalib=None, fc_layers=1, batch=3, size=64, use_cam=False, use_cam_feats=False),
}
SEED0, ALT_SEED0 = 40, 60               # case i runs with seed SEED0 + i (FIXTURE) and ALT_SEED0 + i (ALT_FIXTURE)
# ALT_FIXTURE keeps every output but the vertices whole; of those it keeps this fixed sample, so that it stays small
ALT_VERTEX_IDS = np.sort(np.random.RandomState(0).choice(6890, 96, replace=False))


def alt_sample(out):
    """What ALT_FIXTURE stores of one case's outputs."""
    out = dict(out)
    out['hmr_smpl_vertices'] = out['hmr_smpl_vertices'][:, ALT_VERTEX_IDS]
    return out


def case_inputs(cfg, seed):
    from spec_b200.synthetic import synthetic_batch
    b = synthetic_batch(cfg['batch'], seed)
    g = torch.Generator().manual_seed(seed)
    b['images'] = torch.randn(cfg['batch'], 3, cfg['size'], cfg['size'], generator=g)
    return b


def oracle_models(cfg, seed):
    """Seeded oracle modules; the reference-side modules get their weights by state_dict (strict)."""
    from oracle import models as om
    from spec_b200.synthetic import synthetic_smpl_data, synthetic_mean_params, randomize_module_
    from tests.golden.make_golden import amplify_decoders_
    torch.manual_seed(seed)
    hmr = om.HMR(cfg['hmr'], use_cam=cfg['use_cam'], use_cam_feats=cfg['use_cam_feats'], smpl_data=synthetic_smpl_data(0),
                 mean_params=synthetic_mean_params(0)).eval()
    randomize_module_(hmr.backbone, seed)
    if not cfg['hmr'].startswith('hrnet'):
        amplify_decoders_(hmr)
    cc = None
    if cfg['camcalib']:
        cc = om.CameraRegressorNetwork(cfg['camcalib'], num_fc_layers=cfg['fc_layers']).eval()
        randomize_module_(cc.backbone, seed + 1)
        with torch.no_grad():
            for fc in (cc.fc_vfov, cc.fc_pitch, cc.fc_roll):
                for p in fc.parameters():
                    if p.dim() == 2:
                        p.mul_(8.0)
    return cc, hmr


@torch.no_grad()
def run_reference_case(ref, cfg, seed, tmpdir):
    """The demo / eval sequence with the reference's own functions: CameraRegressorNetwork.forward (model.py:72-81) ->
    convert_preds_to_angles(loss_type='softargmax_l2') (cam_utils.py:121-145; camcalib_demo.py:116-121) -> f_pix
    (camcalib_demo.py:127-129) -> pkl (camcalib_demo.py:131-140) -> read_cam_params (cam_params.py:24-50; tester.py:88) ->
    HMR.forward (hmr.py:82-122).  Returns a flat dict of numpy arrays."""
    import joblib
    cc_o, hmr_o = oracle_models(cfg, seed)
    b = case_inputs(cfg, seed)
    out = {}
    B = cfg['batch']
    hmr = ref['hmr'].HMR(backbone=cfg['hmr'], use_cam=cfg['use_cam'], use_cam_feats=cfg['use_cam_feats']).eval()
    hmr.load_state_dict(hmr_o.state_dict(), strict=True)
    if cfg['camcalib']:
        cc = ref['model'].CameraRegressorNetwork(backbone=cfg['camcalib'], num_fc_layers=cfg['fc_layers']).eval()
        cc.load_state_dict(cc_o.state_dict(), strict=True)
        logits = cc(b['images'])
        for n, l in zip(('vfov', 'pitch', 'roll'), logits):
            out['logits_' + n] = l.numpy()
        vfov, pitch, roll = ref['cam_utils'].convert_preds_to_angles(*logits, loss_type='softargmax_l2')
        out.update(cam_vfov=vfov.numpy(), cam_pitch=pitch.numpy(), cam_roll=roll.numpy())
        Rs, Ks = [], []
        os.makedirs(os.path.join(tmpdir, 'camcalib'), exist_ok=True)
        for i in range(B):
            h, w = float(b['img_h'][i]), float(b['img_w'][i])
            # camcalib_demo.py:123-140: numpy angles, f_pix from the ORIGINAL image height, one pkl per image.
            # ``orig_img_h / 2. / np.tan(pred_vfov / 2.)`` with a float32 0-d array and Python floats is FLOAT64 under the
            # value-based promotion of the NumPy 1.x the reference pins (numba==0.54.1 => numpy < 1.21); NumPy 2 (NEP 50,
            # this container) would keep float32 and read_cam_params' ``tensor[0, 0] = np.float32`` then raises.  The
            # widening is spelled out here so that the unmodified read_cam_params sees what the reference's demo wrote.
            v_np, p_np, r_np = vfov[i].numpy(), pitch[i].numpy(), roll[i].numpy()
            f_pix = h / 2. / np.tan(np.float64(v_np) / 2.)
            joblib.dump({'vfov': v_np, 'f_pix': f_pix, 'pitch': p_np, 'roll': r_np},
                        os.path.join(tmpdir, 'camcalib', f'img{i}.jpg.pkl'))
            R, K, *_ = ref['cam_params'].read_cam_params(tmpdir, f'/somewhere/img{i}.jpg', (h, w))
            Rs.append(R), Ks.append(K)
        R, K = torch.stack(Rs), torch.stack(Ks)
        out.update(cam_rotmat=R.numpy(), cam_intrinsics=K.numpy())
        res = hmr(b['images'], R, K, b['bbox_scale'], b['bbox_center'], b['img_w'], b['img_h'])
    else:
        res = hmr(b['images'])
    out['keys'] = np.array(list(res.keys()))
    for k, v in res.items():
        out['hmr_' + k] = v.numpy()
    return out


@torch.no_grad()
def run_oracle_case(cfg, seed):
    """Same sequence through oracle/models.py + oracle/geometry.py."""
    from oracle import geometry as og
    cc, hmr = oracle_models(cfg, seed)
    b = case_inputs(cfg, seed)
    out = {}
    if cc is not None:
        logits = cc(b['images'])
        for n, l in zip(('vfov', 'pitch', 'roll'), logits):
            out['logits_' + n] = l.numpy()
        vfov, pitch, roll = og.convert_preds_to_angles(*logits)
        R, K, _ = og.cam_params_from_angles(vfov, pitch, roll, b['img_h'], b['img_w'])
        out.update(cam_vfov=vfov.numpy(), cam_pitch=pitch.numpy(), cam_roll=roll.numpy(), cam_rotmat=R.numpy(), cam_intrinsics=K.numpy())
        res = hmr(b['images'], R, K, b['bbox_scale'], b['bbox_center'], b['img_w'], b['img_h'])
    else:
        res = hmr(b['images'])
    out['keys'] = np.array(list(res.keys()))
    for k, v in res.items():
        out['hmr_' + k] = v.numpy()
    return out


def reference_tables(ref_root, ref):
    """The reference's name tables (spec/constants.py), the end points of its soft-argmax bin tables (cam_utils.py:39,55) and
    the argument lists of the drop-in classes' constructors and forwards (model.py:25-31; hmr.py:29-41,82-91)."""
    import ast
    path = os.path.join(ref_root, 'spec', 'constants.py')
    ns = {}
    src = open(path).read()
    exec(compile(src.split('# Permutation of SMPL pose parameters')[0].replace('import numpy as np', ''), path, 'exec'),
         {'np': np}, ns)
    out = {k: ns[k] for k in ('JOINT_NAMES', 'JOINT_MAP', 'H36M_TO_J14', 'IMG_NORM_MEAN')}
    cu = ref['cam_utils']
    out['bins'] = {n: [float(np.min(getattr(cu, n))), float(np.max(getattr(cu, n)))] for n in ('vfov_bins', 'pitch_bins')}
    sigs = {}
    for rel, cls_name in (('spec/models/hmr.py', 'HMR'), ('camcalib/model.py', 'CameraRegressorNetwork')):
        tree = ast.parse(open(os.path.join(ref_root, rel)).read())
        cls = [n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == cls_name][0]
        for f in cls.body:
            if isinstance(f, ast.FunctionDef) and f.name in ('__init__', 'forward'):
                sigs[f'{cls_name}.{f.name}'] = [a.arg for a in f.args.args][1:]
    out['signatures'] = sigs
    return out


def main(ref_root, out_dir=GOLDEN):
    import json
    import tempfile
    if not os.path.exists(os.path.join(ref_root, 'spec', 'models', 'hmr.py')):
        raise SystemExit(f'{ref_root} is not a checkout of the SPEC repository')
    torch.set_num_threads(4)
    ref = load_reference(ref_root)
    blob, alt = {}, {'vertex_ids': ALT_VERTEX_IDS}
    differ = []
    with tempfile.TemporaryDirectory() as tmp:
        for i, (name, cfg) in enumerate(CASES.items()):
            for seed, dst, keep in ((SEED0 + i, blob, lambda o: o), (ALT_SEED0 + i, alt, alt_sample)):
                out = run_reference_case(ref, cfg, seed, tmp)
                ora = run_oracle_case(cfg, seed)       # same process, same CPU kernels: the oracle must agree bit for bit
                differ += [f'{name}/{k} (seed {seed})' for k in out if out[k].shape != ora[k].shape or not np.array_equal(out[k], ora[k])]
                for k, v in keep(out).items():
                    dst[f'{name}/{k}'] = v
    if differ:
        raise SystemExit('the oracle differs from the reference in ' + ', '.join(differ))
    for path, arrays in ((FIXTURE, blob), (ALT_FIXTURE, alt)):
        path = os.path.join(out_dir, os.path.basename(path))
        np.savez_compressed(path, **arrays)
        print('wrote', path, f'{os.path.getsize(path) / 1e6:.2f} MB,', len(arrays), 'arrays')
    path = os.path.join(out_dir, os.path.basename(TABLES))
    with open(path, 'w') as fh:
        json.dump(reference_tables(ref_root, ref), fh, indent=1)
        fh.write('\n')
    print('wrote', path)


if __name__ == '__main__':
    if len(sys.argv) not in (2, 3):
        raise SystemExit('usage: python -m tests.golden.reference_wrappers <SPEC checkout> [output directory]')
    main(*sys.argv[1:])
