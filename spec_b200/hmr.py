"""``HMR`` -- drop-in for /root/reference/spec/models/hmr.py:28-122.

Same constructor keywords, same ``forward(images, cam_rotmat, cam_intrinsics, bbox_scale, bbox_center,
img_w, img_h)`` (positional order is part of the contract: spec/trainer.py:139), same output dict
(``smpl_vertices (B,6890,3)``, ``smpl_joints3d (B,49,3)``, ``smpl_joints2d (B,49,2)``, ``pred_cam_t (B,3)``,
``pred_pose (B,24,3,3)``, ``pred_cam (B,3)``, ``pred_shape (B,10)``, ``pred_pose_6d (B,144)`` -- fp32
tensors on the input device, freshly allocated and writable), same state_dict names
(``backbone.*``, ``head.fc1/fc2/decpose/decshape/deccam.*``, ``head.init_pose/init_shape/init_cam``,
``smpl.smpl.*`` buffers).

Parameter containers only; all arithmetic runs in libspecb200 (trunk kernels + the fused fp32 tail).
"""
import ctypes as C
import os
import warnings

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from . import backbone as _bb
from .constants import JOINT_MAP_49, SMPL_VERTEX_IDS_21, SMPL_PARENTS
from .synthetic import synthetic_smpl_data, synthetic_mean_params

# where the reference keeps its assets (spec/config.py:35-38); all absent offline
SMPL_MODEL_DIR = os.environ.get('SPECB200_SMPL_DIR', 'data/body_models/smpl')
SMPL_MEAN_PARAMS = os.environ.get('SPECB200_SMPL_MEAN_PARAMS', 'data/smpl_mean_params.npz')
JOINT_REGRESSOR_TRAIN_EXTRA = os.environ.get('SPECB200_J_REGRESSOR_EXTRA', 'data/J_regressor_extra.npy')


def synthetic_assets_allowed():
    """Seeded synthetic SMPL constants / mean parameters stand in for the licensed assets ONLY on an explicit opt-in
    (``SPECB200_SYNTHETIC_ASSETS=1``: tests, bench, smoke -- there is no network to fetch the real files) or when the caller
    passes ``smpl_data=`` / ``mean_params=`` itself.  Otherwise a missing file raises, as the reference does
    (smplx raises on a missing model file; pare's HMRHead np.load()s SMPL_MEAN_PARAMS unconditionally)."""
    return os.environ.get('SPECB200_SYNTHETIC_ASSETS', '0') == '1'


def _dense(a):
    return np.asarray(a.toarray() if hasattr(a, 'toarray') else a)


def _read_smpl_file(path):
    """An ``.npz`` export or the ``SMPL_NEUTRAL.pkl`` smplx loads (a latin-1 pickle of arrays; the original chumpy-typed
    release needs ``chumpy`` importable or a one-off export: ``np.savez(npz, **{k: np.array(v) for k, v in pkl.items()})``)."""
    if path.endswith('.npz'):
        return dict(np.load(path, allow_pickle=False))
    import pickle
    try:
        with open(path, 'rb') as fh:
            return dict(pickle.load(fh, encoding='latin1'))
    except ModuleNotFoundError as e:                        # chumpy-typed original release
        raise RuntimeError(f'{path} needs the {e.name!r} package to unpickle; export it to SMPL_NEUTRAL.npz once '
                           '(see spec_b200/hmr.py::_read_smpl_file)') from e


def _load_smpl_data(gender='neutral', need_extra=True):
    """SMPL constants from ``SMPL_NEUTRAL.npz`` / ``SMPL_NEUTRAL.pkl`` under SMPL_MODEL_DIR (spec/config.py:35) plus
    ``J_regressor_extra.npy`` (config.py:36).  ``gender`` picks ``SMPL_{NEUTRAL,MALE,FEMALE}``; ``need_extra=False`` (the
    body model, which has no extra joints) does without ``J_regressor_extra.npy``."""
    if gender not in ('neutral', 'male', 'female'):
        raise ValueError(f"gender must be 'neutral', 'male' or 'female', got {gender!r}")
    stem = 'SMPL_' + gender.upper()
    cands = [os.path.join(SMPL_MODEL_DIR, stem + ext) for ext in ('.npz', '.pkl')]
    path = next((c for c in cands if os.path.exists(c)), None)
    if path is not None and (not need_extra or os.path.exists(JOINT_REGRESSOR_TRAIN_EXTRA)):
        d = _read_smpl_file(path)
        out = {k: _dense(d[k]).astype(np.float32) for k in ('v_template', 'shapedirs', 'J_regressor')}
        out['shapedirs'] = out['shapedirs'][:, :, :10]
        pd = _dense(d['posedirs']).astype(np.float32)
        out['posedirs'] = pd.reshape(-1, pd.shape[-1]).T if pd.ndim == 3 else pd
        out['lbs_weights'] = _dense(d['weights'] if 'weights' in d else d['lbs_weights']).astype(np.float32)
        if need_extra:
            out['J_regressor_extra'] = np.load(JOINT_REGRESSOR_TRAIN_EXTRA).astype(np.float32)
        out['parents'] = np.asarray(SMPL_PARENTS, dtype=np.int64)
        return out
    if not synthetic_assets_allowed():
        raise FileNotFoundError(
            f'SMPL model not found: looked for {cands}' + (f' and {JOINT_REGRESSOR_TRAIN_EXTRA!r}' if need_extra else '') +
            ' (set SPECB200_SMPL_DIR / SPECB200_J_REGRESSOR_EXTRA, pass smpl_data=, or opt in to seeded synthetic constants with '
            'SPECB200_SYNTHETIC_ASSETS=1)')
    warnings.warn(f'SMPL model not found under {SMPL_MODEL_DIR!r}: using seeded SYNTHETIC SMPL constants '
                  '(right shapes, meaningless geometry; SPECB200_SYNTHETIC_ASSETS=1)', stacklevel=3)
    return synthetic_smpl_data(('neutral', 'male', 'female').index(gender))


def _load_mean_params():
    if os.path.exists(SMPL_MEAN_PARAMS):
        d = np.load(SMPL_MEAN_PARAMS)
        return {'pose': d['pose'].astype(np.float32), 'shape': d['shape'].astype(np.float32),
                'cam': d['cam'].astype(np.float32)}
    if not synthetic_assets_allowed():
        raise FileNotFoundError(f'{SMPL_MEAN_PARAMS!r} not found (set SPECB200_SMPL_MEAN_PARAMS, pass mean_params=, or opt in to '
                                'seeded synthetic values with SPECB200_SYNTHETIC_ASSETS=1)')
    warnings.warn(f'{SMPL_MEAN_PARAMS!r} not found: using seeded SYNTHETIC mean parameters (SPECB200_SYNTHETIC_ASSETS=1)', stacklevel=3)
    return synthetic_mean_params(0)


class HMRHead(nn.Module):
    """Parameter container of pare's HMRHead (SURVEY.md A.3): fc1 (C+157[+7] -> 1024), fc2, three
    decoders, ``init_*`` buffers (name evidenced at /root/reference/scripts/spec_eval.py:57)."""

    def __init__(self, num_input_features, use_cam_feats=False, mean_params=None, **unused):
        super().__init__()
        npose = 144
        self.npose = npose
        self.use_cam_feats = use_cam_feats
        self.num_input_features = num_input_features
        self.fc1 = nn.Linear(num_input_features + npose + 13 + (7 if use_cam_feats else 0), 1024)
        self.drop1 = nn.Dropout()
        self.fc2 = nn.Linear(1024, 1024)
        self.drop2 = nn.Dropout()
        self.decpose = nn.Linear(1024, npose)
        self.decshape = nn.Linear(1024, 10)
        self.deccam = nn.Linear(1024, 3)
        for m in (self.decpose, self.decshape, self.deccam):
            nn.init.xavier_uniform_(m.weight, gain=0.01)
        mp = mean_params if mean_params is not None else _load_mean_params()
        self.register_buffer('init_pose', torch.as_tensor(mp['pose']).float().reshape(1, npose))
        self.register_buffer('init_shape', torch.as_tensor(mp['shape']).float().reshape(1, 10))
        self.register_buffer('init_cam', torch.as_tensor(mp['cam']).float().reshape(1, 3))

    def forward(self, *a, **k):
        raise RuntimeError('HMRHead is evaluated inside HMR.forward by libspecb200')


class SMPL(nn.Module):
    """Buffer container of pare.models.SMPL / smplx.SMPL (names as in smplx 0.1.28)."""

    def __init__(self, smpl_data=None):
        super().__init__()
        d = smpl_data if smpl_data is not None else _load_smpl_data()
        f = lambda k: torch.as_tensor(np.asarray(d[k])).float()
        self.register_buffer('v_template', f('v_template'))
        self.register_buffer('shapedirs', f('shapedirs'))
        self.register_buffer('posedirs', f('posedirs'))
        self.register_buffer('J_regressor', f('J_regressor'))
        self.register_buffer('lbs_weights', f('lbs_weights'))
        self.register_buffer('J_regressor_extra', f('J_regressor_extra'))
        self.register_buffer('parents', torch.as_tensor(np.asarray(d['parents'])).long())
        self.register_buffer('joint_map', torch.tensor(JOINT_MAP_49, dtype=torch.long))
        self.register_buffer('vertex_ids', torch.tensor(SMPL_VERTEX_IDS_21, dtype=torch.long))
        assert self.v_template.shape == (6890, 3) and self.posedirs.shape == (207, 20670)


class SMPLCamHead(nn.Module):
    def __init__(self, img_res=224, smpl_data=None):
        super().__init__()
        self.smpl = SMPL(smpl_data)
        self.img_res = img_res


class SMPLHead(nn.Module):
    def __init__(self, focal_length=5000., img_res=224, smpl_data=None):
        super().__init__()
        self.smpl = SMPL(smpl_data)
        self.focal_length = focal_length
        self.img_res = img_res


_OUT_SHAPES = {'smpl_vertices': (6890, 3), 'smpl_joints3d': (49, 3), 'smpl_joints2d': (49, 2), 'pred_cam_t': (3,),
               'pred_pose': (24, 3, 3), 'pred_cam': (3,), 'pred_shape': (10,), 'pred_pose_6d': (144,)}


class HMR(nn.Module):
    def __init__(self, backbone='resnet50', focal_length=5000., img_res=224, pretrained=None, use_cam=False, p=0.0,
                 estimate_var=False, use_separate_var_branch=False, uncertainty_activation='', use_cam_feats=False,
                 smpl_data=None, mean_params=None):
        super().__init__()
        if estimate_var or use_separate_var_branch or uncertainty_activation:
            raise NotImplementedError('uncertainty branches are never enabled on the SPEC hot path '
                                      '(spec/tester.py:53-59, spec/trainer.py:50-56)')
        if backbone.startswith('hrnet'):
            backbone, use_conv = backbone.split('-')                     # hmr.py:44-51
            self.backbone = getattr(_bb, backbone)(pretrained=True, downsample=True, use_conv=(use_conv == 'conv'))
        else:
            self.backbone = getattr(_bb, backbone)(pretrained=True)
        self.use_cam_feats = use_cam_feats
        self.head = HMRHead(num_input_features=_bb.get_backbone_info(backbone)['n_output_channels'],
                            use_cam_feats=use_cam_feats, mean_params=mean_params)
        self.use_cam = use_cam
        if use_cam:
            self.smpl = SMPLCamHead(img_res=img_res, smpl_data=smpl_data)
        else:
            self.smpl = SMPLHead(focal_length=focal_length, img_res=img_res, smpl_data=smpl_data)
        self.focal_length, self.img_res = focal_length, img_res
        self._handle = None
        self._dirty = True
        self._device = None
        self._ws = None
        self._graphs = {}
        self._module_graph = os.environ.get('SPECB200_MODULE_GRAPH', '1') != '0'
        self.graph_max_batch = 32
        self.register_load_state_dict_post_hook(lambda m, k: m._mark_dirty())
        if pretrained is not None:
            self.load_pretrained(pretrained)

    # ---- checkpoint helpers (hmr.py:124-135)
    def load_pretrained(self, file, strict_report=True):
        """hmr.py:124-135: backbone and head are filled from ONE flat state_dict, non-strictly.  Non-strict loading hides
        naming mismatches (the HRNet ``-conv`` tail is ``downsample_layers.{i}.*`` here; upstream pare is believed to call
        it ``downsample_stage_{i+1}.*`` -- un-checkable offline, so both spellings are accepted), so every backbone / head
        tensor that the checkpoint did NOT fill is reported: a RuntimeError with ``strict_report`` (default), else a warning."""
        sd = torch.load(file, map_location='cpu')
        sd = sd.get('model', sd.get('state_dict', sd))
        sd = {k[len('model.'):] if k.startswith('model.') else k: v for k, v in sd.items()}
        missing = self.load_flat_state_dict(sd)
        if missing:
            msg = (f'{file}: {len(missing)} backbone/head tensors were not found in the checkpoint and keep their random '
                   f'initialisation, e.g. {missing[:6]}')
            if strict_report:
                raise RuntimeError(msg)
            warnings.warn(msg, stacklevel=2)
        return missing

    _KEY_ALIASES = tuple((f'downsample_stage_{i + 1}.', f'downsample_layers.{i}.') for i in range(3))

    def load_flat_state_dict(self, sd):
        """Fills ``backbone`` and ``head`` from a flat (un-prefixed or ``backbone.`` / ``head.``-prefixed) state_dict; returns
        the list of own parameter/buffer names that stayed unfilled (``num_batches_tracked`` excluded)."""
        flat = {}
        for k, v in sd.items():
            for pre in ('backbone.', 'head.'):
                if k.startswith(pre):
                    k = k[len(pre):]
            for theirs, ours in self._KEY_ALIASES:
                if k.startswith(theirs):
                    k = ours + k[len(theirs):]
            flat[k] = v
        missing = []
        for name, mod in (('backbone', self.backbone), ('head', self.head)):
            own = mod.state_dict()
            take = {k: v for k, v in flat.items() if k in own and own[k].shape == v.shape}
            mod.load_state_dict(take, strict=False)
            missing += [f'{name}.{k}' for k in own if k not in take and not k.endswith('num_batches_tracked')]
        self._mark_dirty()
        self.backbone.mark_dirty()
        return missing

    # ---- engine
    def _mark_dirty(self):
        self._dirty = True

    def _apply(self, fn, *a, **k):
        self._dirty = True
        return super()._apply(fn, *a, **k)

    def _release(self):
        if self._handle is not None:
            _lib.lib().specb200_hmrtail_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self._release()
        except Exception:
            pass

    def _weights_changed(self):
        """True when a parameter / buffer of the head or the SMPL layer was modified in place (optimizer step,
        ``param.data.copy_``) since the folded weights were uploaded."""
        w = getattr(self, '_watch', None)
        return w is None or w.changed()

    def _ensure(self, device):
        if self._handle is not None and not self._dirty and self._device == device and not self._weights_changed():
            return
        _lib.require_device()
        self._release()
        self._graphs.clear()
        hd, sm = self.head, self.smpl.smpl
        keep = []

        def fp(t):
            t = t.detach().float().contiguous().cpu()
            keep.append(t)
            return t.data_ptr()

        def ip(t):
            t = t.detach().to(torch.int32).contiguous().cpu()
            keep.append(t)
            return t.data_ptr()

        p = _lib.HmrParams()
        p.in_features = hd.num_input_features
        p.use_cam_feats = int(self.use_cam_feats)
        p.use_cam = int(self.use_cam)
        p.focal_length = float(self.focal_length)
        p.img_res = float(self.img_res)
        p.fc1_w, p.fc1_b, p.fc2_w, p.fc2_b = fp(hd.fc1.weight), fp(hd.fc1.bias), fp(hd.fc2.weight), fp(hd.fc2.bias)
        p.decpose_w, p.decpose_b = fp(hd.decpose.weight), fp(hd.decpose.bias)
        p.decshape_w, p.decshape_b = fp(hd.decshape.weight), fp(hd.decshape.bias)
        p.deccam_w, p.deccam_b = fp(hd.deccam.weight), fp(hd.deccam.bias)
        p.init_pose, p.init_shape, p.init_cam = fp(hd.init_pose), fp(hd.init_shape), fp(hd.init_cam)
        p.v_template, p.shapedirs, p.posedirs = fp(sm.v_template), fp(sm.shapedirs), fp(sm.posedirs)
        p.J_regressor, p.lbs_weights, p.J_regressor_extra = fp(sm.J_regressor), fp(sm.lbs_weights), fp(sm.J_regressor_extra)
        p.parents, p.joint_map, p.vertex_ids = ip(sm.parents), ip(sm.joint_map), ip(sm.vertex_ids)
        h = C.c_void_p()
        with torch.cuda.device(device):
            _lib.check(_lib.lib().specb200_hmrtail_create(C.byref(h), C.byref(p)))
        self._handle = h
        self._x_ld = int(_lib.lib().specb200_hmrtail_x_ld(h))
        self._device = device
        self._dirty = False
        self._watch = _lib.VersionWatch(self.head, self.smpl)

    def _workspace(self, B, device):
        n = _lib.lib().specb200_hmrtail_workspace_bytes(self._handle, B)
        if self._ws is None or self._ws.numel() < n or self._ws.device != device:
            self._ws = torch.empty(n, dtype=torch.uint8, device=device)
        return self._ws

    @staticmethod
    def _f32(x, B, device, shape):
        if x is None:
            return None
        if not torch.is_tensor(x):
            x = torch.as_tensor(x)
        x = x.to(device=device, dtype=torch.float32)       # img_h / img_w arrive as int64 at trainer.py:239-240
        return x.reshape((B,) + shape).contiguous()

    def forward(self, images, cam_rotmat=None, cam_intrinsics=None, bbox_scale=None, bbox_center=None,
                img_w=None, img_h=None, _out=None):
        """``_out``: optional dict name -> (tensor view, per-image stride in floats) to write the outputs
        into caller-provided (e.g. packed all-gather) storage instead of fresh tensors.

        Small batches (the demo loop runs one forward per image with batch = #detections, spec/tester.py:143-151) are
        launch-bound (60 kernels of a few microseconds): for B <= ``graph_max_batch`` the forward is captured once per
        input shape into a CUDA graph and replayed (SPECB200_MODULE_GRAPH=0 disables)."""
        _lib.refuse_training(self)
        if (_out is None and self._module_graph and images.is_cuda and images.shape[0] <= self.graph_max_batch
                and images.shape[0] > 0 and not torch.cuda.is_current_stream_capturing()):
            return self._forward_graphed(images, cam_rotmat, cam_intrinsics, bbox_scale, bbox_center, img_w, img_h)
        return self._forward_impl(images, cam_rotmat, cam_intrinsics, bbox_scale, bbox_center, img_w, img_h, _out)

    def _forward_graphed(self, images, cam_rotmat, cam_intrinsics, bbox_scale, bbox_center, img_w, img_h):
        _lib.require_device(images)
        dev, B = images.device, images.shape[0]
        args = {'cam_rotmat': (cam_rotmat, (3, 3)), 'cam_intrinsics': (cam_intrinsics, (3, 3)), 'bbox_scale': (bbox_scale, ()),
                'bbox_center': (bbox_center, (2,)), 'img_w': (img_w, ()), 'img_h': (img_h, ())}
        key = (dev, tuple(images.shape), self.backbone.precision, tuple(k for k, (v, _) in args.items() if v is not None))
        if self._dirty or self.backbone._dirty or self._weights_changed() or self.backbone._weights_changed():
            self._graphs.clear()                                   # weights changed: captured graphs hold stale handles
        g = self._graphs.get(key)
        if g is None:
            st = {'images': torch.empty(images.shape, dtype=torch.float32, device=dev)}
            for k, (v, shp) in args.items():
                st[k] = None if v is None else torch.empty((B,) + shp, dtype=torch.float32, device=dev)
            def load():
                st['images'].copy_(images)
                for k, (v, shp) in args.items():
                    if v is not None:
                        st[k].copy_(self._f32(v, B, dev, shp))
            load()
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):                          # warm-up outside capture: packs weights, sizes workspaces
                self._forward_impl(st['images'], st['cam_rotmat'], st['cam_intrinsics'], st['bbox_scale'], st['bbox_center'],
                                   st['img_w'], st['img_h'], None)
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                outs = self._forward_impl(st['images'], st['cam_rotmat'], st['cam_intrinsics'], st['bbox_scale'],
                                          st['bbox_center'], st['img_w'], st['img_h'], None)
            if len(self._graphs) >= 8:
                self._graphs.pop(next(iter(self._graphs)))
            # the graph baked in raw workspace pointers: keep those tensors alive for as long as the graph lives
            keep = [self._ws] + list(self.backbone._ws.values())
            g = self._graphs[key] = (graph, st, outs, keep)
        graph, st, outs, _keep = g
        st['images'].copy_(images, non_blocking=True)
        for k, (v, shp) in args.items():
            if v is not None:
                st[k].copy_(self._f32(v, B, dev, shp), non_blocking=True)
        graph.replay()
        return {k: v.clone() for k, v in outs.items()}             # fresh tensors owned by the caller

    def _forward_impl(self, images, cam_rotmat, cam_intrinsics, bbox_scale, bbox_center, img_w, img_h, _out):
        _lib.require_device(images)
        dev = images.device
        B = images.shape[0]
        if B == 0:
            raise ValueError('empty batch')
        if self.use_cam or self.use_cam_feats:
            if cam_rotmat is None or cam_intrinsics is None or img_h is None:
                raise ValueError('cam_rotmat, cam_intrinsics and img_h are required with use_cam / use_cam_feats')
        if self.use_cam and (bbox_scale is None or bbox_center is None or img_w is None):
            raise ValueError('bbox_scale, bbox_center and img_w are required with use_cam')
        self._ensure(dev)
        R = self._f32(cam_rotmat, B, dev, (3, 3))
        K = self._f32(cam_intrinsics, B, dev, (3, 3))
        bs = self._f32(bbox_scale, B, dev, ())
        bc = self._f32(bbox_center, B, dev, (2,))
        iw = self._f32(img_w, B, dev, ())
        ih = self._f32(img_h, B, dev, ())
        ws = self._workspace(B, dev)
        # trunk writes the pooled feature straight into the head's input rows
        self.backbone.run(images, pooled=ws.data_ptr(), pooled_ld=self._x_ld)
        o = _lib.HmrOutputs()
        result = {}
        for key in _lib.OUTPUT_KEYS:
            if _out is not None:
                t, ld = _out[key]
            else:
                t = torch.empty((B,) + _OUT_SHAPES[key], dtype=torch.float32, device=dev)
                ld = int(np.prod(_OUT_SHAPES[key]))
            result[key] = t
            setattr(o, key, t.data_ptr())
            setattr(o, 'ld_' + key.split('_', 1)[1], ld)
        ptr = lambda t: t.data_ptr() if t is not None else 0
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().specb200_hmrtail_forward(
                self._handle, B, ws.data_ptr(), ws.numel(), ptr(R), ptr(K), ptr(bs), ptr(bc), ptr(iw), ptr(ih),
                C.byref(o), torch.cuda.current_stream(dev).cuda_stream))
        # same insertion order as the reference: smpl_output first, then updated with hmr_output (hmr.py:113)
        return {k: result[k] for k in ('smpl_vertices', 'smpl_joints3d', 'smpl_joints2d', 'pred_cam_t',
                                       'pred_pose', 'pred_cam', 'pred_shape', 'pred_pose_6d')}

    def last_launches(self):
        n = self.backbone.last_launches()
        if self._handle is not None:
            n += int(_lib.lib().specb200_hmrtail_last_launches(self._handle))
        return n
