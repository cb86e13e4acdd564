"""Times one batch of the SPEC evaluation protocol (compute_error.py:142-203: two SMPL forwards, the 14- and 24-joint world
and camera-frame errors, vertex errors) two ways on the same inputs:

  * spec_b200.SPECErrorEval.batch (BodyModel + the eval kernels, nothing leaves the device);
  * the way the reference runs it: the oracle's torch ops on the GPU (SMPL, regressions, rotations) and the Procrustes /
    vertex errors in numpy on the host after ``.cpu()`` (oracle.body_eval / oracle.eval_metrics).

CUDA events around each call after a warm-up; prints images/s, the card's name and power limit, one JSON line per size.

    python tools/eval_protocol_time.py [--sizes 256 2048] [--iters 20]
"""
import argparse
import json
import os
import subprocess
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault('SPECB200_SYNTHETIC_ASSETS', '1')

import spec_b200 as sb                                      # noqa: E402
from spec_b200.synthetic import synthetic_smpl_data          # noqa: E402
from oracle import body_eval as ob, eval_metrics as oe       # noqa: E402
from oracle.constants import H36M_TO_J14                     # noqa: E402


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                  # the measurement is still valid; say the card was not read
        q = f'unavailable ({e})'
    return torch.cuda.get_device_name(0), q


def inputs(B, dev, seed=0):
    g = np.random.RandomState(seed)
    t = lambda a: torch.from_numpy(np.asarray(a, np.float32)).to(dev)
    smpl = synthetic_smpl_data(0)
    J = g.rand(17, 6890) ** 8
    J = (J / J.sum(1, keepdims=True)).astype(np.float32)
    gt_pose, gt_betas = t(g.randn(B, 72) * 0.4), t(g.randn(B, 10))
    gt_pose_cam = gt_pose.clone()
    gt_pose_cam[:, :3] = t(g.randn(B, 3) * 0.8)
    rot = lambda s: ob.batch_rodrigues(torch.from_numpy(g.randn(B, 3) * s)).float().to(dev)
    bm = sb.BodyModel(smpl_data=smpl).to(dev)
    gv = bm(betas=gt_betas, global_orient=gt_pose[:, :3], body_pose=gt_pose[:, 3:]).vertices
    pred = 1.05 * torch.bmm(gv, rot(0.3).transpose(1, 2)) + 0.01 * torch.randn(gv.shape, device=dev, generator=torch.Generator(dev).manual_seed(seed))
    return dict(smpl=smpl, J=J, bm=bm, pred=pred.contiguous(), gt_pose=gt_pose, gt_pose_cam=gt_pose_cam, gt_betas=gt_betas,
                pred_cam_rotmat=rot(0.6))


def reference_batch(x, sm, Jh, Jr):
    """compute_error.py:142-203 (pose_cam branch) as the reference runs it: torch on the GPU, numpy SVD on the host."""
    pred = x['pred']
    gt_v, gt_j = ob.smpl_forward(sm, x['gt_betas'], x['gt_pose'][:, :3], x['gt_pose'][:, 3:])
    gc_v, gc_j = ob.smpl_forward(sm, x['gt_betas'], x['gt_pose_cam'][:, :3], x['gt_pose_cam'][:, 3:])
    pj = torch.einsum('bik,ji->bjk', [pred, Jr])
    pv_cam = torch.bmm(x['pred_cam_rotmat'], pred.transpose(2, 1)).transpose(2, 1)
    pcj = torch.einsum('bik,ji->bjk', [pv_cam, Jr])

    def eval_single(p, g):
        a, b = torch.matmul(Jh, p), torch.matmul(Jh, g)
        ap, bp = a[:, [0]].clone(), b[:, [0]].clone()
        a, b = a[:, H36M_TO_J14] - ap, b[:, H36M_TO_J14] - bp
        v2v = oe.compute_error_verts((p - ap).cpu().numpy(), (g - bp).cpu().numpy())
        pa = oe.reconstruction_error(a.cpu().numpy(), b.cpu().numpy())
        return torch.sqrt(((a - b) ** 2).sum(-1)).mean(-1).cpu().numpy(), pa, v2v

    def eval_j_24(p, g):
        p, g = p - p[:, [0]].clone(), g - g[:, [0]].clone()
        pa = oe.reconstruction_error(p.cpu().numpy(), g.cpu().numpy())
        return torch.sqrt(((p - g) ** 2).sum(-1)).mean(-1).cpu().numpy(), pa

    out = eval_single(pred, gt_v) + eval_single(pv_cam, gc_v) + eval_j_24(pj, gt_j) + eval_j_24(pcj, gc_j)
    return out


def timed(fn, iters):
    fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(iters):
        fn()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / iters


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('--sizes', type=int, nargs='+', default=[256, 2048])
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--ref-iters', type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('no CUDA device: this tool measures on the GPU only')
    dev = torch.device('cuda:0')
    name, smi = card()
    for B in a.sizes:
        x = inputs(B, dev)
        ev = sb.SPECErrorEval(x['J'], x['bm']).to(dev)
        run = lambda: ev.batch(x['pred'], x['gt_pose'], x['gt_betas'], x['pred_cam_rotmat'], gt_pose_cam=x['gt_pose_cam'])
        ms = timed(run, a.iters)
        sm = types.SimpleNamespace(**{k: torch.as_tensor(v).float().to(dev) for k, v in x['smpl'].items() if k != 'parents'})
        Jh, Jr = torch.from_numpy(x['J']).to(dev), sm.J_regressor
        with torch.device(dev):                          # the oracle builds its identity / padding tensors on the default device
            ms_ref = timed(lambda: reference_batch(x, sm, Jh, Jr), a.ref_iters)
        print(json.dumps({'batch': B, 'spec_b200_ms': round(ms, 4), 'spec_b200_images_per_s': round(B / ms * 1e3, 1),
                          'reference_style_ms': round(ms_ref, 3), 'reference_style_images_per_s': round(B / ms_ref * 1e3, 1),
                          'iters': a.iters, 'ref_iters': a.ref_iters, 'device': name, 'nvidia_smi_name_power_limit': smi}))


if __name__ == '__main__':
    main()
