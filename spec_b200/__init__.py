"""spec_b200 -- B200-native (sm_100a) implementation of the SPEC per-image inference hot path:
CamCalib camera regression -> camera-conditioned SMPL regression -> SMPL mesh -> projection.

Drop-in modules (same constructors / forward signatures / state_dict names as the reference):
  ``spec_b200.CameraRegressorNetwork``  for /root/reference/camcalib/model.py
  ``spec_b200.HMR``                     for /root/reference/spec/models/hmr.py
All arithmetic runs in libspecb200.so (hand-written CUDA behind a C ABI, include/specb200.h).
There is no CPU fallback: forward() on a non-sm_100 device raises.
"""
from .camcalib import CameraRegressorNetwork
from .hmr import HMR, HMRHead, SMPLCamHead, SMPLHead
from .backbone import get_backbone_info, resnet18, resnet34, resnet50, resnet101, hrnet_w32, hrnet_w48
from .cam_utils import convert_preds_to_angles, decode_logits
from .pipeline import (SPECPipeline, unpack_record, all_gather_records, shard_range, RecordGatherer, PeerGatherer, make_gatherer,
                       bind_process_to_gpu_numa, unbind_process)
from .metrics import EvalMetrics, SPECErrorEval, joint_errors
from .body_model import BodyModel
from .preprocess import Preprocessor, get_single_image_crop_demo, camcalib_transform

__all__ = ['CameraRegressorNetwork', 'HMR', 'HMRHead', 'SMPLCamHead', 'SMPLHead', 'get_backbone_info',
           'resnet18', 'resnet34', 'resnet50', 'resnet101', 'hrnet_w32', 'hrnet_w48',
           'convert_preds_to_angles', 'decode_logits', 'SPECPipeline', 'unpack_record', 'all_gather_records',
           'shard_range', 'RecordGatherer', 'PeerGatherer', 'make_gatherer', 'bind_process_to_gpu_numa', 'unbind_process', 'EvalMetrics', 'SPECErrorEval', 'joint_errors', 'BodyModel', 'Preprocessor', 'get_single_image_crop_demo',
           'camcalib_transform']
