"""CPU oracle for the SPEC inference hot path — TEST INFRASTRUCTURE, NOT PRODUCT.

This package restates, in plain fp32 PyTorch on the CPU, the arithmetic of the
reference path CamCalib -> backbone -> HMR head -> SMPL/LBS -> projection
(SURVEY.md section 8a, Appendix A).  Only ``tests/``, ``__graft_entry__.smoke()``
and the ``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may import
it.  The product (``spec_b200``) never does, and fails loudly without its CUDA
library.

PARITY STATUS: the WRAPPER LAYER of the path is pinned to outputs of the reference's own code; the ResNet trunk is pinned
to torchvision; the INPUT SIDE is pinned bit-exactly to cv2 / Pillow / torchvision; the internals of pare's HRNet / HMRHead /
SMPL and of smplx's LBS remain restated from the published algorithms -- *parity unpinned* for those.

The reference keeps the arithmetic of this path in two un-vendored third-party packages -- ``pare``
(git+https://github.com/mkocabas/PARE.git, NO commit pinned, /root/reference/requirements.txt:28) and ``smplx==0.1.28``
(requirements.txt:7) -- neither of which is present offline, and it ships no tests, golden vectors or fixtures
(SURVEY.md section 4, 8c).  What IS pinned, and how:

* the four reference files that hold this path's own code -- camcalib/model.py:24-81 (CameraRegressorNetwork),
  spec/models/hmr.py:28-122 (HMR), camcalib/cam_utils.py:39-63,110-145 (soft-argmax decode, bin tables) and
  spec/utils/cam_params.py:24-50 (pkl hand-off, R / K assembly) -- are EXECUTED UNMODIFIED from /root/reference with ``pare``
  stubbed in sys.modules by this package's restatements (tests/golden/reference_wrappers.py).  oracle/models.py and
  oracle/geometry.py agree with them BIT FOR BIT on three configurations (checked whenever tests/golden/reference_wrappers.py regenerates
  the fixtures), and the outputs of that reference run are committed as tests/golden/reference_wrappers.npz, which
  the oracle (CPU test) and the CUDA path (tests/test_gpu_parity.py::test_against_reference_wrapper_fixture) are compared
  with everywhere.  That run surfaced one real discrepancy, fixed in geometry.cam_params_from_angles: the demo computes
  f_pix in NumPy float64 (NumPy-1.x promotion) before it is stored in the float32 K;
* the ResNet trunk is checked layer-for-layer against torchvision's own ``resnet50``/``resnet34`` (pare's trunk is a copy of
  torchvision's with avgpool/fc removed) in tests/test_oracle.py;
* the input side (oracle/preprocess.py: person crops and the CamCalib resize) is pinned bit-exactly against cv2 / Pillow /
  torchvision, which ARE installed here;
* name tables are diffed against /root/reference/spec/constants.py:20-113 when it is mounted; domain invariants (rotation
  orthonormality, identity-pose LBS, optical-axis projection, soft-argmax of uniform logits) and oracle-made golden vectors
  (tests/golden/spec_resnet50_b2.npz) are tested.

STILL RECALLED (behind the stubs): pare.models.backbone.hrnet (architecture and parameter names of the ``-conv`` / ``-interp``
tails), pare.models.head.HMRHead (concatenation order of the camera features), pare.models.head.SMPLCamHead / pare.models.SMPL
(the 54-candidate joint assembly), pare.utils.geometry (rot6d, convert_pare_to_full_img_cam, perspective_projection,
batch_euler2matrix), pare.models.layers.softargmax1d, smplx.lbs -- SURVEY.md Appendix A.
"""
