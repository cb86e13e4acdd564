"""The full SPEC inference step as BASELINE.json times it: CamCalib(images) -> angles -> (R, K) ->
HMR(images, R, K, boxes) -> packed per-image output record, optionally captured in one CUDA graph
and sharded over ranks with ONE all-gather of the packed records (SURVEY.md 8e).

This replaces, in-process, the subprocess + pkl hand-off of the reference demo
(/root/reference/spec/tester.py:86-88, spec/utils/cam_params.py:24-50) and the per-key
``.cpu().numpy()`` loop (spec/tester.py:153-154).
"""
import torch

from . import _lib
from .constants import RECORD_LAYOUT, RECORD_FLOATS
from .camcalib import CameraRegressorNetwork
from .hmr import HMR

_OFFSETS = {}
_off = 0
for _k, _n, _s in RECORD_LAYOUT:
    _OFFSETS[_k] = (_off, _n, _s)
    _off += _n


def unpack_record(record):
    """(B, RECORD_FLOATS) -> dict of strided views (no copy); works on the local or the gathered buffer."""
    B = record.shape[0]
    return {k: record[:, o:o + n].view((B,) + s) for k, (o, n, s) in _OFFSETS.items()}


class SPECPipeline:
    def __init__(self, camcalib: CameraRegressorNetwork, hmr: HMR, use_graph=True):
        if not (hmr.use_cam and hmr.use_cam_feats):
            raise ValueError('the SPEC pipeline uses HMR(use_cam=True, use_cam_feats=True) (spec/tester.py:53-59)')
        self.camcalib, self.hmr = camcalib, hmr
        self.use_graph = use_graph
        self._graph = None
        self._static = None
        self._keep = None
        self._precisions = None
        self._bound = None

    # ---- eager
    def _step(self, images, bbox_scale, bbox_center, img_w, img_h, record):
        B = images.shape[0]
        out = {k: (record[:, _OFFSETS[k][0]:_OFFSETS[k][0] + _OFFSETS[k][1]].view((B,) + _OFFSETS[k][2]), RECORD_FLOATS)
               for k in _lib.OUTPUT_KEYS}
        o, n, _ = _OFFSETS['cam_angles']
        # The two trunks run one after the other on one stream.  CamCalib on a side stream beside the HMR trunk was measured
        # slower on B200 (12.5 vs 8.2 ms/step at B=256): the conv kernels are persistent one-CTA-per-SM kernels with ~200 KB
        # of smem, so two of them time-slice instead of back-filling.
        angles, R, K, _ = self.camcalib.predict_camera(images, img_h, img_w)
        record[:, o:o + n].copy_(angles)
        self.hmr(images, R, K, bbox_scale, bbox_center, img_w, img_h, _out=out)
        return record

    @torch.no_grad()
    def forward_packed(self, images, bbox_scale, bbox_center, img_w, img_h, bind_inputs=False):
        """Returns the (B, 21294) fp32 record buffer.  With use_graph the buffer is reused between calls.

        ``bind_inputs=True`` (serving loops that refill the SAME device staging buffers every step): the CUDA graph is
        captured directly on the caller's tensors -- no device-to-device copy of the 154 MB image batch into a private static
        buffer -- and cached per set of buffer addresses (up to 4 sets, e.g. the two halves of a double-buffered H2D ring).
        The caller promises that the tensors stay allocated and keep their addresses."""
        _lib.require_device(images)
        if not self.use_graph:
            rec = torch.empty(images.shape[0], RECORD_FLOATS, dtype=torch.float32, device=images.device)
            return self._step(images, bbox_scale, bbox_center, img_w, img_h, rec)
        if bind_inputs:
            return self._replay_bound(images, bbox_scale, bbox_center, img_w, img_h)
        st = self._static
        if st is None or st['images'].shape != images.shape or st['images'].device != images.device or self._weights_stale():
            self._capture(images, bbox_scale, bbox_center, img_w, img_h)
            st = self._static
        st['images'].copy_(images, non_blocking=True)
        st['bbox_scale'].copy_(bbox_scale, non_blocking=True)
        st['bbox_center'].copy_(bbox_center, non_blocking=True)
        st['img_w'].copy_(img_w, non_blocking=True)
        st['img_h'].copy_(img_h, non_blocking=True)
        self._graph.replay()
        return st['record']

    def _replay_bound(self, images, bbox_scale, bbox_center, img_w, img_h):
        args = (images, bbox_scale, bbox_center, img_w, img_h)
        for t in args:
            if not (torch.is_tensor(t) and t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
                raise ValueError('bind_inputs=True needs contiguous fp32 CUDA tensors for every input')
        if self._weights_stale() or self._bound is None:
            self._graph, self._static, self._keep = None, None, None
            self._bound = {}
        key = tuple(t.data_ptr() for t in args) + (tuple(images.shape),)
        ent = self._bound.get(key)
        if ent is None:
            if len(self._bound) >= 4:
                self._bound.pop(next(iter(self._bound)))
            dev = images.device
            rec = torch.empty(images.shape[0], RECORD_FLOATS, dtype=torch.float32, device=dev)
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):                        # warm-up: packs weights, sizes workspaces, sets attributes
                for _ in range(2):
                    self._step(*args, rec)
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._step(*args, rec)
            keep = [self.hmr._ws, self.camcalib._ws] + list(self.hmr.backbone._ws.values()) + list(self.camcalib.backbone._ws.values()) + list(args)
            ent = self._bound[key] = (g, rec, keep)
            self._precisions = (self.hmr.backbone.precision, self.camcalib.backbone.precision)
        ent[0].replay()
        return ent[1]

    def _weights_stale(self):
        """The captured graph baked in the device pointers of the packed weights: any event that makes a module re-pack
        (load_state_dict, .to(), set_precision, an in-place parameter update) must drop the graph BEFORE the old handles are
        released, or the replay would read freed memory."""
        mods = (self.hmr, self.hmr.backbone, self.camcalib, self.camcalib.backbone)
        return (any(m._dirty for m in mods) or self.hmr._weights_changed() or self.hmr.backbone._weights_changed()
                or self.camcalib.backbone._weights_changed() or self._precisions != (self.hmr.backbone.precision, self.camcalib.backbone.precision))

    def _capture(self, images, bbox_scale, bbox_center, img_w, img_h):
        self._graph, self._static, self._keep = None, None, None       # drop the old graph first (it holds raw pointers)
        self._bound = None
        dev = images.device
        B = images.shape[0]
        f = lambda t, shape: torch.empty((B,) + shape, dtype=torch.float32, device=dev).copy_(
            torch.as_tensor(t).to(dev, torch.float32).reshape((B,) + shape))
        st = {'images': images.detach().clone().float().contiguous(), 'bbox_scale': f(bbox_scale, ()),
              'bbox_center': f(bbox_center, (2,)), 'img_w': f(img_w, ()), 'img_h': f(img_h, ()),
              'record': torch.empty(B, RECORD_FLOATS, dtype=torch.float32, device=dev)}
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):                    # warm-up: packs weights, sizes workspaces, sets attributes
            for _ in range(2):
                self._step(st['images'], st['bbox_scale'], st['bbox_center'], st['img_w'], st['img_h'], st['record'])
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self._step(st['images'], st['bbox_scale'], st['bbox_center'], st['img_w'], st['img_h'], st['record'])
        # the graph baked in raw workspace pointers: keep those tensors alive for as long as the graph lives
        self._keep = [self.hmr._ws, self.camcalib._ws] + list(self.hmr.backbone._ws.values()) + list(self.camcalib.backbone._ws.values())
        self._graph, self._static = g, st
        self._precisions = (self.hmr.backbone.precision, self.camcalib.backbone.precision)

    def __call__(self, images, bbox_scale, bbox_center, img_w, img_h):
        return unpack_record(self.forward_packed(images, bbox_scale, bbox_center, img_w, img_h))

    @torch.no_grad()
    def run_on_frame(self, frame, detections, bgr=False, camcalib_min_size=600, crop_size=224, preprocessor=None):
        """One iteration of the demo loop (/root/reference/spec/tester.py:99-167) for a frame that is already on the GPU:
        ``frame`` uint8 (H, W, 3) [``bgr=True`` if it is what cv2.imread returns]; ``detections`` (N, 4) host array of
        (c_x, c_y, size, size) boxes as the detector produces them (tester.py:101,116).

        CamCalib sees the whole frame at min-side ``camcalib_min_size`` (camcalib/pano_dataset.py:156-162) and yields ONE
        camera for the frame (scripts/camcalib_demo.py:112-140, f_pix from the original height); every detection is
        cropped on the device (tester.py:118-125), ``bbox_scale = size / 200``, ``bbox_center = (c_x, c_y)``
        (tester.py:127-128).  Returns the output dict for the N detections plus ``cam_angles`` (N, 3) and the crops
        (``inp_images``); an empty dict when there are no detections (tester.py:102-103 skips the frame)."""
        import numpy as np
        from .preprocess import default_preprocessor
        _lib.require_device(frame)
        det = np.asarray(detections, dtype=np.float64).reshape(-1, 4)
        n = det.shape[0]
        if n == 0:
            return {}
        P = preprocessor or default_preprocessor()
        dev = frame.device
        H, W = int(frame.shape[0]), int(frame.shape[1])
        full = P.resize(frame, min_size=camcalib_min_size, bgr=bgr)
        angles, R, K, _ = self.camcalib.predict_camera(full, H, W)
        crops = P.crop(frame, det, scale=1.0, crop_size=crop_size, bgr=bgr)
        bbox_scale = torch.as_tensor(det[:, 2] / 200.0, dtype=torch.float32).to(dev)
        bbox_center = torch.as_tensor(det[:, :2], dtype=torch.float32).to(dev)
        img_h = torch.full((n,), float(H), dtype=torch.float32, device=dev)
        img_w = torch.full((n,), float(W), dtype=torch.float32, device=dev)
        out = self.hmr(crops, R.expand(n, 3, 3).contiguous(), K.expand(n, 3, 3).contiguous(), bbox_scale, bbox_center, img_w, img_h)
        out = dict(out)
        out['cam_angles'] = angles.expand(n, 3)
        out['inp_images'] = crops
        return out

    def launches_per_step(self):
        """Kernels of libspecb200 enqueued by one step (trunk x2 + both tails + decode)."""
        return self.camcalib.backbone.last_launches() + 2 + self.hmr.last_launches()


def all_gather_records(record, group=None):
    """ONE collective per step: every rank contributes its (B_local, 21294) record block; returns the
    (world*B_local, 21294) buffer, rank-major (= image order under a contiguous batch split)."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    out = torch.empty(world * record.shape[0], record.shape[1], dtype=record.dtype, device=record.device)
    dist.all_gather_into_tensor(out, record.contiguous(), group=group)
    return out


class RecordGatherer:
    """Overlapped form of ``all_gather_records`` for a steady-state loop: the gather of step i runs on NCCL's stream
    while step i+1 computes.  Two send/receive buffer pairs alternate; ``submit`` returns the gathered buffer of the
    PREVIOUS step (None on the first call), ``flush`` the last one."""

    def __init__(self, batch_local, device, group=None):
        import torch.distributed as dist
        self.dist, self.group = dist, group
        world = dist.get_world_size(group)
        self.send = [torch.empty(batch_local, RECORD_FLOATS, dtype=torch.float32, device=device) for _ in range(2)]
        self.recv = [torch.empty(world * batch_local, RECORD_FLOATS, dtype=torch.float32, device=device) for _ in range(2)]
        self.work = [None, None]
        self.i = 0

    def submit(self, record):
        k = self.i & 1
        if self.work[k] is not None:          # buffers k were used two steps ago
            self.work[k].wait()
        self.send[k].copy_(record, non_blocking=True)             # the graph's record buffer is overwritten by the next replay
        self.work[k] = self.dist.all_gather_into_tensor(self.recv[k], self.send[k], group=self.group, async_op=True)
        prev = None
        if self.i > 0:
            self.work[k ^ 1].wait()
            prev = self.recv[k ^ 1]
        self.i += 1
        return prev

    def flush(self):
        if self.i == 0:
            return None
        k = (self.i - 1) & 1
        self.work[k].wait()
        return self.recv[k]


class PeerGatherer:
    """The ONE collective of the data path as a PUT over NVLink peer memory (``specb200_allgather_outputs``,
    spec_b200/csrc/gather.cu) instead of an NCCL kernel: every rank's receive region is mapped by all peers through CUDA
    IPC (handles exchanged once with ``all_gather_object``); per step each rank's copy engines write its
    (B_local, 21294) fp32 block into all peers' regions (``mode='copy'``, SM-free) or one small kernel stores it
    (``mode='push'``), followed by a sequence-number flag exchange.  Same interface as ``RecordGatherer``: ``submit``
    returns the gathered buffer of the PREVIOUS step (its gather ran under this step's compute), valid until the next
    ``submit``; ``flush`` returns the last one.

    Three receive slots: a peer's PUT of step i into slot i%3 is issued after it observed this rank's signal of step
    i-1, which this rank's gather stream issues only after (an event covering) everything the caller enqueued up to its
    ``submit(i-1)`` call -- i.e. after all consumers of the buffer returned by ``submit(i-2)`` (slot (i-3)%3 = i%3)."""

    SLOTS = 3

    def __init__(self, batch_local, device, group=None, mode=None):
        import ctypes as C
        import os
        import torch.distributed as dist
        self.dist, self.group, self.device = dist, group, torch.device(device)
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.batch_local = batch_local
        mode = mode or os.environ.get('SPECB200_GATHER', 'copy')
        if mode not in ('copy', 'push'):
            raise ValueError("PeerGatherer mode must be 'copy' or 'push'")
        self.mode = mode
        L = _lib.lib()
        block = batch_local * RECORD_FLOATS * 4
        h = C.c_void_p()
        handle = (C.c_uint8 * 64)()
        with torch.cuda.device(self.device):
            _lib.check(L.specb200_gather_create(C.byref(h), self.rank, self.world, block, self.SLOTS, handle))
            self._h = h
            handles = [None] * self.world
            dist.all_gather_object(handles, bytes(handle), group=group)
            blob = (C.c_uint8 * (64 * self.world)).from_buffer_copy(b''.join(handles))
            _lib.check(L.specb200_gather_connect(h, blob))
        dist.barrier(group)                                    # every rank has mapped every region before the first PUT
        self.stream = torch.cuda.Stream(device=self.device, priority=-1)
        self.done = [None] * self.SLOTS
        self.i = 0
        self._views = {}

    def _recv(self, slot):
        """(world * B_local, 21294) fp32 view of receive slot ``slot`` (library-owned memory, no copy)."""
        v = self._views.get(slot)
        if v is None:
            ptr = _lib.lib().specb200_gather_recv_ptr(self._h, slot)

            class _Wrap:                                        # zero-copy view of library-owned device memory
                __cuda_array_interface__ = {'shape': (self.world * self.batch_local, RECORD_FLOATS), 'typestr': '<f4',
                                            'data': (int(ptr), False), 'version': 2}
            with torch.cuda.device(self.device):
                v = self._views[slot] = torch.as_tensor(_Wrap(), device=self.device)
        return v

    def submit(self, record):
        main = torch.cuda.current_stream(self.device)
        k = self.i % self.SLOTS
        B = self.batch_local
        # own block: copied on the CALLER's stream (the pipeline's record buffer is overwritten by its next graph replay), after
        # the consumers of slot k's previous content, which the caller enqueued before this call
        own = self._recv(k)[self.rank * B:(self.rank + 1) * B]
        own.copy_(record, non_blocking=True)
        ready = torch.cuda.Event()
        ready.record(main)
        self.stream.wait_event(ready)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().specb200_allgather_outputs(self._h, own.data_ptr(), k, self.i // self.SLOTS + 1,
                                                             0 if self.mode == 'copy' else 1, self.stream.cuda_stream))
        self.done[k] = torch.cuda.Event()
        self.done[k].record(self.stream)
        prev = None
        if self.i > 0:
            kp = (self.i - 1) % self.SLOTS
            main.wait_event(self.done[kp])
            prev = self._recv(kp)
        self.i += 1
        return prev

    def flush(self):
        if self.i == 0:
            return None
        k = (self.i - 1) % self.SLOTS
        torch.cuda.current_stream(self.device).wait_event(self.done[k])
        return self._recv(k)

    def close(self):
        if getattr(self, '_h', None) is not None:
            torch.cuda.synchronize(self.device)
            self.dist.barrier(self.group)                      # nobody unmaps while a peer may still PUT
            _lib.lib().specb200_gather_destroy(self._h)
            self._h = None


def make_gatherer(batch_local, device, group=None):
    """PeerGatherer when the peer-memory path can be set up on every rank (SPECB200_GATHER=copy|push, default copy), else the
    NCCL RecordGatherer (SPECB200_GATHER=nccl forces it).  Returns (gatherer, description)."""
    import os
    import torch.distributed as dist
    want = os.environ.get('SPECB200_GATHER', 'copy')
    if want != 'nccl':
        ok, err = 1, ''
        g = None
        try:
            g = PeerGatherer(batch_local, device, group, mode=want)
        except Exception as e:                                  # no peer access / IPC refused in this container
            ok, err = 0, repr(e)[:200]
        flag = torch.tensor([ok], device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
        if int(flag.item()) == 1:
            return g, f'peer-memory PUT over NVLink ({"copy engines" if want == "copy" else "push kernel"}), specb200_allgather_outputs'
        import warnings
        warnings.warn(f'peer-memory gather unavailable ({err or "failed on another rank"}): falling back to NCCL all-gather')
    return RecordGatherer(batch_local, device, group), 'NCCL all_gather_into_tensor (RecordGatherer)'


def shard_range(total, rank, world):
    """Contiguous batch split (SURVEY.md 8e): rank r owns images [lo, hi)."""
    per = (total + world - 1) // world
    lo = min(rank * per, total)
    return lo, min(lo + per, total)


def bind_process_to_gpu_numa(device_index):
    """Pin the calling process to the CPUs that are local to GPU ``device_index`` (sysfs ``local_cpulist`` of its PCI function)
    so that the pinned host staging buffers it allocates afterwards land on the GPU's NUMA node.  A serving / eval process
    that feeds 19 GB/s of images to one B200 (31 k img/s x 602 KB) through staging buffers on the REMOTE socket was measured
    at ~22 k img/s end to end instead of ~31 k.  Returns a dict describing what was done (for logs); never raises."""
    import os
    info = {'bound': False}
    try:
        import pynvml as nv
        nv.nvmlInit()
        vis = os.environ.get('CUDA_VISIBLE_DEVICES')
        idx = int(vis.split(',')[device_index]) if vis and vis.split(',')[0].isdigit() else device_index
        bus = nv.nvmlDeviceGetPciInfo(nv.nvmlDeviceGetHandleByIndex(idx)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        dom, rest = bus.split(':', 1)
        dev_dir = f'/sys/bus/pci/devices/{dom[-4:].lower()}:{rest.lower()}'
        cpus = set()
        for part in open(dev_dir + '/local_cpulist').read().strip().split(','):
            if part:
                lo, _, hi = part.partition('-')
                cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0)
        local = allowed & cpus
        node = open(dev_dir + '/numa_node').read().strip()
        info.update(pci=bus, numa_node=node, local_cpus=len(cpus), allowed_cpus=len(allowed))
        if local and local != allowed:
            os.sched_setaffinity(0, local)
            info.update(bound=True, cpus=len(local), previous=sorted(allowed))
        # memory policy too (CPU affinity alone leaves page placement to first touch): prefer the GPU's node for every
        # allocation this thread makes from here on -- the pinned staging buffers.  set_mempolicy(MPOL_PREFERRED = 1)
        if node.lstrip('-').isdigit() and int(node) >= 0:
            import ctypes
            n = int(node)
            mask = (ctypes.c_ulong * 16)()
            mask[n // 64] = 1 << (n % 64)
            rc = ctypes.CDLL(None, use_errno=True).syscall(238, 1, mask, ctypes.c_ulong(16 * 64 + 1))
            info['mempolicy'] = 'preferred:%d' % n if rc == 0 else 'set_mempolicy failed (errno %d)' % ctypes.get_errno()
    except Exception as e:                                   # no sysfs / no NVML / restricted container: leave the affinity alone
        info['error'] = repr(e)[:120]
    return info


def unbind_process(info):
    """Undo ``bind_process_to_gpu_numa`` for every thread of the process (OpenMP workers inherited the mask) and restore the
    default memory policy."""
    import ctypes
    import os
    if info.get('bound'):
        for tid in os.listdir('/proc/self/task'):
            try:
                os.sched_setaffinity(int(tid), info['previous'])
            except OSError:
                pass
    if str(info.get('mempolicy', '')).startswith('preferred'):
        ctypes.CDLL(None).syscall(238, 0, None, ctypes.c_ulong(0))          # MPOL_DEFAULT
