#!/usr/bin/env python
"""bench.py -- images/sec of the SPEC full forward (CamCalib -> (R,K) -> HMR -> SMPL -> projection),
224x224, batch 256 per GPU (BASELINE.json configs[2]; weak scaling over GPUs), synthetic data, random weights.

  python bench.py --gpus 1 --steps 20 --warmup 5              # our arm (B200, libspecb200)
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
         bench.py --gpus N --steps K --warmup W               # N ranks, one per GPU, NCCL all-gather of records
  python bench.py --impl reference --steps 3 --warmup 3       # the reference path's CPU restatement (oracle)
  python bench.py --steps 20 --warmup 5 --dump-outputs DIR     # also write the last timed step's outputs to DIR/<name>.npy

Prints ONE JSON line (contract in the task statement): value = whole-job images/s with inputs resident in HBM,
e2e = same metric through the public API with pinned-host inputs (H2D and D2H inside the timed region),
roofline = conv FLOPs / event-timed conv-kernel time against the measured bf16 peak, cpu_baseline = the oracle
on the host cores for a bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import warnings

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
warnings.simplefilter('ignore')

import torch  # noqa: E402

METRIC = 'images/sec SPEC fwd (224^2, b256)'
UNIT = 'images/s'


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return {'hbm_gbs': d['hbm_gbs'], 'tf_burst': d['bf16_tflops'], 'tf_sustained': d.get('bf16_tflops_sustained', d['bf16_tflops']),
                'source': 'measured (MEASURED_PEAKS.json)'}
    return {'hbm_gbs': 6650.0, 'tf_burst': 1590.0, 'tf_sustained': 1400.0, 'source': 'fallback (B200_PROFILING.md)'}


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region through NVML: ``sample()`` -- called once in the middle of
    the K timed steps, while the GPU is busy with the steps already enqueued -- only WAKES a helper thread, which makes the
    one NVML query.  The launching thread must never block inside the timed loop: at 8 GPUs (driver's nvidia-smi poller
    holding NVML) an inline query blocked rank 0's host thread for ~190 ms, its launch queue drained and the all-gather
    stalled every rank (SCALE_r01.json: one 195 ms step).  Polling is out too: every NVML query perturbs the GPU briefly
    (10 Hz nvidia-smi: -20 %; a 20 Hz sampler thread: ~3 ms outlier steps), so exactly one query per request.
    Falls back to a slow nvidia-smi poll thread when pynvml is missing."""
    BITS = (('hw_slowdown', 0x8), ('hw_thermal_slowdown', 0x40), ('sw_thermal_slowdown', 0x20), ('sw_power_cap', 0x4))

    def __init__(self, index):
        self.index, self.sm, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._want = threading.Event()
        self.t = None
        self.mode = None
        self._nvml = None

    def sample(self):
        """Non-blocking: asks the helper thread for one NVML query."""
        self._want.set()

    def _nvml_loop(self):
        while True:
            self._want.wait()
            self._want.clear()
            if self._stop.is_set():
                return
            self._query()

    def _query(self):
        if self._nvml is None:
            return
        h, nv = self._nvml
        try:
            self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(nv, 'nvmlDeviceGetCurrentClocksEventReasons') \
                else nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            for name, bit in self.BITS:
                if r & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def _smi_loop(self):
        q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
            'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
        while not self._stop.is_set():
            try:
                o = subprocess.run(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader,nounits', '-i', str(self.index)],
                                   capture_output=True, text=True, timeout=5).stdout.strip().split(', ')
                self.sm.append(float(o[0])); self.max_mhz = float(o[1])
                for name, v in zip([b[0] for b in self.BITS], o[2:6]):
                    if v.strip().lower().startswith('active'):
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.5)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get('CUDA_VISIBLE_DEVICES')
            idx = int(vis.split(',')[self.index]) if vis and vis.split(',')[0].isdigit() else self.index
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.mode = 'nvml'
            self._nvml = (h, nv)
            self.t = threading.Thread(target=self._nvml_loop, daemon=True)
            self.t.start()
        except Exception:
            self.mode = 'nvidia-smi'
            self.t = threading.Thread(target=self._smi_loop, daemon=True)
            self.t.start()

    def stop(self):
        self._stop.set()
        self._want.set()
        if self.t is not None:
            self.t.join(3)
        sm = sorted(self.sm)
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons),
                'samples': len(sm), 'via': self.mode}


# =============================================================================================== reference arm / cpu baseline
def build_oracle(backbone):
    from oracle import models as om
    from spec_b200.synthetic import synthetic_smpl_data, synthetic_mean_params, randomize_module_
    torch.manual_seed(0)
    hmr = om.HMR(backbone, use_cam=True, use_cam_feats=True, smpl_data=synthetic_smpl_data(0),
                 mean_params=synthetic_mean_params(0)).eval()
    randomize_module_(hmr.backbone, 0)
    cc = om.CameraRegressorNetwork('resnet50').eval()
    randomize_module_(cc.backbone, 1)
    return cc, hmr


def pick_cpu_threads(cc, sample):
    """All the host threads the oracle can USE: eager PyTorch convs stop scaling (and collapse under
    oversubscription / cgroup quotas) well before 128 threads, so calibrate on one CamCalib forward and keep
    the fastest count among {8,16,32,64,all}."""
    try:
        avail = len(os.sched_getaffinity(0))
    except Exception:
        avail = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, avail) if c <= avail}) or [avail]
    x = torch.randn(sample, 3, 224, 224)
    best, best_t = cands[-1], float('inf')
    for c in cands:
        torch.set_num_threads(c)
        with torch.no_grad():
            cc(x)
            t0 = time.perf_counter()
            cc(x)
            dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    return best


def time_oracle(backbone, sample, steps, warmup):
    """Oracle (CPU restatement of the reference path) on the host cores; returns (images/s, ms per sample step, threads)."""
    from oracle.models import spec_full_forward
    from spec_b200.synthetic import synthetic_batch
    cc, hmr = build_oracle(backbone)
    cores = pick_cpu_threads(cc, sample)
    torch.set_num_threads(cores)
    b = synthetic_batch(sample, 0)
    args = (b['images'], b['bbox_scale'], b['bbox_center'], b['img_w'], b['img_h'])
    for _ in range(warmup):
        spec_full_forward(cc, hmr, *args)
    t0 = time.perf_counter()
    for _ in range(steps):
        spec_full_forward(cc, hmr, *args)
    dt = time.perf_counter() - t0
    return sample * steps / dt, dt / steps * 1e3, cores


def run_reference(a):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return                                                  # other ranks exit 0 without work
    sample = a.cpu_sample
    if a.batch <= 0:
        a.batch = 256
    ips, ms, cores = time_oracle(a.backbone, sample, a.steps, a.warmup)
    desc = f'{sample} of {a.batch} images per step (bounded CPU sample), fp32 PyTorch oracle, {cores} threads'
    _emit({
        'impl': 'reference', 'metric': METRIC, 'value': ips, 'unit': UNIT, 'n_gpus': a.gpus, 'steps': a.steps,
        'warmup': a.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': f'SPEC full forward (CamCalib->{a.backbone}->HMR head->SMPL->proj), 224x224, batch {a.batch}',
                   'backbone': a.backbone, 'note': 'reference arithmetic (pare/smplx) is not installable offline; this is its CPU restatement (oracle/)'},
        'cpu_baseline': {'value': ips, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': desc},
        'e2e': {'value': ips, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    })


# =============================================================================================== our arm
def host_link_probe(dev, nbytes=128 << 20):
    """Standalone pinned-host <-> device copy rates (GB/s) and the NUMA node(s) the pinned pages landed on -- printed next to
    ``e2e`` so that a link-bound e2e number can be told from a pipeline-bound one (VERDICT r1 item 7)."""
    import ctypes
    h = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    h.fill_(1)                                                     # touch: pages are placed now
    d = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    out = {}
    for name, (dst, src) in (('h2d_gbs', (d, h)), ('d2h_gbs', (h, d))):
        best = 0.0
        for _ in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            dst.copy_(src, non_blocking=True)
            e1.record()
            torch.cuda.synchronize(dev)
            best = max(best, nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9)
        out[name] = round(best, 2)
    try:                                                           # move_pages(2) with nodes=NULL reports each page's node
        libc = ctypes.CDLL(None, use_errno=True)
        n = 64
        step = nbytes // n
        pages = (ctypes.c_void_p * n)(*[(h.data_ptr() + i * step) & ~4095 for i in range(n)])
        status = (ctypes.c_int * n)()
        if libc.syscall(279, 0, ctypes.c_ulong(n), pages, None, status, 0) == 0:
            out['pinned_pages_numa_nodes'] = sorted({int(x) for x in status if x >= 0})
    except Exception:
        pass
    return out


def load_ncu_traffic(backbone, batch, precision):
    """dram__bytes_read.sum + dram__bytes_write.sum over the conv launches of ONE step, from the committed ``ncu --set full``
    summary of the current kernels (profiles/ncu_traffic.json, written by tools/summarize_ncu.py); None when there is no
    capture for this configuration."""
    p = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    try:
        d = json.load(open(p))
        e = d.get(f'{backbone}|{batch}|{precision}')
        return (e['bytes_per_step'], e.get('source')) if e else (None, None)
    except Exception:
        return None, None


def run_ours(a):
    import torch.distributed as dist
    import spec_b200 as sb
    from spec_b200.synthetic import synthetic_batch, synthetic_camera_matrices, synthetic_smpl_data, synthetic_mean_params, randomize_module_
    from spec_b200.constants import RECORD_FLOATS

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world != a.gpus:
        raise SystemExit(f'--gpus {a.gpus} but WORLD_SIZE={world}: launch N>1 with torch.distributed.run')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    numa = sb.bind_process_to_gpu_numa(local)                      # CPU affinity + memory policy: pinned staging on the GPU's node
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)

    c4 = a.mode == 'c4'                                            # BASELINE configs[3]: CamCalib bypassed, dataset-supplied (R, K)
    B = a.batch if a.batch > 0 else (128 if c4 else 256)           # per-GPU batch (weak scaling)
    torch.manual_seed(0)                                           # the heads' constructor initialisation: same weights every run
    cc = sb.CameraRegressorNetwork('resnet50')
    randomize_module_(cc.backbone, 1)
    hmr = sb.HMR(a.backbone, use_cam=True, use_cam_feats=True, smpl_data=synthetic_smpl_data(0), mean_params=synthetic_mean_params(0))
    randomize_module_(hmr.backbone, 0)
    for m in (cc, hmr):
        m.eval()
        m.backbone.set_precision(a.precision)
        m.backbone.chunk = a.chunk
        m.to(dev)
    pipe = sb.SPECPipeline(cc, hmr, use_graph=not a.no_graph)
    b = synthetic_batch(B, seed=rank, device=dev)                 # each rank generates its own shard
    args = (b['images'], b['bbox_scale'], b['bbox_center'], b['img_w'], b['img_h'])
    if c4:
        R, K = synthetic_camera_matrices(B, seed=rank, device=dev)        # what CamDataset reads from its npz (cam_dataset.py:617-653)
        orig_shape = torch.stack([b['img_h'], b['img_w']], 1).long()     # int64, as CamDataset yields it (cam_dataset.py:350,486)
        c4_rec = torch.empty(B, RECORD_FLOATS, dtype=torch.float32, device=dev)
        c4_out = {k: (v, RECORD_FLOATS) for k, v in sb.unpack_record(c4_rec).items() if k != 'cam_angles'}

    gatherer, gather_desc = (sb.make_gatherer(B, dev) if world > 1 else (None, None))

    c4_graphs = {}

    @torch.no_grad()
    def compute(inp=None, bound=False):
        if c4:                                                     # trainer.py:235-245 call, outputs written into the packed record
            im = inp['images'] if inp is not None else b['images']
            run = lambda: hmr(im, R, K, b['bbox_scale'], b['bbox_center'], orig_shape[:, 1], orig_shape[:, 0], _out=c4_out)
            if a.no_graph:
                run()
                return c4_rec
            g = c4_graphs.get(im.data_ptr())                       # one CUDA graph per (static) input buffer, like SPECPipeline
            if g is None:
                side = torch.cuda.Stream(device=dev)
                side.wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.stream(side):
                    run(); run()
                torch.cuda.current_stream(dev).wait_stream(side)
                torch.cuda.synchronize(dev)
                g = c4_graphs[im.data_ptr()] = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    run()
            g.replay()
            return c4_rec
        if inp is None:
            return pipe.forward_packed(*args)
        return pipe.forward_packed(inp['images'], inp['bbox_scale'], inp['bbox_center'], inp['img_w'], inp['img_h'], bind_inputs=bound)

    def step():
        rec = compute()
        if world > 1:
            return gatherer.submit(rec)                           # the ONE collective of the data path; overlaps the next step
        return rec

    def timed(fn, steps, warmup, mid=None):
        t_w = time.perf_counter()
        n_w = 0
        while n_w < warmup or time.perf_counter() - t_w < 0.4:     # >= W steps AND ~0.4 s so the clocks have ramped
            fn()
            n_w += 1
            if n_w % 4 == 0:
                torch.cuda.synchronize(dev)
        # events are created (and each recorded once, which is where CUDA really allocates them) BEFORE the bracket, so that
        # nothing but the record of e0 sits between the synchronize and the first timed step
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]     # per-step spread (diagnostic only)
        for ev in [e0, e1] + marks:
            ev.record()
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        e0.record()
        t_host0 = time.perf_counter()
        host_ms = []
        for i in range(steps):
            host_ms.append((time.perf_counter() - t_host0) * 1e3)  # when the launching thread STARTED enqueuing step i
            last = fn()
            marks[i].record()
            if mid is not None and i % 64 == min(steps // 2, 32):
                mid()                                              # wakes the NVML helper thread; never blocks this thread
        if gatherer is not None:
            last = gatherer.flush()                                # the last gather completes inside the timed region
        e1.record()
        torch.cuda.synchronize(dev)
        timed.last = last.cpu() if a.dump_outputs else None       # the buffer is reused by later calls: copy it out now
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        raw = [a_.elapsed_time(b_) for a_, b_ in zip([e0] + marks[:-1], marks)]
        per = sorted(raw)
        timed.step_ms = {'min': per[0], 'median': per[len(per) // 2], 'max': per[-1], 'argmax': raw.index(per[-1]),
                         'first_step_ms': raw[0], 'host_enqueue_start_ms': [round(h, 3) for h in host_ms[:4]]}
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)             # max over ranks
        return ms.item()

    # ---- value: inputs resident in HBM
    if a.profile_range:
        for _ in range(a.warmup):
            step()
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.start()
        for _ in range(a.steps):
            step()
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.stop()
        return None
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    total_ms = timed(step, a.steps, a.warmup, mid=sampler.sample if rank == 0 else None)
    step_spread = dict(timed.step_ms)
    if world > 1:                                                  # every rank's spread (which rank, which step was slow)
        spreads = [None] * world
        dist.all_gather_object(spreads, step_spread)
        step_spread['per_rank'] = spreads
    clocks = sampler.stop() if rank == 0 else None
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, timed.last, [k for k in c4_out] if c4 else None)
    ms_per_step = total_ms / a.steps
    value = world * B * a.steps / (total_ms * 1e-3)
    launches_per_step = hmr.last_launches() if c4 else pipe.launches_per_step()

    # ---- e2e: public API with HOST (pinned) inputs; every step copies its inputs H2D and its results D2H inside the
    # timed region.  The copies ride on side streams (double-buffered staging) so they overlap the previous /
    # next step's kernels -- what a serving loop built on the public API does.  The CUDA graph is captured directly on the two
    # staging sets (bind_inputs): no device-side copy of the inputs.
    link = host_link_probe(dev)
    host = {k: v.cpu().pin_memory() for k, v in b.items()}
    keys = ('images', 'bbox_scale', 'bbox_center', 'img_w', 'img_h')
    staging = [{k: torch.empty_like(host[k], device=dev) for k in keys} for _ in range(2)]
    rec_dev = [torch.empty(B, RECORD_FLOATS, dtype=torch.float32, device=dev) for _ in range(2)]
    host_rec = [torch.empty(B, RECORD_FLOATS, dtype=torch.float32).pin_memory() for _ in range(2)]
    s_h2d, s_d2h = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    main = torch.cuda.current_stream(dev)
    e2e_gather = None
    if world > 1:
        if gatherer is not None and hasattr(gatherer, 'close'):
            gatherer.close()                                       # frees the value loop's receive regions before the e2e ones exist
        e2e_gather, _ = sb.make_gatherer(B, dev)

    def e2e_run(steps):
        ev_h2d = [torch.cuda.Event() for _ in range(2)]
        ev_used = [None, None]
        ev_d2h = [None, None]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

        def issue_h2d(i):
            sl = i % 2
            with torch.cuda.stream(s_h2d):
                if ev_used[sl] is not None:
                    s_h2d.wait_event(ev_used[sl])                 # staging slot consumed by step i-2
                for k in keys:
                    staging[sl][k].copy_(host[k], non_blocking=True)
                ev_h2d[sl].record(s_h2d)

        def read_back(rec, sl):
            rec_dev[sl].copy_(rec, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(main)
            with torch.cuda.stream(s_d2h):
                s_d2h.wait_event(ev)
                host_rec[sl].copy_(rec_dev[sl], non_blocking=True)
                ev_d2h[sl] = torch.cuda.Event()
                ev_d2h[sl].record(s_d2h)

        with torch.cuda.stream(s_h2d):
            e0.record(s_h2d)
        issue_h2d(0)
        for i in range(steps):
            sl = i % 2
            if i + 1 < steps:
                issue_h2d(i + 1)
            main.wait_event(ev_h2d[sl])
            if ev_d2h[sl] is not None:
                main.wait_event(ev_d2h[sl])                       # rec_dev[sl] read back by step i-2
            rec = compute(staging[sl], bound=True)
            ev_used[sl] = torch.cuda.Event()
            ev_used[sl].record(main)                               # inputs consumed (the record is complete): slot may be refilled
            if world > 1:                                          # gather of step i overlaps step i+1; this rank reads back its own rows
                prev = e2e_gather.submit(rec)
                if prev is not None:
                    read_back(prev[rank * B:(rank + 1) * B], (i - 1) % 2)
            else:
                read_back(rec, sl)
        if world > 1:
            read_back(e2e_gather.flush()[rank * B:(rank + 1) * B], (steps - 1) % 2)
        with torch.cuda.stream(s_d2h):
            e1.record(s_d2h)
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1)

    e2e_steps = max(4, min(a.steps, 20))
    e2e_run(8)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    e2e_ms_t = torch.tensor([e2e_run(e2e_steps)], device=dev)
    if world > 1:
        dist.barrier()
        dist.all_reduce(e2e_ms_t, op=dist.ReduceOp.MAX)
    e2e_ms = e2e_ms_t.item()
    e2e_value = world * B * e2e_steps / (e2e_ms * 1e-3)
    h2d = sum(v.numel() * v.element_size() for v in host.values())
    d2h = host_rec[0].numel() * 4
    link['h2d_floor_ms_per_step'] = round(h2d / (link['h2d_gbs'] * 1e9) * 1e3, 3)
    link['d2h_floor_ms_per_step'] = round(d2h / (link['d2h_gbs'] * 1e9) * 1e3, 3)
    if world > 1:
        links = [None] * world
        dist.all_gather_object(links, link)
        link = {'per_rank': links}

    out = None
    if rank == 0:
        # ---- roofline: per-op CUDA-event timing of both trunks (live, eager, on the launching stream)
        peaks = load_peaks()
        conv_ms, conv_flops, step_ops_ms, conv_bytes = 0.0, 0.0, 0.0, 0
        trunks = (hmr,) if c4 else (cc, hmr)
        for m in trunks:
            m.backbone.profile_ops(b['images'])                   # warm
            rows = m.backbone.profile_ops(b['images'])
            conv_ms += sum(r['ms'] for r in rows if r['flops'] > 0)
            conv_flops += sum(r['flops'] for r in rows)
            conv_bytes += sum(r.get('bytes', 0) for r in rows if r['flops'] > 0)
            step_ops_ms += sum(r['ms'] for r in rows)
        achieved = conv_flops / (conv_ms * 1e-3) / 1e12
        n_conv = sum(1 for m in trunks for o in m.backbone._program.ops if o['type'] == 1)
        traffic, traffic_src = (None, None) if c4 else load_ncu_traffic(a.backbone, B, a.precision)
        # ---- cpu baseline (bounded sample, rank 0, N=1 only)
        cpu = None
        if world == 1 and not a.no_cpu_baseline and not c4:
            sb.unbind_process(numa)                                # the CPU baseline may use every host core again
            ips, _, cores = time_oracle(a.backbone, a.cpu_sample, 2, 1)
            cpu = {'value': ips, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                   'sample': f'{a.cpu_sample}-image batches x2 of the same workload, fp32 PyTorch oracle (oracle/), {cores} threads'}
        workload = (f'HMR forward with dataset-supplied camera (SPEC-SYN eval loop shape, trainer.py:235-245: int64 orig_shape, pre-computed R/K), '
                    f'{a.backbone} -> HMR head -> SMPL -> projection, 224x224, batch {B}/GPU, random weights') if c4 else \
                   f'SPEC full forward (CamCalib resnet50 -> (R,K) -> HMR {a.backbone} -> SMPL -> projection), 224x224, batch {B}/GPU, random weights'
        out = {
            'metric': METRIC if not c4 else 'images/sec HMR fwd with dataset cameras (224^2, b128)', 'value': value, 'unit': UNIT, 'n_gpus': world,
            'steps': a.steps, 'warmup': a.warmup,
            'ms_per_step': ms_per_step, 'step_ms_spread': step_spread, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': a.precision, 'data': 'synthetic',
            'config': {'workload': workload,
                       'backbone': a.backbone, 'batch_per_gpu': B, 'global_batch': B * world, 'cuda_graph': not a.no_graph and not c4,
                       'numa': {k: v for k, v in numa.items() if k != 'previous'},
                       'l2': f'inputs {B * 602112 / 1e6:.0f} MB/step/GPU > 126 MB L2, no explicit flush (weights stay L2-resident as in steady-state serving)',
                       'parallelism': f'dp{world} (batch shard + one all-gather of 85,176 B/image records)' if world > 1 else 'single GPU',
                       'gather': gather_desc},
            'clocks': clocks,
            'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h, 'ms_per_step': e2e_ms / e2e_steps,
                    'steps': e2e_steps, 'host_link': link,
                    'how': 'pinned host inputs -> H2D (double-buffered staging, graph captured on the staging buffers) -> forward -> D2H of the packed records; copies on side streams'},
            'gpu_launches': int(launches_per_step * a.steps),
            'roofline': {'bound': 'tensor', 'achieved': achieved, 'peak': peaks['tf_sustained'], 'unit': 'TFLOP/s',
                         'frac': achieved / peaks['tf_sustained'],
                         'traffic': traffic, 'traffic_source': traffic_src,
                         'algorithmic_bytes': conv_bytes,
                         'kernel': 'tcgen05 implicit-GEMM conv family (conv_tcp / conv_tcp2 cta_group::2 / conv_tc / conv3x3_halo / bottleneck / conv_stem7), %d conv ops/step' % n_conv,
                         'how': 'sum of conv FLOPs of the trunks / sum of per-launch CUDA-event times (specb200_trunk_profile, eager, same stream)',
                         'peak_source': peaks['source'] + ' bf16 sustained', 'conv_ms_per_step': conv_ms,
                         'conv_share_of_trunk_ops': conv_ms / step_ops_ms if step_ops_ms else None,
                         'step_frac_of_peak': conv_flops / (ms_per_step * 1e-3) / 1e12 / peaks['tf_sustained']},
            'cpu_baseline': cpu,
        }
        _emit(out)
    if world > 1:
        if e2e_gather is not None and hasattr(e2e_gather, 'close'):
            e2e_gather.close()
        dist.barrier()
        dist.destroy_process_group()
    return out


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, record, keys=None):
    """Writes the per-image arrays a caller of the timed path receives from its last step (``unpack_record`` of the packed
    records, every rank's rows after the all-gather) as ``out_dir/<name>.npy``, float32.  Above DUMP_LIMIT_BYTES in all, a
    fixed seeded sample of the images is written (same rows for the same arguments), so two builds can be compared."""
    import numpy as np
    import spec_b200 as sb
    n = record.shape[0]
    keep = max(1, min(n, DUMP_LIMIT_BYTES // (record.shape[1] * 4)))
    if keep < n:
        record = record[torch.from_numpy(np.sort(np.random.RandomState(0).choice(n, keep, replace=False)))]
    os.makedirs(out_dir, exist_ok=True)
    for k, v in sb.unpack_record(record).items():
        if keys is None or k in keys:
            np.save(os.path.join(out_dir, f'{k}.npy'), v.numpy().astype(np.float32))


_JSON_FD = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner on stdout when the
    first communicator is created), so everything that goes to fd 1 from here on is sent to stderr and the JSON line is
    written to the saved descriptor by ``_emit``."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def _emit(obj):
    line = (json.dumps(obj) + '\n').encode()
    if _JSON_FD is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_JSON_FD, line)


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--batch', type=int, default=0, help='images per GPU per step (default 256; 128 with --mode c4)')
    ap.add_argument('--mode', default='spec', choices=['spec', 'c4'], help="spec: CamCalib -> HMR (BASELINE configs 2,3,5); c4: HMR with dataset cameras (config 4)")
    ap.add_argument('--backbone', default='resnet50')
    ap.add_argument('--precision', default='bf16', choices=['bf16', 'fp16', 'fp32'])
    ap.add_argument('--chunk', type=int, default=int(os.environ.get('SPECB200_CHUNK', '0')))
    ap.add_argument('--no-graph', action='store_true')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--profile-range', action='store_true', help='only run the steps inside cudaProfilerStart/Stop (for ncu --profile-from-start off)')
    ap.add_argument('--cpu-sample', type=int, default=16, help='images per CPU-oracle step (bounded sample)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy (float32, at most 64 MB: a fixed sample of the images beyond that)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.dump_outputs and a.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of --impl ours')
    if a.warmup < 3:
        a.warmup = 3
    if a.impl == 'reference':
        run_reference(a)
    else:
        run_ours(a)


if __name__ == '__main__':
    main()
