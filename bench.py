#!/usr/bin/env python
"""bench.py — CPR head img/s @1333x800 (BASELINE.json metric) on N B200s + HBM roofline of the neighbor gather.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Step = one pass of the CPR head over one batch of synthetic FPN tensors: CPRHead.simple_test == forward (4x conv3x3+GN+
ReLU towers + class-logit map: hand-written tcgen05 implicit GEMM, fp32-accurate two-term fp16 split) + get_bboxes (fused bag
sampling / arg-max / nearest+classify filters / merge).
Workload = BASELINE.json configs[1]: CPR R50-FPN 1333x800 (pad 800x1344 -> 100x168x256 map at stride 8), 500 points per
image, 80 classes, radius 8 (K=289), batch 8 per GPU, fp32 (the reference runs fp32; no AMP in its CPR configs).
Image-parallel, weak scaling: every rank owns its own 8 images; no data-path collective (SURVEY.md §8e).

  value   img/s with inputs resident in HBM, timed with CUDA events over exactly K steps, max over ranks
  e2e     same call with HOST (pinned) inputs: H2D of the FPN tensor + GT boxes and D2H of the detections inside the region
  roofline        dominant kernel of the step = the tcgen05 conv3x3 (tensor bound): algorithmic FLOPs / CUDA-event time vs the
                  measured bf16 GEMM peak (MEASURED_PEAKS.json)
  roofline_gather neighbor-gather kernel (ptb_cpr_bag_gather, C=256 — the kernel BASELINE.json's target names), timed alone with
                  CUDA events in this process; algorithmic bytes per SURVEY.md §8d (166.5 MB/img); peak = MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the oracle port of the reference head (torch CPU ops, all host threads) on a bounded sample
--impl reference: the reference's own CPU implementation of the same step (oracle port: the reference is pure Python
and /root/reference does not exist on the GPU box) on all host cores: floor(cores/16) processes x 16 threads, one image each per step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

CFG = dict(B=8, pad_hw=(800, 1344), img_hw=(800, 1333), stride=8, n=500, radius=8, num_classes=80, C=256)
METRIC = 'cpr_head_refine_img_per_s_1333x800'


def head_cfg():
    r = CFG['radius']
    return dict(
        type='CPRHead', norm_cfg=dict(type='GN', num_groups=32, requires_grad=True), num_classes=CFG['num_classes'],
        in_channels=CFG['C'], feat_channels=CFG['C'], stacked_convs=4, num_cls_fcs=0, strides=[CFG['stride']],
        loss_mil=dict(type='MILLoss', binary_ins=False, loss_weight=0.25), loss_type=0,
        loss_cfg=dict(with_neg=True, neg_loss_weight=0.75, refine_bag_policy='only_refine_bag', random_remove_rate=0.4,
                      with_gt_loss=True, gt_loss_weight=0.125, with_mil_loss=True),
        normal_cfg=dict(prob_cls_type='sigmoid', out_bg_cls=False),
        train_pts_extractor=dict(pos_generator=dict(type='CirclePtFeatGenerator', radius=r),
                                 neg_generator=dict(type='OutCirclePtFeatGenerator', radius=r, class_wise=True)),
        refine_pts_extractor=dict(pos_generator=dict(type='CirclePtFeatGenerator', radius=r),
                                  neg_generator=dict(type='OutCirclePtFeatGenerator', radius=r, keep_wh=True, class_wise=True)),
        point_refiner=dict(merge_th=0.1, refine_th=0.1, classify_filter=True, nearest_filter=True),
        train_cfg=None, test_cfg=dict(nms_pre=1000, score_thr=0.05, nms=dict(type='nms', iou_threshold=0.5), max_per_img=100))


def synth_batch(B, seed):
    """synthetic FPN tensor + random point annotations on the HOST (seeded CPU generator)."""
    g = torch.Generator().manual_seed(seed)
    ph, pw = CFG['pad_hw']
    H, W = ph // CFG['stride'], pw // CFG['stride']
    x = torch.randn(B, CFG['C'], H, W, generator=g)
    gtb, gtl, aid, metas = [], [], [], []
    for b in range(B):
        pts = torch.rand(CFG['n'], 2, generator=g) * torch.tensor([float(pw), float(ph)])
        gtb.append(torch.cat([pts - 8, pts + 8], 1))
        gtl.append(torch.randint(0, CFG['num_classes'], (CFG['n'],), generator=g))
        aid.append(torch.arange(b * CFG['n'], (b + 1) * CFG['n']))
        metas.append(dict(pad_shape=(ph, pw, 3), img_shape=CFG['img_hw'] + (3,), scale_factor=[1.0, 1.0, 1.0, 1.0]))
    return x, gtb, gtl, aid, metas


def head_weights(seed=7):
    """random-init weights of the head under the reference's parameter names, "trained-like" scale on the classifiers so that the
    probabilities span (0, 1) (SURVEY.md §8d); the same dict feeds the GPU head and the CPU arm."""
    g = torch.Generator().manual_seed(seed)
    C, ncls = CFG['C'], CFG['num_classes']
    w = {}
    for i in range(4):
        w[f'cls_convs.{i}.conv.weight'] = torch.randn(C, C, 3, 3, generator=g) * (1.4 / (C * 9) ** 0.5)
        w[f'cls_convs.{i}.gn.weight'] = 1 + 0.1 * torch.randn(C, generator=g)
        w[f'cls_convs.{i}.gn.bias'] = 0.1 * torch.randn(C, generator=g)
    w['cls_out.weight'] = torch.randn(ncls, C, generator=g) * 0.01 * 8.0
    w['cls_out.bias'] = torch.full((ncls,), -float(np.log(99.0)))
    w['ins_out.weight'] = torch.randn(ncls, C, generator=g) * 0.01 * 8.0
    w['ins_out.bias'] = torch.zeros(ncls)
    return w


def synth_rpn_outputs(seed, B, size=(512, 640), A=3, strides=(4, 8, 16, 32, 64)):
    """RPN logits ~ N(-3, 1.5) and deltas ~ N(0, 0.3) for a (h, w) tile, one (B, A, H, W) / (B, 4A, H, W) pair per level."""
    g = torch.Generator().manual_seed(seed)
    cls, box = [], []
    for s in strides:
        H, W = -(-size[0] // s), -(-size[1] // s)
        cls.append(torch.randn(B, A, H, W, generator=g) * 1.5 - 3.0)
        box.append(torch.randn(B, 4 * A, H, W, generator=g) * 0.3)
    return cls, box, [(size[0] - 3 * (b % 4), size[1] - 5 * (b % 4), 3) for b in range(B)]


def synth_dense_anchors(seed, n_anchor=81840, n_gt=300, n_ign=5, size=(512, 640)):
    """dense-anchor-like boxes (4 sizes x 3 ratios at random centres), GT boxes, labels, ignore regions."""
    g = torch.Generator().manual_seed(seed)
    h, w = size
    wh_img = torch.tensor([w, h], dtype=torch.float32)
    c = torch.rand(n_anchor, 2, generator=g) * wh_img
    s = torch.tensor([8., 16., 32., 64.])[torch.randint(0, 4, (n_anchor,), generator=g)]
    r = torch.tensor([0.5, 1.0, 2.0])[torch.randint(0, 3, (n_anchor,), generator=g)]
    ws, hs = s * r.sqrt(), s / r.sqrt()
    anchors = torch.stack([c[:, 0] - ws / 2, c[:, 1] - hs / 2, c[:, 0] + ws / 2, c[:, 1] + hs / 2], 1)
    gc = torch.rand(n_gt, 2, generator=g) * wh_img
    gs = torch.rand(n_gt, 2, generator=g) * 60 + 4
    ic = torch.rand(n_ign, 2, generator=g) * wh_img
    return anchors, torch.cat([gc - gs / 2, gc + gs / 2], 1), torch.randint(0, 5, (n_gt,), generator=g), torch.cat([ic - 40, ic + 40], 1)


# --------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock / throttle (clocks-event) reasons sampled DURING the timed region (B200_PROFILING.md recipe).  NVML is polled from
    a thread of this process every 5 ms (the timed region of the default run lasts ~100 ms, shorter than nvidia-smi's start-up);
    when pynvml is missing the same fields are read from an `nvidia-smi -lms` child process instead."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
    NAMES = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []          # (timestamp, sm_mhz, max_mhz, power_w, set(reasons))
        self.nvml = None
        self._stop = threading.Event()
        self.source = None

    # ---- NVML thread
    def _nvml_loop(self):
        nv, h = self.nvml, self.handle
        bits = [(nv.nvmlClocksEventReasonHwSlowdown, 'hw_slowdown'), (nv.nvmlClocksEventReasonHwThermalSlowdown, 'hw_thermal_slowdown'),
                (nv.nvmlClocksEventReasonSwThermalSlowdown, 'sw_thermal_slowdown'), (nv.nvmlClocksEventReasonSwPowerCap, 'sw_power_cap')]
        try:
            mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        except Exception:
            mx = float('nan')
        while not self._stop.is_set():
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
                try:
                    pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                except Exception:
                    pw = float('nan')
                self.lines.append((time.perf_counter(), sm, mx, pw, {n for b, n in bits if mask & b}))
            except Exception:
                pass
            self._stop.wait(0.005)

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical devices: honour CUDA_VISIBLE_DEVICES when it is a plain index list
            vis = os.environ.get('CUDA_VISIBLE_DEVICES', '')
            phys = self.idx
            if vis and all(t.strip().isdigit() for t in vis.split(',')):
                ids = [int(t) for t in vis.split(',')]
                if self.idx < len(ids):
                    phys = ids[self.idx]
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
            self.source = 'nvml'
            self.t = threading.Thread(target=self._nvml_loop, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '100',
                                          '-i', str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = 'nvidia-smi'
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            f = [t.strip() for t in line.strip().split(',')]
            if len(f) < 8:
                continue
            try:
                self.lines.append((time.perf_counter(), float(f[1]), float(f[2]), float(f[3]),
                                   {n for n, v in zip(self.NAMES, f[4:8]) if v.lower().startswith('active')}))
            except ValueError:
                continue

    def stop(self, t0=None, t1=None):
        if self.nvml is None and self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['neither NVML nor nvidia-smi available'])
        self._stop.set()
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        else:
            self.t.join(timeout=1)
        inside = [r for r in self.lines if t0 is None or (t0 <= r[0] <= t1)]
        window = 'timed region'
        if not inside:          # region shorter than the sampling latency: use everything since the warm-up began
            inside, window = list(self.lines), 'warm-up + timed region'
        if not inside:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['no samples'], source=self.source)
        reasons = set()
        for r in inside:
            reasons |= r[4]
        pw = [r[3] for r in inside if r[3] == r[3]]
        return dict(sm_mhz=float(np.median([r[1] for r in inside])), sm_max_mhz=float(max(r[2] for r in inside)),
                    power_w_max=float(max(pw)) if pw else None, samples=len(inside), window=window, source=self.source,
                    reasons=sorted(reasons))


def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs, burst copy)'
    return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


def measured_tensor_peak():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d['bf16_tflops']), 'measured (MEASURED_PEAKS.json bf16_tflops, burst cuBLAS bf16 GEMM)'
    return 1590.0, 'fallback (B200_PROFILING.md 1.59 PFLOP/s bf16)'


# --------------------------------------------------------------------------------------------------------------------
def cpu_reference_step(x, gtb, gtl, aid, metas, weights, cfg):
    """the reference head's CPU path (oracle port): forward towers + get_bboxes for the given images."""
    from oracle import cpr as ocpr
    with torch.no_grad():
        feat = ocpr.tower_forward(x, weights, cfg)
        return ocpr.cpr_get_bboxes(feat, weights, gtb, gtl, aid, metas, cfg)


def oracle_cfg():
    from oracle import cpr as ocpr
    return ocpr.default_cfg(num_classes=CFG['num_classes'], in_channels=CFG['C'], feat_channels=CFG['C'], stride=CFG['stride'],
                            pos_radius=CFG['radius'], neg_radius=CFG['radius'])


WORKLOAD = ('BASELINE.json configs[1]: CPR R50-FPN 1333x800 (pad 800x1344 -> 100x168x256 FPN map, stride 8), 500 pts/img, r=8 (K=289), '
            '80 classes, bs=8 per GPU; step = CPRHead.simple_test (forward towers + get_bboxes)')


def bench_config(world):
    """the `config` object of the JSON line — IDENTICAL for both arms (the driver's same_config check); what differs per arm (how a
    step samples the workload) is stated in cpu_baseline.sample / extra."""
    return dict(workload=WORKLOAD, global_batch=CFG['B'] * world, parallelism=f'image-parallel x{world}, no data-path collective',
                l2='two rotating input sets, each 137.6 MB > 126 MB L2 (inputs larger than L2)',
                fpn_layout='channels_last (NHWC storage, as an FPN run with memory_format=torch.channels_last emits it); an NCHW-contiguous '
                           'FPN output costs one extra transpose per step, reported as extra.nchw_to_nhwc_ms',
                towers='tcgen05 implicit-GEMM conv3x3 (fp16 two-term split = fp32-level accuracy) + GN + ReLU (libptb_b200.so); point '
                       'path = libptb_b200.so; no cuDNN/cuBLAS in the step')


def _cpu_worker(idx, threads, steps, warm, seed, start_evt, q):
    """one process of the CPU arm: the oracle port of the reference head on its own image, `threads` ATen threads."""
    torch.set_num_threads(threads)
    weights, cfg = head_weights(), oracle_cfg()
    x, gtb, gtl, aid, metas = synth_batch(1, seed + idx)
    for _ in range(warm):
        cpu_reference_step(x, gtb, gtl, aid, metas, weights, cfg)
    q.put(('ready', idx, 0.0))
    start_evt.wait()
    t0 = time.perf_counter()
    for _ in range(steps):
        cpu_reference_step(x, gtb, gtl, aid, metas, weights, cfg)
    q.put(('done', idx, time.perf_counter() - t0))


def cpu_arm(steps, warm=1, seed=100):
    """the reference head's CPU path at its best on this host: floor(cores / 16) processes x 16 ATen threads (the reference's many small
    ops stop scaling beyond ~16 threads), every process refining its own image; one "step" = all processes finish one image.
    returns (img/s over the whole host, seconds per step, processes, threads per process)."""
    import multiprocessing as mp
    ncpu = os.cpu_count() or 1
    threads = min(16, ncpu)
    procs = max(1, ncpu // 16)
    ctx = mp.get_context('spawn')
    q, start_evt = ctx.Queue(), ctx.Event()
    ps = [ctx.Process(target=_cpu_worker, args=(i, threads, steps, warm, seed, start_evt, q), daemon=True) for i in range(procs)]
    for p_ in ps:
        p_.start()
    try:
        for _ in range(procs):
            tag, _, _ = q.get(timeout=1800)
            assert tag == 'ready'
        t0 = time.perf_counter()
        start_evt.set()
        for _ in range(procs):
            tag, _, _ = q.get(timeout=3600)
            assert tag == 'done'
        wall = time.perf_counter() - t0
    finally:
        for p_ in ps:
            p_.join(timeout=30)
            if p_.is_alive():
                p_.terminate()
    return procs * steps / wall, wall / steps, procs, threads


def run_reference(args, rank):
    if rank != 0:
        return
    v, s_per_step, procs, threads = cpu_arm(args.steps, warm=max(args.warmup, 1))
    line = dict(metric=METRIC, value=v, unit='img/s', n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * s_per_step, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='fp32',
                data='synthetic', impl='reference', config=bench_config(args.gpus),
                cpu_baseline=dict(value=v, unit='img/s', cores=procs * threads, host_cores=os.cpu_count(), kind='port',
                                  sample=f'{args.steps} steps; a step = {procs} processes x {threads} threads each refining ONE image of the '
                                         f'workload concurrently (bounded sample of the 8-image batch); oracle port of the reference head '
                                         f'(forward towers + get_bboxes, torch CPU fp32)'),
                e2e=dict(value=v, unit='img/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------------------------------
T_MAIN = 0.0      # perf_counter at the start of main(): extra.wall_s_cumulative says where the bench's own wall-clock goes


class _SkipP2PTrain(Exception):      # control flow only: a side measurement that is switched off for this run
    pass


def main():
    global T_MAIN
    T_MAIN = time.perf_counter()
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extra', action='store_true')
    ap.add_argument('--p2p-train', action='store_true', help='also time a P2PHead training step (its two narrow output convs run on cuDNN under '
                    'autograd: the first cuDNN use pages the library in, minutes on a cold box)')
    ap.add_argument('--profile', action='store_true', help='for runs under ncu: no load-holding steps, no e2e, no extras')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the detections of the last timed step (rank 0) to DIR/*.npy, so that two '
                    'builds can be compared output for output on the same seeded inputs')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    args.warmup = max(args.warmup, 3) if args.impl == 'ours' else args.warmup
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    if args.impl == 'reference':
        return run_reference(args, rank)

    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit('bench.py --impl ours needs a CUDA device (there is no CPU fallback)')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    torch.backends.cudnn.allow_tf32 = False          # parity mode: 1e-4 logits need fp32 towers
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.benchmark = True

    from pointtinybenchmark_b200 import cpr_head, ops  # noqa: F401
    from pointtinybenchmark_b200.registry import build_head
    head = build_head(head_cfg()).to(dev).eval()
    sd = head.state_dict()
    sd.update(head_weights())
    head.load_state_dict(sd)

    B = CFG['B']
    # two rotating input sets (2 x 137.6 MB > 126 MB L2) so no step finds its input in L2
    host = []
    for i in range(2):
        x, gtb, gtl, aid, metas = synth_batch(B, 1234 + rank * 10 + i)
        host.append((x.pin_memory(), gtb, gtl, aid, metas))
    devs = []
    for x, gtb, gtl, aid, metas in host:
        devs.append((x.to(dev).contiguous(memory_format=torch.channels_last), [t.to(dev) for t in gtb], [t.to(dev) for t in gtl],
                     [t.to(dev) for t in aid], metas))

    def step_resident(i):
        x, gtb, gtl, aid, metas = devs[i % 2]
        with torch.no_grad():
            return head.simple_test((x,), metas, gt_bboxes=gtb, gt_labels=gtl, gt_anns_id=aid)

    gt_host_packed = []
    for x, gtb, gtl, aid, metas in host:
        gt_host_packed.append((torch.cat(gtb).pin_memory(), torch.cat(gtl).pin_memory(), torch.cat(aid).pin_memory()))

    # ---- end-to-end: host (pinned) inputs -> H2D -> CPRHead.simple_test -> D2H of the detections, every step inside the
    # timed region.  Double-buffered like a pin_memory dataloader: the H2D of step i+1 runs on a copy stream while step i
    # computes; the host blocks on step i-1's result while step i is in flight.
    copy_stream = torch.cuda.Stream()
    n_pts = CFG['n']
    dev_in = [dict(x=torch.empty_like(devs[0][0]), b=torch.empty((B * n_pts, 4), device=dev),
                   l=torch.empty((B * n_pts,), dtype=torch.long, device=dev), a=torch.empty((B * n_pts,), dtype=torch.long, device=dev),
                   ready=torch.cuda.Event(), free=torch.cuda.Event()) for _ in range(2)]
    host_out = [torch.empty((B * n_pts, 6), pin_memory=True) for _ in range(2)]
    host_x_cl = [h[0].contiguous(memory_format=torch.channels_last).pin_memory() for h in host]   # host layout = device layout

    def upload(i):
        slot = dev_in[i % 2]
        pb, pl, pa = gt_host_packed[i % 2]
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(slot['free'])            # the step that last used this slot has finished
            slot['x'].copy_(host_x_cl[i % 2], non_blocking=True)
            slot['b'].copy_(pb, non_blocking=True); slot['l'].copy_(pl, non_blocking=True); slot['a'].copy_(pa, non_blocking=True)
            slot['ready'].record(copy_stream)
        return slot

    def run_e2e(steps):
        cur_stream = torch.cuda.current_stream()
        done = [torch.cuda.Event(), torch.cuda.Event()]
        for sl in dev_in:
            sl['free'].record(cur_stream)
        nxt = upload(0)
        for i in range(steps):
            slot = nxt
            cur_stream.wait_event(slot['ready'])
            if i + 1 < steps:
                nxt = upload(i + 1)
            metas = host[i % 2][4]
            with torch.no_grad():
                res = head.simple_test((slot['x'],), metas, gt_bboxes=list(slot['b'].split(n_pts)), gt_labels=list(slot['l'].split(n_pts)),
                                       gt_anns_id=list(slot['a'].split(n_pts)))
            if i >= 2:
                done[i % 2].synchronize()                   # host_out[i % 2] of step i-2 has landed before it is overwritten
            host_out[i % 2].copy_(torch.cat([r[0] for r in res]), non_blocking=True)
            slot['free'].record(cur_stream)
            done[i % 2].record(cur_stream)
            if i >= 1:
                done[(i - 1) % 2].synchronize()             # the user consumes step i-1's detections here
        done[(steps - 1) % 2].synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ops.launch_count()
        e0.record()
        for i in range(steps):
            out = fn(i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        launches = ops.launch_count() - l0
        barrier()
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), launches, out

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for i in range(args.warmup):
        step_resident(i)
    for i in range(0 if args.profile else 20):   # keep the GPU under load while nvidia-smi starts sampling (untimed)
        step_resident(i)
    wall = {'setup': time.perf_counter() - T_MAIN}
    t_begin = time.perf_counter()
    ms, launches, last_out = timed(step_resident, args.steps)
    wall['timed_steps'] = time.perf_counter() - T_MAIN
    t_end = time.perf_counter()
    clocks = sampler.stop(t_begin, t_end) if rank == 0 else None
    value = world * B * args.steps / (ms / 1e3)
    if args.dump_outputs and rank == 0:
        # what CPRHead.simple_test hands its caller, per image: dets (n, 6) = [x1, y1, x2, y2, score, ann_id] and labels (n,);
        # every image has CFG['n'] points, so the images stack.  96 KB in all at the default workload.
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, 'dets.npy'), torch.stack([d for d, _ in last_out]).cpu().numpy().astype(np.float32))
        np.save(os.path.join(args.dump_outputs, 'labels.npy'), torch.stack([l for _, l in last_out]).cpu().numpy().astype(np.float64))

    if args.profile:
        if rank == 0:
            print(json.dumps(dict(profile_run=True, ms_per_step=ms / args.steps, note='number taken under a profiler: not a bench value')))
        return
    run_e2e(2)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run_e2e(args.steps)
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_e2e = float(t[0])
    e2e_value = world * B * args.steps / (ms_e2e / 1e3)
    h2d = host[0][0].numel() * 4 + sum(t.numel() * t.element_size() for t in gt_host_packed[0])
    d2h = B * CFG['n'] * 6 * 4
    assert host_out[0].abs().sum() > 0

    wall['e2e'] = time.perf_counter() - T_MAIN
    # ---- roofline of the neighbor-gather kernel + per-kernel breakdown (rank 0, kernels timed alone)
    roofline, roofline_gather, extra = None, None, {}
    if rank == 0:
        peak, peak_src = measured_peaks()
        x, gtb, gtl, aid, metas = devs[0]
        from pointtinybenchmark_b200.cpr_head import _BatchGT
        gt = _BatchGT(gtb, gtl, metas, dev)
        off = head._offsets(head.refine_pts_extractor['pos_generator'], dev)
        K = off.shape[0]
        with torch.no_grad():
            feat = head((x,))[0][0]
        fmap = ops.to_nhwc(feat)
        Bq, H, W, C = fmap.shape
        G = gt.G
        flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)

        def ktime(fn, n=20):
            for _ in range(3):
                fn()
            ts = []
            for _ in range(n):
                flush.add_(1.0)                       # flush L2 (256 MB write) between timed launches
                s, e = torch.cuda.Event(True), torch.cuda.Event(True)
                s.record(); fn(); e.record(); torch.cuda.synchronize()
                ts.append(s.elapsed_time(e))
            return float(np.mean(ts))

        alg = Bq * H * W * C * 4 + G * K * 8 + G * K * C * 4 + G * K       # SURVEY.md §8d: 166.5 MB/img x 8
        t_g = ktime(lambda: ops.bag_gather(fmap, gt.centers, gt.bag_img, off, CFG['stride'], gt.pad_hw))
        ach = alg / (t_g * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, 'profiles', 'r01_gather_traffic.json')
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get('dram_bytes_per_launch')
        roofline_gather = dict(kernel='ptb_cpr_bag_gather<C=256> (neighbor gather, reference data flow)', bound='hbm', achieved=ach,
                        peak=peak, unit='GB/s', frac=ach / peak, traffic=traffic, peak_source=peak_src,
                        algorithmic_bytes_per_launch=alg, ms_per_launch=t_g, units_per_launch=f'{Bq} images x {CFG["n"]} bags x {K} samples',
                        timing='CUDA events on the launching stream, kernel alone, L2 flushed between launches')
        # dominant kernel of the step (~70 % of the device time, profiles/r01_step_launches_v*.json): the tcgen05 conv
        conv_traffic = None
        ctp = os.path.join(ROOT, 'profiles', 'r01_conv_traffic.json')
        if os.path.exists(ctp):
            conv_traffic = json.load(open(ctp)).get('dram_bytes_per_launch')       # DRAM bytes per launch from the ncu --set full capture
        from pointtinybenchmark_b200.layers import _packed_weight, _packed_weight_f16
        flops = 2.0 * 9 * C * 256 * Bq * H * W                                   # algorithmic (fp32 semantics), 158.5 GFLOP
        tpeak, tsrc = measured_tensor_peak()
        xin = ops.to_nhwc(x).contiguous()
        if head.last_tower_backend == 'tcgen05-f16x2':
            h16, l16, dinv = ops.split_f16(xin, auto_scale=True)
            wh, wl, invw = _packed_weight_f16(head.cls_convs[0])
            t_c = ktime(lambda: ops.conv3x3_c256_f16(h16, l16, wh, wl, invw, dinv))
            kname, mma_peak, mma_kind = 'ptb::conv_tc_kernel<3,true> (CTA-pair tcgen05.mma.cta_group::2, fp16 two-term split, kind::f16)', tpeak, 'fp16'
        else:
            xh, xl = ops.split_tf32(xin)
            wh, wl = _packed_weight(head.cls_convs[0])
            t_c = ktime(lambda: ops.conv3x3_c256(xh, xl, wh, wl))
            kname, mma_peak, mma_kind = 'ptb::conv_tc_kernel<1,false> (3xTF32, kind::tf32)', tpeak / 2, 'tf32'
        ach_t = flops / (t_c * 1e-3) / 1e12
        roofline = dict(kernel=kname + ': conv3x3 256->256 of the head towers, 4 launches per step', bound='tensor',
                        achieved=ach_t, peak=tpeak, unit='TFLOP/s', frac=ach_t / tpeak, traffic=conv_traffic, peak_source=tsrc,
                        algorithmic_flops_per_launch=flops, ms_per_launch=t_c,
                        note='achieved = algorithmic fp32 conv FLOPs / CUDA-event time.  For fp32-level accuracy the kernel issues 3 '
                             'tensor-core products per algorithmic one (h*h + l*h + h*l), so the tensor pipe runs at mma_tflops; '
                             'mma_frac = mma_tflops / the measured peak for that operand type (tf32 = half the bf16 figure)',
                        mma_tflops=3 * ach_t, mma_operand_type=mma_kind, mma_frac=3 * ach_t / mma_peak,
                        timing='CUDA events on the launching stream, kernel alone, L2 flushed between launches')
        if not args.no_extra:
            with torch.no_grad():
                N = CFG['num_classes']
                groups = ops.label_groups(gt.bag_img, gt.labels, N)
                rc = ops._refine_cfg(0.1, 0.5, 0.1, True, True, False)
                lmap = ops.linear_rows(fmap.reshape(-1, C), head.cls_out.weight, head.cls_out.bias).view(Bq, H, W, N)
                t_lin = ktime(lambda: ops.linear_rows(fmap.reshape(-1, C), head.cls_out.weight, head.cls_out.bias))
                t_ref = ktime(lambda: ops.refine_fused(lmap, N, gt.centers, gt.labels, gt.bag_img, off, CFG['stride'], gt.pad_hw,
                                                       gt.img_hw, groups, rc))
                t_tow = ktime(lambda: head((x,)), n=5)
                t_g80 = ktime(lambda: ops.bag_gather(lmap, gt.centers, gt.bag_img, off, CFG['stride'], gt.pad_hw, pts=False, valid=False))
                t_neg = ktime(lambda: ops.neg_mask(Bq, H, W, CFG['stride'], gt.pad_hw, gt.centers, gt.labels, gt.img_ptr,
                                                   CFG['stride'] * CFG['radius'], N, True))
                x_nchw = x.contiguous()             # what an FPN in torch's default memory format emits
                t_tr = ktime(lambda: x_nchw.contiguous(memory_format=torch.channels_last))
                del x_nchw
            extra['nchw_to_nhwc_ms'] = t_tr       # NOT inside the timed step: the step takes the FPN tensor channels_last (config.fpn_layout)
            step_ms = ms / args.steps
            extra['kernels_ms_per_batch'] = dict(
                towers_tcgen05=t_tow, linear_rows_256x80=t_lin, refine_fused=t_ref, bag_gather_c256=t_g, bag_gather_c80=t_g80,
                neg_mask=t_neg)
            extra['share_of_step'] = dict(towers_tcgen05=t_tow / step_ms, linear_rows=t_lin / step_ms, refine_fused=t_ref / step_ms)
            extra['tower_backend'] = head.last_tower_backend
            extra['towers_effective_fp32_tflops'] = 4 * 2 * 9 * C * C * Bq * H * W / (t_tow * 1e-3) / 1e12
            extra['linear_rows_tflops'] = 2 * Bq * H * W * C * N / (t_lin * 1e-3) / 1e12
            # P2P post-processing at BASELINE.json configs[2] shape (16 x 16800 proposals, nms_pre 1000, iou 0.01): decode + top-k + NMS
            try:
                if world > 1:                 # side measurements are reported by the 1-GPU run only
                    raise _SkipP2PTrain()
                g2 = torch.Generator().manual_seed(5)
                Bp = 16
                cls_map = (torch.randn(Bp, H, W, N, generator=g2) * 1.5 - 3.0).to(dev)
                reg_map = torch.randn(Bp, H, W, 2, generator=g2).to(dev)
                ihw = torch.tensor([[800, 1333]] * Bp, dtype=torch.int32, device=dev)
                anc = torch.zeros(1, 2, device=dev)

                def p2p_post():
                    idx, pts, sc = ops.p2p_decode_topk(cls_map, reg_map, N, 1, anc, CFG['stride'], 1.0, ihw, 1000)
                    return ops.multiclass_nms(pts, sc, (32, 32), 0.05, 0.01, 100)
                t_p2p = ktime(p2p_post, n=10)
                extra['p2p_postproc'] = dict(ms_per_batch16=t_p2p, img_per_s=Bp / (t_p2p * 1e-3),
                                             what='ptb_p2p_decode_topk + ptb_multiclass_nms, 16 x (100x168x80 logits), nms_pre 1000, '
                                                  'score_thr 0.05, iou 0.01, max 100 (reference CPU: ~10 s/img, SURVEY.md §6)')
            except _SkipP2PTrain:
                pass
            except Exception as ex:  # pragma: no cover
                extra['p2p_postproc_error'] = repr(ex)[:200]
            # P2P training assignment at configs[2] shape: cost matrix + HungarianAssignerV2 (topk_k 5) for 16 images x 16 800 proposals,
            # 100 GTs each, on the GPU; beside it the reference route (cost.cpu() + 5 scipy solves per image) on ONE image (bounded sample)
            try:
                if world > 1:                 # side measurements are reported by the 1-GPU run only
                    raise _SkipP2PTrain()
                import time as _time
                from scipy.optimize import linear_sum_assignment as _lsa
                g3 = torch.Generator().manual_seed(9)
                Bh, Qh, nh = 16, H * W, 100
                clsh = (torch.randn(Bh, Qh, N, generator=g3) * 1.5 - 3.0).to(dev)
                xs = (torch.arange(Qh) % W).float() * CFG['stride']
                ys = (torch.arange(Qh) // W).float() * CFG['stride']
                prop = (torch.stack([xs, ys], 1)[None] + torch.randn(Bh, Qh, 2, generator=g3) * 4).to(dev).contiguous()
                gts_h = (torch.rand(Bh, nh, 2, generator=g3) * torch.tensor([1333., 800.])).to(dev)
                gl_h = torch.randint(0, N, (Bh, nh), generator=g3).int().to(dev)
                cost_flat = torch.empty(Bh * Qh * nh, device=dev)
                gi_out = torch.zeros(Bh * Qh, dtype=torch.int64, device=dev)
                shapes_h = [(Qh, nh)] * Bh

                def p2p_assign():
                    for b in range(Bh):
                        ops.p2p_cost_matrix(clsh[b], prop[b], None, gts_h[b], gl_h[b], 2.0, 0.25, 2.0, 1e-12, 0.1, 1333.0, 800.0,
                                            out=cost_flat[b * Qh * nh:(b + 1) * Qh * nh])
                    gi_out.zero_()
                    return ops.hungarian_v2_batch(cost_flat, shapes_h, 5, gi_out, [b * Qh for b in range(Bh)])
                t_as = ktime(p2p_assign, n=5)
                st_h = p2p_assign().cpu()
                c0 = cost_flat[:Qh * nh].view(Qh, nh)
                t0 = _time.perf_counter()
                c_host = c0.cpu().numpy()
                free = np.ones(Qh, bool)
                ref_gi = np.zeros(Qh, np.int64)
                for _ in range(5):
                    idx = np.nonzero(free)[0]
                    r_, c_ = _lsa(c_host[free])
                    ref_gi[idx[r_]] = c_ + 1
                    free[idx[r_]] = False
                t_sc = (_time.perf_counter() - t0) * 1e3
                same = bool(np.array_equal(ref_gi, gi_out[:Qh].cpu().numpy()))
                extra['p2p_hungarian'] = dict(ms_per_batch16=t_as, img_per_s=Bh / (t_as * 1e-3), status_ok=bool(int(st_h.max()) == 0),
                                              scipy_ms_per_image=t_sc, scipy_ms_per_batch16_extrapolated=t_sc * Bh,
                                              identical_to_scipy_on_sample=same,
                                              what='ptb_p2p_cost_matrix + ptb_hungarian_v2_batch (topk_k 5), 16 x (16800 proposals x 100 GTs); '
                                                   'scipy = cost.cpu() + 5 linear_sum_assignment solves of image 0 (reference route, hungarian_assigner.py:229-268)')
                del clsh, cost_flat, gi_out
            except _SkipP2PTrain:
                pass
            except Exception as ex:  # pragma: no cover
                extra['p2p_hungarian_error'] = repr(ex)[:300]
            # BASELINE.json configs[3] pieces (640x512 tile, 5 levels, 3 anchors per cell = 81 840 anchors): RPN proposal generation and
            # MaxIoUAssigner for a batch of 16 tiles, beside the oracle port of the reference on the host (bounded sample: 2 tiles / 1 tile)
            try:
                if world > 1:                 # side measurements are reported by the 1-GPU run only
                    raise _SkipP2PTrain()
                import time as _time
                from oracle import anchors as _oa          # CPU leg only (the oracle port timed on the host)
                from pointtinybenchmark_b200.rpn import AnchorGenerator as _AG
                cls4, box4, shp4 = synth_rpn_outputs(21, 16)
                c4 = dict(scales=[2], ratios=[0.5, 1.0, 2.0], strides=[4, 8, 16, 32, 64], means=(0., 0., 0., 0.), stds=(1., 1., 1., 1.),
                          nms_pre=1000, max_per_img=1000, iou_threshold=0.7, min_bbox_size=0)    # faster_rcnn_r50_fpn_1x_TinyPerson640.py:25-40,106-112
                ag4 = _AG(scales=c4['scales'], ratios=c4['ratios'], strides=c4['strides'])
                cls4d, box4d = [t.to(dev) for t in cls4], [t.to(dev) for t in box4]
                base4 = torch.stack(ag4.base_anchors).to(dev)
                ihw4 = torch.tensor([[sh[0], sh[1]] for sh in shp4], dtype=torch.int32, device=dev)

                def rpn_run():
                    return ops.rpn_proposals(cls4d, box4d, base4, ag4.strides, ihw4, c4['means'], c4['stds'], 16 / 1000, 1000, 0, 0.7, 1000)
                t_rpn = ktime(rpn_run, n=10)
                t0 = _time.perf_counter()
                _oa.rpn_proposals([t[:2] for t in cls4], [t[:2] for t in box4], shp4[:2], dict(c4))
                t_rpn_cpu = (_time.perf_counter() - t0) * 1e3 / 2
                a4, g4, l4, i4 = synth_dense_anchors(11)
                a4d, g4d, l4d, i4d = a4.to(dev), g4.to(dev), l4.to(dev), i4.to(dev)
                kw4 = dict(pos_iou_thr=0.7, neg_iou_thr=0.3, min_pos_iou=0.3, match_low_quality=True, ignore_iof_thr=0.5)
                t_mi = ktime(lambda: ops.max_iou_assign(a4d, g4d, l4d, i4d, **kw4), n=10)
                t0 = _time.perf_counter()
                _oa.max_iou_assign(a4, g4, l4, i4, **kw4)
                t_mi_cpu = (_time.perf_counter() - t0) * 1e3
                extra['config4_dense_anchor'] = dict(
                    rpn_proposals_ms_per_batch16=t_rpn, rpn_tiles_per_s=16 / (t_rpn * 1e-3), rpn_cpu_oracle_ms_per_tile=t_rpn_cpu,
                    max_iou_assign_ms_per_tile=t_mi, max_iou_assign_cpu_oracle_ms_per_tile=t_mi_cpu,
                    what='ptb_rpn_proposals: 16 tiles x 81 840 anchors, nms_pre 1000/level, iou 0.7, max 1000; ptb_max_iou_assign: 81 840 anchors x '
                         '300 GTs + 5 ignore boxes; CPU = oracle port of the reference (torch CPU), single tile')
                del cls4d, box4d
            except _SkipP2PTrain:
                pass
            except Exception as ex:  # pragma: no cover
                extra['config4_dense_anchor_error'] = repr(ex)[:300]
            # P2PHead inference at BASELINE.json configs[2] shape (bs 16): two tcgen05 towers + output convs + decode/top-k/NMS
            try:
                if world > 1:                 # side measurements are reported by the 1-GPU run only
                    raise _SkipP2PTrain()
                from pointtinybenchmark_b200 import p2p_head as _p2p  # noqa: F401
                pcfg = dict(type='P2PHead', norm_cfg=dict(type='GN', num_groups=32, requires_grad=True), num_classes=N, in_channels=C,
                            feat_channels=C, stacked_convs=4, strides=[CFG['stride']], point_anchor=[(0., 0.)],
                            loss_cls=dict(type='FocalLoss', use_sigmoid=True, gamma=2.0, alpha=0.25, loss_weight=1.0),
                            loss_reg=dict(type='SmoothL1Loss', beta=1.0 / 9.0, loss_weight=0.5), pts_gamma=1, reg_norm=1,
                            train_cfg=None, test_cfg=dict(nms_pre=1000, min_bbox_size=0, score_thr=0.05, pseudo_wh=(32, 32),
                                                          nms=dict(type='nms', iou_threshold=0.01), max_per_img=100))
                ph = build_head(pcfg).to(dev).eval()
                xp = torch.randn(16, C, H, W, generator=torch.Generator().manual_seed(11)).to(dev).contiguous(memory_format=torch.channels_last)
                mp = [dict(pad_shape=CFG['pad_hw'] + (3,), img_shape=CFG['img_hw'] + (3,), scale_factor=[1.0, 1.0, 1.0, 1.0])] * 16
                with torch.no_grad():
                    t_ph = ktime(lambda: ph.simple_test((xp,), mp), n=5)
                extra['p2p_head_infer'] = dict(ms_per_batch16=t_ph, img_per_s=16 / (t_ph * 1e-3),
                                               what='P2PHead.simple_test, 16 x (256x100x168), random-init weights')
                del ph
                # P2PHead training step at the same shape: forward (two tensor-core towers) + cost matrix + GPU Hungarian matching
                # (topk_k 5) + focal / smooth-L1 losses + backward; 20 GT points per image
                if not args.p2p_train:
                    raise _SkipP2PTrain()
                pcfg_t = dict(pcfg, train_cfg=dict(neg_weight=1.0, assigner=dict(
                    type='HungarianAssignerV2', cls_costs=dict(type='FocalLossCost', weight=2.0),
                    reg_costs=dict(type='DisCostV2', weight=0.1, norm_with_img_wh=False), topk_k=5), sampler=dict(type='PseudoSampler')))
                pht = build_head(pcfg_t).to(dev).train()
                g4 = torch.Generator().manual_seed(13)
                gtb_p = []
                for _ in range(16):
                    cxy = torch.rand(20, 2, generator=g4) * torch.tensor([1300., 780.]) + 10
                    gtb_p.append(torch.cat([cxy - 8, cxy + 8], 1).to(dev))
                gtl_p = [torch.randint(0, N, (20,), generator=g4).to(dev) for _ in range(16)]
                xpt = xp.clone().requires_grad_(True)

                def p2p_train():
                    pht.zero_grad(set_to_none=True)
                    ls = pht.forward_train((xpt,), mp, gtb_p, gtl_p)
                    (sum(ls['loss_cls']) + sum(ls['loss_pts'])).backward()
                t_pt = ktime(p2p_train, n=3)
                extra['p2p_head_train'] = dict(ms_per_batch16=t_pt, img_per_s=16 / (t_pt * 1e-3),
                                               what='P2PHead.forward_train + backward, 16 x (256x100x168), 20 GTs per image, HungarianAssignerV2 '
                                                    'topk_k 5 on the GPU (no host round trip)')
                del pht, xp, xpt
            except _SkipP2PTrain:
                pass
            except Exception as ex:  # pragma: no cover
                extra['p2p_head_infer_error'] = repr(ex)[:200]

    wall['rooflines_and_extras'] = time.perf_counter() - T_MAIN
    # ---- training step of the head on EVERY rank (forward + loss + backward, image-parallel) with the path's only collective:
    #      one flat-bucket gradient all-reduce over NCCL (pointtinybenchmark_b200/dist.py).  Whole-job img/s, max over ranks.
    try:
        from pointtinybenchmark_b200.dist import GradBucket
        x_t, gtb_t, gtl_t, _, metas_t = devs[0]
        xg = x_t.clone().requires_grad_(True)
        head.train()
        # gradients live in one persistent flat buffer; per-bucket NCCL all-reduces (mean) are launched from post-accumulate hooks on a
        # side stream as soon as a bucket's last gradient kernel is queued: they run under the rest of backward
        bucket = GradBucket(head, overlap=os.environ.get('PTB_GRAD_OVERLAP', '0') == '1')
        # the reference trains the head with SGD (momentum 0.9, weight decay 1e-4: configs/_base_/schedules/schedule_1x.py:2); the step is
        # inside the timed region (multi-tensor kernels over the parameter list; the tower weights are re-packed for the tensor cores next
        # step, like after any real update); lr is tiny so that the synthetic batch cannot blow the weights up over the bench's few steps
        opt = torch.optim.SGD(head.parameters(), lr=1e-7, momentum=0.9, weight_decay=1e-4, foreach=True)

        def train_step():
            bucket.zero()
            xg.grad = None
            cf, inf = head((xg,))
            losses = head.loss(cf, inf, gtb_t, gtl_t, metas_t)
            sum(v for k, v in losses.items() if 'loss' in k).backward()
            nb_ = bucket.wait()
            opt.step()
            return nb_
        for _ in range(2):
            train_step()
        barrier()
        s_ev, e_ev = torch.cuda.Event(True), torch.cuda.Event(True)
        s_ev.record()
        for _ in range(5):
            nb = train_step()
        e_ev.record(); torch.cuda.synchronize()
        tt = torch.tensor([s_ev.elapsed_time(e_ev)], device=dev)
        # the collective alone: one all-reduce of the whole flat buffer, timed on its own (what an un-overlapped exchange would add)
        t_ar = 0.0
        if world > 1:
            for _ in range(3):
                dist.all_reduce(bucket.flat, op=dist.ReduceOp.AVG)
            barrier()
            a0, a1 = torch.cuda.Event(True), torch.cuda.Event(True)
            a0.record()
            for _ in range(10):
                dist.all_reduce(bucket.flat, op=dist.ReduceOp.AVG)
            a1.record(); torch.cuda.synchronize()
            t_ar = a0.elapsed_time(a1) / 10
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        if rank == 0:
            extra['train_step_img_per_s'] = world * B * 5 / (float(tt[0]) * 1e-3)
            extra['train_step_ms_per_batch'] = float(tt[0]) / 5
            extra['train_tower_backend'] = head.last_tower_backend
            extra['train_step_contents'] = 'forward (towers + loss) + backward + gradient all-reduce (N > 1) + SGD(momentum) step'
            extra['train_grad_allreduce'] = dict(bytes_per_rank=int(nb), backend='nccl' if world > 1 else None, buckets=len(bucket.ranges),
                                                 allreduce_alone_ms=t_ar,
                                                 overlap_hooks=bucket.overlap,
                                                 what='gradients are views of one persistent flat fp32 buffer (no copy-in / copy-out, mean = NCCL AVG): '
                                                      'ONE all-reduce of the 9.6 MB after backward (allreduce_alone_ms, timed on its own). '
                                                      'PTB_GRAD_OVERLAP=1 selects per-bucket all-reduces from post-accumulate hooks on a side stream; '
                                                      'measured on 2 x B200 it is slower (9.30 vs ~8.7 ms per step): the exchange takes 0.05 ms, the '
                                                      'hooks cost more host time than that in a backward pass that is partly launch-bound')
        bucket.close()
        del opt
        head.zero_grad(set_to_none=True)
        sd_ = head.state_dict(); sd_.update(head_weights()); head.load_state_dict(sd_)      # undo the (tiny) updates
        head.eval()
    except Exception as ex:  # pragma: no cover
        if rank == 0:
            extra['train_step_error'] = repr(ex)[:200]
        barrier()

    wall['train_step'] = time.perf_counter() - T_MAIN
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, s_per_step, procs, threads = cpu_arm(3, warm=1)
        cpu_baseline = dict(value=v, unit='img/s', cores=procs * threads, host_cores=os.cpu_count(), kind='port',
                            sample=f'3 timed steps (+1 warm-up); a step = {procs} processes x {threads} threads each refining ONE image of '
                                   f'the workload concurrently; oracle port of the reference head (forward + get_bboxes), torch CPU fp32')
    if rank == 0:
        wall['cpu_baseline'] = time.perf_counter() - T_MAIN
        extra['wall_s_cumulative'] = {k: round(v, 2) for k, v in wall.items()}     # host seconds since main() started, at the end of each phase
        line = dict(metric=METRIC, value=value, unit='img/s', n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=ms / args.steps, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='fp32',
                    data='synthetic',
                    config=bench_config(world),
                    clocks=clocks,
                    e2e=dict(value=e2e_value, unit='img/s', h2d_bytes_per_step=int(h2d), d2h_bytes_per_step=int(d2h),
                             ms_per_step=ms_e2e / args.steps,
                             h2d_gb_per_s_per_gpu=h2d / (ms_e2e / args.steps * 1e-3) / 1e9,
                             bound='host->device link: the fp32 FPN tensor (137.6 MB per step and GPU) moves at the rate shown, the PCIe Gen5 x16 practical ceiling is ~55 GB/s',
                             pipeline='pinned host buffers; H2D of step i+1 on a copy stream overlaps step i; D2H of every step inside the region'),
                    gpu_launches=int(launches * world), roofline=roofline, roofline_gather=roofline_gather,
                    cpu_baseline=cpu_baseline, extra=extra)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
