"""Times the R-CNN box stage at the config-4 shape (16 tiles 640 x 512, FPN levels 160 x 128 .. 20 x 16, C = 256, 1000 proposals per
tile, Shared2FCBBoxHead 12544 -> 1024 -> 1024 -> 2 | 4) with CUDA events and writes JSON under --out:
  python tools/bench_rcnn.py --out DIR [--iters 20] [--no-oracle]
Achieved bytes and FLOP/s are computed from the shapes below; the oracle's CPU time for the same batch is measured once."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def timed(fn, iters):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--no-oracle', action='store_true')
    a = ap.parse_args()
    from oracle import roi as orr
    from pointtinybenchmark_b200 import ops, registry
    dev = torch.device('cuda:0')
    B, size, C, n, OH = 16, (512, 640), 256, 1000, 7
    g = torch.Generator().manual_seed(0)
    feats = [torch.randn(B, C, size[0] // s, size[1] // s, generator=g).to(dev) for s in orr.STRIDES]
    xy = torch.rand(B, n, 2, generator=g) * torch.tensor([size[1] - 8., size[0] - 8.])
    wh = torch.exp(torch.rand(B, n, 2, generator=g) * 5.5) + 2
    props = [torch.cat([xy[b], torch.minimum(xy[b] + wh[b], torch.tensor([size[1] * 1., size[0] * 1.])), torch.rand(n, 1, generator=g)], 1).to(dev)
             for b in range(B)]
    metas = [dict(img_shape=(size[0], size[1], 3), scale_factor=np.ones(4, np.float32)) for _ in range(B)]
    registry.register_roi_heads()
    cfg = orr.roi_head_cfg(C)
    head = registry.build_head(dict(type='StandardRoIHead', **cfg)).to(dev)
    head.bbox_head.load_state_dict({k: v.to(dev) for k, v in orr.head_weights(1, C, 'trained').items()})
    rcnn = cfg['test_cfg']['rcnn']
    M = B * n
    rois = torch.cat([torch.cat([torch.full((n, 1), float(b), device=dev), p[:, :4]], 1) for b, p in enumerate(props)]).contiguous()
    maps = [ops.to_nhwc(f).contiguous() for f in feats]
    scales = [1 / s for s in orr.STRIDES]
    bh = head.bbox_head
    p6, p7, pout = bh._packs()
    h, l, inv = ops.roi_align(maps, rois, (OH, OH), scales, 0, True, f16_pair=True)
    y6 = ops.linear_tc_f16(h, l, p6, 1024, bh.shared_fcs[0].bias.detach(), inv)
    h6, l6 = ops.relu_split_f16(y6, 1024)
    y7 = ops.linear_tc_f16(h6, l6, p7, 1024, bh.shared_fcs[1].bias.detach())
    h7, l7 = ops.relu_split_f16(y7, 1024)
    bias = torch.cat([bh.fc_cls.bias.detach(), bh.fc_reg.bias.detach()])
    y8 = ops.linear_tc_f16(h7, l7, pout, 6, bias)
    K6 = C * OH * OH
    t = {}
    t['roi_align_fp32_ms'] = timed(lambda: ops.roi_align(maps, rois, (OH, OH), scales, 0, True), a.iters)
    t['roi_align_f16_pair_ms'] = timed(lambda: ops.roi_align(maps, rois, (OH, OH), scales, 0, True, f16_pair=True), a.iters)
    t['fc6_gemm_ms'] = timed(lambda: ops.linear_tc_f16(h, l, p6, 1024, bh.shared_fcs[0].bias.detach(), inv), a.iters)
    t['relu_split_ms'] = timed(lambda: ops.relu_split_f16(y6, 1024), a.iters)
    t['fc7_gemm_ms'] = timed(lambda: ops.linear_tc_f16(h6, l6, p7, 1024, bh.shared_fcs[1].bias.detach()), a.iters)
    t['cls_reg_gemm_ms'] = timed(lambda: ops.linear_tc_f16(h7, l7, pout, 6, bias), a.iters)
    img_hw = torch.tensor([[size[0], size[1]]] * B, dtype=torch.int32, device=dev)

    def decode_nms():
        boxes, _, cand = ops.rcnn_bbox_decode(rois, n, y8[:M, :2], y8[:M, 2:6], 1, orr.MEANS, orr.STDS, img_hw, mask_padding=True,
                                              want_scores=False)
        cnt = ops.multiclass_nms_boxes(boxes.view(B, n, 4), cand, 0.05, 0.5, 1024)[0]
        cnt.cpu()
    t['decode_nms_ms'] = timed(decode_nms, a.iters)
    t['stage_ms'] = timed(lambda: head.simple_test_bboxes(feats, metas, list(props), rcnn), a.iters)
    Mp = h.shape[0]
    fl6, fl7 = 2.0 * M * K6 * 1024, 2.0 * M * 1024 * 1024
    map_bytes = sum(f.numel() * 4 for f in feats)
    res = dict(
        shape=dict(tiles=B, tile_hw=list(size), C=C, rois=M, rows_padded=Mp, fc6_K=K6),
        times_ms=t,
        tiles_per_s=B / (t['stage_ms'] / 1e3),
        roi_align_fp32_GBps=(M * K6 * 4 + map_bytes) / (t['roi_align_fp32_ms'] / 1e3) / 1e9,
        roi_align_f16_pair_GBps=(M * K6 * 4 + 2 * map_bytes) / (t['roi_align_f16_pair_ms'] / 1e3) / 1e9,
        bytes_note='RoIAlign writes M*C*49*4 B (fp32, or two fp16 terms); reads the level maps once (plus once more for max|feat| in '
                   'the fp16 mode); the sampled taps themselves are L2 hits and are not counted',
        fc6_GFLOP=fl6 / 1e9, fc7_GFLOP=fl7 / 1e9,
        fc6_TFLOPs=fl6 / (t['fc6_gemm_ms'] / 1e3) / 1e12, fc7_TFLOPs=fl7 / (t['fc7_gemm_ms'] / 1e3) / 1e12,
        flop_note='useful fp32-equivalent FLOP (2*M*K*N); the tensor cores run three fp16 products per step (h*h + l*h + h*l)',
    )
    try:
        res['gpu'] = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                                    capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:      # noqa: BLE001
        res['gpu'] = f'unknown ({e})'
    res['device_name'] = torch.cuda.get_device_name(0)
    if not a.no_oracle:
        torch.set_num_threads(os.cpu_count())
        cpu_feats = [f.cpu() for f in feats]
        cpu_props = [p.cpu() for p in props]
        t0 = time.perf_counter()
        orr.simple_test_bboxes(cpu_feats, cpu_props, metas, orr.head_weights(1, C, 'trained'), rcnn, orr.STRIDES, orr.MEANS, orr.STDS)
        res['oracle_cpu_s'] = time.perf_counter() - t0
        res['oracle_cpu_threads'] = torch.get_num_threads()
    os.makedirs(a.out, exist_ok=True)
    path = os.path.join(a.out, 'bench_rcnn.json')
    json.dump(res, open(path, 'w'), indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()
