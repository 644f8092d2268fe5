"""R-CNN box stage on the B200 (pointtinybenchmark_b200/roi_head.py over ptb_roi_align, ptb_conv_tc_f16x2, ptb_relu_split_f16,
ptb_rcnn_bbox_decode and ptb_multiclass_nms_boxes) against oracle/roi.py and the reference's golden detections."""
import os

import numpy as np
import pytest
import torch

from oracle import p2p as op2p
from oracle import roi as orr
from tests.test_roi_oracle import edge_rois, planted_level_rois

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), 'golden')
DEV = torch.device('cuda:0')


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / max(float(b.abs().max()), 1e-30)) if b.numel() else 0.0


def build_head(C, weights=None, num_classes=1):
    from pointtinybenchmark_b200 import registry
    registry.register_roi_heads()
    cfg = orr.roi_head_cfg(C, num_classes)
    head = registry.build_head(dict(type='StandardRoIHead', **cfg)).to(DEV)
    if weights is not None:
        head.bbox_head.load_state_dict({k: v.to(DEV) for k, v in weights.items()})
    return head, cfg


@pytest.mark.parametrize('aligned', [True, False])
@pytest.mark.parametrize('sr', [0, 2])
def test_roi_align_features_and_levels(aligned, sr):
    from pointtinybenchmark_b200 import ops
    g = torch.Generator().manual_seed(5)
    feats = [torch.randn(2, 64, -(-100 // s), -(-120 // s), generator=g) for s in orr.STRIDES]
    rois = torch.cat([edge_rois(6, 200, 2, (100, 120)), torch.tensor([[1., 0., 0., 100., 90.], [0., 2., 3., 119., 99.]])])
    maps = [ops.to_nhwc(f.to(DEV)).contiguous() for f in feats]
    out, lvl = ops.roi_align(maps, rois.to(DEV), (7, 7), [1 / s for s in orr.STRIDES], sr, aligned, want_levels=True)
    ref = orr.roi_extract(feats, rois, orr.STRIDES, (7, 7), sr, aligned)
    e = rel(out.permute(0, 3, 1, 2), ref)
    print(f'roi_align aligned={aligned} sr={sr}: max scale-relative error {e:.2e}')
    assert e <= 1e-4
    assert torch.equal(lvl.long().cpu(), orr.map_roi_levels(rois, 4))
    one = ops.roi_align(maps[:1], rois.to(DEV), (7, 7), [0.25], sr, aligned)
    assert rel(one.permute(0, 3, 1, 2), orr.roi_extract(feats[:1], rois, [4], (7, 7), sr, aligned)) <= 1e-4
    # fp16 pair mode: (h + l) / scale reproduces the fp32 mode to 2^-20 of max|feat|
    h, l, inv = ops.roi_align(maps, rois.to(DEV), (7, 7), [1 / s for s in orr.STRIDES], sr, aligned, f16_pair=True)
    M = rois.shape[0]
    assert h.shape[0] % 16 == 0 and bool((h[M:] == 0).all())
    pair = (h[:M].double() + l[:M].double()) * float(inv)
    amax = max(float(f.abs().max()) for f in feats)
    d = float((pair - out.reshape(M, -1).double()).abs().max())
    print(f'fp16 pair vs fp32: {d / amax:.2e} of max|feat|')
    assert d <= 2 ** -20 * amax


def test_planted_levels_bit_exact():
    from pointtinybenchmark_b200 import roi_head
    rois = planted_level_rois()
    ext = roi_head.SingleRoIExtractor(dict(type='RoIAlign', output_size=7, sampling_ratio=0), 256, [4, 8, 16, 32, 64])
    for L in (4, 5):
        assert torch.equal(ext.map_roi_levels(rois.to(DEV), L).cpu(), orr.map_roi_levels(rois, L))


def test_box_head_gemms_vs_float64():
    head, _ = build_head(256, orr.head_weights(3, 256, 'trained'))
    g = torch.Generator().manual_seed(4)
    x = torch.randn(300, 256, 7, 7, generator=g).abs()
    cls, reg = head.bbox_head(x.to(DEV))
    w = {k: v.double() for k, v in orr.head_weights(3, 256, 'trained').items()}
    rc, rr = orr.bbox_head_forward(x.double(), w)
    print(f'box head: cls {rel(cls, rc):.2e}, reg {rel(reg, rr):.2e}')
    assert rel(cls, rc) <= 1e-4 and rel(reg, rr) <= 1e-4


def match_err(a, r):
    """scale-relative error of the best one-to-one pairing of two detection sets (rows of near-equal scores may come in either order)."""
    from scipy.optimize import linear_sum_assignment
    a, r = a.double().cpu(), r.double().cpu()
    if r.shape[0] == 0:
        return 0.0
    cost = (a[:, None, :] - r[None, :, :]).abs().amax(-1)
    i, j = linear_sum_assignment(cost.numpy())
    return float(cost[i, j].max()) / max(float(r.abs().max()), 1e-30)


@pytest.mark.parametrize('case', [c['name'] for c in orr.GOLDEN_CASES])
@pytest.mark.parametrize('rescale', [False, True])
def test_simple_test_bboxes_vs_golden(case, rescale):
    gold = np.load(os.path.join(GOLD, 'rcnn_box_stage.npz'))
    c = [c for c in orr.GOLDEN_CASES if c['name'] == case][0]
    inp = orr.synth_rcnn_inputs(**c)
    head, cfg = build_head(inp['C'], inp['weights'])
    feats = [f.to(DEV) for f in inp['feats']]
    dets, labels = head.simple_test_bboxes(feats, inp['img_metas'], [p.to(DEV) for p in inp['proposals']],
                                           cfg["test_cfg"]["rcnn"], rescale=rescale)
    worst = 0.0
    for b in range(len(dets)):
        gd = torch.from_numpy(gold[f'{case}_r{int(rescale)}_dets{b}'])
        assert dets[b].shape == gd.shape, (b, dets[b].shape, gd.shape)
        assert np.array_equal(np.sort(labels[b].cpu().numpy()), np.sort(gold[f'{case}_r{int(rescale)}_labels{b}']))
        e = match_err(dets[b], gd)
        worst = max(worst, e)
        assert e <= 1e-4
        n_pad = max(p.shape[0] for p in inp['proposals']) - inp['proposals'][b].shape[0]
        assert int(((dets[b][:, :4] == 0).all(1) & (dets[b][:, 4] == 0.5)).sum()) >= n_pad     # the reference's padding detections
    print(f'{case} rescale={rescale}: max scale-relative error {worst:.2e}')
    # run to run: bit-identical
    d2, _ = head.simple_test_bboxes(feats, inp['img_metas'], [p.to(DEV) for p in inp['proposals']], cfg['test_cfg']['rcnn'], rescale=rescale)
    assert all(torch.equal(x, y) for x, y in zip(dets, d2))
    res = head.simple_test(feats, [p.to(DEV) for p in inp['proposals']], inp['img_metas'], rescale=rescale)
    assert len(res) == len(dets) and res[0][0].shape == (dets[0].shape[0], 5)


def test_config4_shape_keep_lists_replay():
    """16 tiles 640 x 512, levels 160 x 128 .. 20 x 16, C = 256, proposals from the library's own RPNProposals: the oracle NMS fed with
    the product's boxes and scores reproduces the product's detections exactly."""
    from oracle import anchors as oa
    from pointtinybenchmark_b200 import ops
    from pointtinybenchmark_b200.rpn import RPNProposals
    B, size, C = 16, (512, 640), 256
    cls, box, shapes = oa.synth_rpn_inputs(21, B=B, size=size)
    rpn = RPNProposals(dict(type='AnchorGenerator', scales=[2], ratios=[0.5, 1.0, 2.0], strides=[4, 8, 16, 32, 64]),
                       test_cfg=dict(nms_pre=1000, max_per_img=1000, nms=dict(type='nms', iou_threshold=0.7), min_bbox_size=0))
    metas = [dict(img_shape=sh, scale_factor=np.ones(4, np.float32), pad_shape=(size[0], size[1], 3)) for sh in shapes]
    props = rpn.get_bboxes([c.to(DEV) for c in cls], [b.to(DEV) for b in box], metas)
    g = torch.Generator().manual_seed(22)
    feats = [torch.randn(B, C, size[0] // s, size[1] // s, generator=g).to(DEV) for s in orr.STRIDES]
    head, cfg = build_head(C, orr.head_weights(23, C, 'trained'))
    dets, labels = head.simple_test_bboxes(feats, metas, list(props), cfg['test_cfg']['rcnn'])
    n = max(p.shape[0] for p in props)
    rois = torch.zeros((B, n, 5), device=DEV)
    rois[..., 0] = torch.arange(B, device=DEV, dtype=torch.float32)[:, None]
    rois[..., 1:] = torch.stack([torch.cat([p.new_zeros((n - p.shape[0], 5)), p]) for p in props])[..., :4]
    rois = rois.view(-1, 5)
    r = head._bbox_forward(feats, rois)
    img_hw = torch.tensor([[s[0], s[1]] for s in shapes], dtype=torch.int32, device=DEV)
    boxes, scores, _ = ops.rcnn_bbox_decode(rois, n, r['cls_score'], r['bbox_pred'], 1, orr.MEANS, orr.STDS, img_hw, mask_padding=True,
                                            want_candidates=False)
    for b in range(B):
        od, ol, _, _ = op2p.multiclass_nms(boxes.view(B, n, 4)[b].cpu(), scores.view(B, n, 2)[b].cpu(), 0.05, 0.5, -1)
        assert torch.equal(od, dets[b].cpu()) and torch.equal(ol, labels[b].cpu()), b
    # end to end against the oracle where the score margins are decisive
    e2e = orr.simple_test_bboxes([f[:2].cpu() for f in feats], [p.cpu() for p in props[:2]], metas[:2], orr.head_weights(23, C, 'trained'),
                                 cfg['test_cfg']['rcnn'], orr.STRIDES, orr.MEANS, orr.STDS)
    d2, _ = head.simple_test_bboxes([f[:2] for f in feats], metas[:2], list(props[:2]), cfg['test_cfg']['rcnn'])
    for b in range(2):
        assert d2[b].shape == e2e[0][b].shape
        e = match_err(d2[b], e2e[0][b])
        print(f'config-4 shape image {b}: {d2[b].shape[0]} dets, max scale-relative error vs oracle {e:.2e}')
        assert e <= 1e-4


def test_cpu_tensors_and_limits_raise():
    head, cfg = build_head(64)
    with pytest.raises(RuntimeError):
        head.simple_test_bboxes([torch.zeros(1, 64, 8, 8)] * 4, [dict(img_shape=(32, 32, 3), scale_factor=np.ones(4))],
                                [torch.zeros(3, 5)], cfg['test_cfg']['rcnn'])
    big, cfg5 = build_head(64, num_classes=5)
    props = [torch.tensor([[0., 0., 10., 10., 0.9]], device=DEV).repeat(1000, 1)]
    with pytest.raises(NotImplementedError):
        big.simple_test_bboxes([torch.zeros(1, 64, 8, 8, device=DEV)] * 4, [dict(img_shape=(32, 32, 3), scale_factor=np.ones(4))], props,
                               cfg5['test_cfg']['rcnn'])
    from pointtinybenchmark_b200 import ops
    with pytest.raises(ValueError):
        ops.roi_align([torch.zeros(1, 4, 4, 48, device=DEV)], torch.zeros(1, 5, device=DEV))
