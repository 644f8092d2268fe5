"""Torch-CPU restatement of the R-CNN box stage (BASELINE.json config 4): the checker of pointtinybenchmark_b200/roi_head.py.

  roi_align            mmcv RoIAlign forward (avg pooling; mmcv/ops/csrc/common/cuda/roi_align_cuda_kernel.cuh, third-party), in
                       torchvision's CPU operation order; pinned against torchvision.ops.roi_align in tests/test_roi_oracle.py
  map_roi_levels       single_level_roi_extractor.py:34-53
  roi_extract          single_level_roi_extractor.py:55-100 (levels, then one roi_align per level)
  bbox_head_forward    convfc_bbox_head.py:151-190 (Shared2FCBBoxHead: flatten, fc6 + ReLU, fc7 + ReLU, fc_cls, fc_reg)
  get_bboxes           bbox_head.py:310-435 (softmax, delta2bbox with clip, rescale, multiclass_nms per image)
  simple_test_bboxes   test_mixins.py:50-155 (zero padding rows PREPENDED per image, their scores / deltas zeroed)
"""
import numpy as np
import torch
import torch.nn.functional as F

from oracle import p2p as op2p


def roi_align(feat, rois, output_size=(7, 7), spatial_scale=1.0, sampling_ratio=0, aligned=True, chunk=256):
    """feat (B, C, H, W), rois (M, 5) -> (M, C, oh, ow) fp32."""
    B, C, H, W = feat.shape
    oh, ow = output_size
    M = rois.shape[0]
    out = feat.new_zeros((M, C, oh, ow))
    fl = feat.permute(0, 2, 3, 1).reshape(-1, C)                 # (B*H*W, C)
    off = 0.5 if aligned else 0.0
    for s in range(0, M, chunk):
        r = rois[s:s + chunk].float()
        n = r.shape[0]
        b = r[:, 0].long()
        x0 = r[:, 1] * spatial_scale - off
        y0 = r[:, 2] * spatial_scale - off
        rw = r[:, 3] * spatial_scale - off - x0
        rh = r[:, 4] * spatial_scale - off - y0
        if not aligned:
            rw, rh = rw.clamp(min=1.0), rh.clamp(min=1.0)
        bw, bh = rw / ow, rh / oh
        if sampling_ratio > 0:
            gh = torch.full((n,), sampling_ratio, dtype=torch.long)
            gw = gh.clone()
        else:
            gh, gw = torch.ceil(rh / oh).long(), torch.ceil(rw / ow).long()
        cnt = (gh * gw).clamp(min=1).float()
        acc = feat.new_zeros((n, oh, ow, C))
        ph = torch.arange(oh, dtype=torch.float32)
        pw = torch.arange(ow, dtype=torch.float32)
        for iy in range(int(gh.max().clamp(min=0)) if n else 0):
            y = (y0[:, None] + ph[None] * bh[:, None]) + (iy + 0.5) * bh[:, None] / gh[:, None].float()      # (n, oh)
            for ix in range(int(gw.max().clamp(min=0))):
                x = (x0[:, None] + pw[None] * bw[:, None]) + (ix + 0.5) * bw[:, None] / gw[:, None].float()  # (n, ow)
                yy, xx = y[:, :, None].expand(n, oh, ow), x[:, None, :].expand(n, oh, ow)
                ok = ((iy < gh) & (ix < gw))[:, None, None] & ~((yy < -1) | (yy > H) | (xx < -1) | (xx > W))
                yc, xc = yy.clamp(min=0), xx.clamp(min=0)
                yc, xc = torch.where(ok, yc, 0.), torch.where(ok, xc, 0.)      # masked samples (grid 0: 0/0) read a valid cell
                ylo, xlo = yc.long(), xc.long()
                yhi_clip, xhi_clip = ylo >= H - 1, xlo >= W - 1
                ylo = torch.where(yhi_clip, torch.full_like(ylo, H - 1), ylo)
                xlo = torch.where(xhi_clip, torch.full_like(xlo, W - 1), xlo)
                yhi = torch.where(yhi_clip, ylo, ylo + 1)
                xhi = torch.where(xhi_clip, xlo, xlo + 1)
                yc = torch.where(yhi_clip, ylo.float(), yc)
                xc = torch.where(xhi_clip, xlo.float(), xc)
                ly, lx = yc - ylo.float(), xc - xlo.float()
                hy, hx = 1. - ly, 1. - lx
                base = (b * H * W)[:, None, None]

                def tap(yi, xi):
                    return fl[(base + yi * W + xi).reshape(-1)].view(n, oh, ow, C)
                val = ((hy * hx)[..., None] * tap(ylo, xlo) + (hy * lx)[..., None] * tap(ylo, xhi)) + (ly * hx)[..., None] * tap(yhi, xlo)
                val = val + (ly * lx)[..., None] * tap(yhi, xhi)
                acc += torch.where(ok[..., None], val, val.new_zeros(()))
        out[s:s + n] = (acc / cnt[:, None, None, None]).permute(0, 3, 1, 2)
    return out


def map_roi_levels(rois, num_levels, finest_scale=56):
    """single_level_roi_extractor.py:34-53 (fp32 torch ops, exactly the reference's)."""
    scale = torch.sqrt((rois[:, 3] - rois[:, 1]) * (rois[:, 4] - rois[:, 2]))
    lv = torch.floor(torch.log2(scale / finest_scale + 1e-6))
    return lv.clamp(min=0, max=num_levels - 1).long()


def roi_extract(feats, rois, strides, output_size=(7, 7), sampling_ratio=0, aligned=True, finest_scale=56):
    """single_level_roi_extractor.py:55-100 -> (M, C, oh, ow)."""
    L = len(feats)
    if L == 1:
        return roi_align(feats[0], rois, output_size, 1.0 / strides[0], sampling_ratio, aligned)
    out = feats[0].new_zeros((rois.shape[0], feats[0].shape[1]) + tuple(output_size))
    lv = map_roi_levels(rois, L, finest_scale)
    for i in range(L):
        idx = (lv == i).nonzero(as_tuple=False).squeeze(1)
        if idx.numel():
            out[idx] = roi_align(feats[i], rois[idx], output_size, 1.0 / strides[i], sampling_ratio, aligned)
    return out


def bbox_head_forward(x, w):
    """convfc_bbox_head.py:151-190; w: state_dict of Shared2FCBBoxHead.  x (M, C, oh, ow) -> cls_score, bbox_pred."""
    h = x.flatten(1)
    h = F.relu(F.linear(h, w['shared_fcs.0.weight'], w['shared_fcs.0.bias']))
    h = F.relu(F.linear(h, w['shared_fcs.1.weight'], w['shared_fcs.1.bias']))
    return F.linear(h, w['fc_cls.weight'], w['fc_cls.bias']), F.linear(h, w['fc_reg.weight'], w['fc_reg.bias'])


def delta2bbox(rois, deltas, means, stds, max_shape, wh_ratio_clip=16 / 1000):
    """delta_xywh_bbox_coder.py:144-270 for (n, 4) rois and (n, 4N) deltas, clipped to max_shape (h, w)."""
    n, N4 = deltas.shape
    d = deltas * deltas.new_tensor(stds).repeat(N4 // 4) + deltas.new_tensor(means).repeat(N4 // 4)
    dx, dy, dw, dh = d[:, 0::4], d[:, 1::4], d[:, 2::4], d[:, 3::4]
    px = ((rois[:, 0] + rois[:, 2]) * 0.5)[:, None]
    py = ((rois[:, 1] + rois[:, 3]) * 0.5)[:, None]
    pw = (rois[:, 2] - rois[:, 0])[:, None]
    ph = (rois[:, 3] - rois[:, 1])[:, None]
    mr = np.abs(np.log(wh_ratio_clip))
    dw, dh = dw.clamp(min=-mr, max=mr), dh.clamp(min=-mr, max=mr)
    gw, gh = pw * dw.exp(), ph * dh.exp()
    gx, gy = px + pw * dx, py + ph * dy
    b = torch.stack([gx - gw * 0.5, gy - gh * 0.5, gx + gw * 0.5, gy + gh * 0.5], dim=-1).view(n, N4)
    mx = b.new_tensor([max_shape[1], max_shape[0]] * (N4 // 2))
    b = torch.where(b < 0, b.new_tensor(0.), b)
    return torch.where(b > mx, mx.expand_as(b), b)


def get_bboxes_single(rois, cls_score, bbox_pred, img_shape, scale_factor, rescale, cfg, means, stds, return_inds=False):
    """bbox_head.py:310-435 for one image: rois (n, 5)."""
    scores = F.softmax(cls_score, dim=-1)
    boxes = delta2bbox(rois[:, 1:], bbox_pred, means, stds, img_shape)
    if rescale and boxes.shape[0] > 0:
        boxes = boxes / boxes.new_tensor(np.asarray(scale_factor, dtype=np.float32)).repeat(boxes.shape[1] // 4)
    if cfg is None:
        return boxes, scores
    nms = dict(cfg['nms'])
    dets, labels, keep, _ = op2p.multiclass_nms(boxes, scores, cfg['score_thr'], nms.get('iou_threshold', 0.5), cfg['max_per_img'])
    return (dets, labels, keep) if return_inds else (dets, labels)


def simple_test_bboxes(feats, proposals, img_metas, w, cfg, strides, means, stds, rescale=False, roi_kw=None, return_inds=False):
    """test_mixins.py:50-155 (padding quirk included) -> (dets list, labels list[, keep list])."""
    n = max(p.shape[0] for p in proposals)
    B = len(proposals)
    padded = [torch.cat([p.new_zeros((n - p.shape[0], p.shape[1])), p]) for p in proposals]
    rois = torch.cat([torch.arange(B, dtype=torch.float32).view(-1, 1, 1).expand(B, n, 1), torch.stack(padded)[..., :4]], -1).view(-1, 5)
    x = roi_extract(feats, rois, strides, **(roi_kw or {}))
    cls, reg = bbox_head_forward(x, w)
    rois = rois.view(B, n, 5)
    cls, reg = cls.view(B, n, -1).clone(), reg.view(B, n, -1).clone()
    mask = rois.abs()[..., 1:].sum(dim=-1) == 0
    cls[mask] = 0
    reg[mask] = 0
    out = [get_bboxes_single(rois[b], cls[b], reg[b], img_metas[b]['img_shape'], img_metas[b]['scale_factor'], rescale, cfg, means, stds,
                             return_inds) for b in range(B)]
    return tuple(list(t) for t in zip(*out))


# ---- seeded inputs of the golden fixture and the tests (faster_rcnn_r50_fpn_1x_TinyPerson640.py:45-70, 100-120) ----
MEANS, STDS = (0., 0., 0., 0.), (0.1, 0.1, 0.2, 0.2)
STRIDES = (4, 8, 16, 32)
GOLDEN_CASES = [dict(name='init', seed=11, variant='init', keep=(None, 180, 0)),
                dict(name='trained', seed=12, variant='trained', keep=(None, 230, 60))]


def roi_head_cfg(C, num_classes=1, fc_out=1024):
    return dict(
        bbox_roi_extractor=dict(type='SingleRoIExtractor', roi_layer=dict(type='RoIAlign', output_size=7, sampling_ratio=0), out_channels=C,
                                featmap_strides=list(STRIDES)),
        bbox_head=dict(type='Shared2FCBBoxHead', in_channels=C, fc_out_channels=fc_out, roi_feat_size=7, num_classes=num_classes,
                       bbox_coder=dict(type='DeltaXYWHBBoxCoder', target_means=list(MEANS), target_stds=list(STDS)), reg_class_agnostic=False,
                       loss_cls=dict(type='CrossEntropyLoss', use_sigmoid=False, loss_weight=1.0), loss_bbox=dict(type='L1Loss', loss_weight=1.0)),
        test_cfg=dict(rcnn=dict(score_thr=0.05, nms=dict(type='nms', iou_threshold=0.5), max_per_img=-1)))


def head_weights(seed, C, variant, num_classes=1, fc_out=1024):
    """'init': the reference's init (Xavier-uniform fcs, N(0, 0.01) fc_cls, N(0, 0.001) fc_reg, zero biases);
    'trained': larger predictor weights and biases so that the foreground scores spread over (0, 1) and the boxes move."""
    g = torch.Generator().manual_seed(seed)

    def xavier(o, i):
        a = float(np.sqrt(6.0 / (i + o)))
        return (torch.rand(o, i, generator=g) * 2 - 1) * a
    w = {'shared_fcs.0.weight': xavier(fc_out, C * 49), 'shared_fcs.0.bias': torch.zeros(fc_out),
         'shared_fcs.1.weight': xavier(fc_out, fc_out), 'shared_fcs.1.bias': torch.zeros(fc_out),
         'fc_cls.weight': torch.randn(num_classes + 1, fc_out, generator=g) * 0.01, 'fc_cls.bias': torch.zeros(num_classes + 1),
         'fc_reg.weight': torch.randn(4 * num_classes, fc_out, generator=g) * 0.001, 'fc_reg.bias': torch.zeros(4 * num_classes)}
    if variant == 'trained':
        w['shared_fcs.0.bias'] = torch.randn(fc_out, generator=g) * 0.05
        w['shared_fcs.1.bias'] = torch.randn(fc_out, generator=g) * 0.05
        w['fc_cls.weight'] = torch.randn(num_classes + 1, fc_out, generator=g) * 0.3
        w['fc_cls.bias'] = torch.randn(num_classes + 1, generator=g) * 0.5
        w['fc_reg.weight'] = torch.randn(4 * num_classes, fc_out, generator=g) * 0.1
    return w


def synth_rcnn_inputs(name='init', seed=11, variant='init', keep=(None, None), C=64, size=(128, 160), num_classes=1):
    """4-level FPN maps (B, C, ceil(h/s), ceil(w/s)), proposals of oracle.anchors' seeded RPN outputs through the RPN oracle, image b keeping
    its first keep[b] proposals (unequal counts: the padding path), metas with scale factors != 1, head weights of `variant`."""
    from oracle import anchors as oa
    B = len(keep)
    g = torch.Generator().manual_seed(seed)
    feats = [torch.randn(B, C, -(-size[0] // s), -(-size[1] // s), generator=g) for s in STRIDES]
    cls, box, shapes = oa.synth_rpn_inputs(seed, B=B, size=size)
    props = oa.rpn_proposals(cls, box, shapes, dict(oa.RPN_CFG, nms_pre=1000, max_per_img=1000))
    props = [p[:k] if k is not None else p for p, k in zip(props, keep)]
    metas = [dict(img_shape=sh, scale_factor=np.array([1.25, 1.5, 1.25, 1.5], dtype=np.float32), pad_shape=(size[0], size[1], 3))
             for sh in shapes]
    return dict(feats=feats, proposals=props, img_metas=metas, strides=list(STRIDES), C=C,
                weights=head_weights(seed + 1000, C, variant, num_classes))
