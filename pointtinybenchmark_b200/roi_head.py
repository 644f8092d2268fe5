"""R-CNN box stage of the dense-anchor detector (BASELINE.json config 4, TinyPerson Faster R-CNN) — mirrors of the reference classes
with their names, constructor keywords, method signatures, return structures and state_dict keys:

  SingleRoIExtractor   roi_extractors/single_level_roi_extractor.py:8-100 (+ base_roi_extractor.py) over ptb_roi_align: level choice
                       and mmcv RoIAlign of every RoI of the batch on every level in one launch.
  Shared2FCBBoxHead    bbox_heads/convfc_bbox_head.py:193-207 + bbox_head.py: fc6 / fc7 (+ ReLU) and the fused fc_cls | fc_reg GEMM on
                       the tcgen05 kernel (ptb_conv_tc_f16x2, 1 tap, RoIs as pixels), ReLU + operand split in one kernel
                       (ptb_relu_split_f16); get_bboxes over ptb_rcnn_bbox_decode + ptb_multiclass_nms_boxes.
  StandardRoIHead      standard_roi_head.py + test_mixins.py:50-155: simple_test_bboxes / simple_test for the whole batch, with the
                       reference's padding of unequal proposal counts (zero rows PREPENDED; they score 1 / (N + 1) and come out as
                       zero-area detections at (0, 0, 0, 0)), one NMS launch and one device-to-host copy of the counts per batch.

Inference only (forward_train, mask and shared heads raise NotImplementedError).  CUDA tensors only: there is no CPU path.
"""
import numpy as np
import torch
import torch.nn as nn

from . import ops
from .layers import PackedWeightsMixin
from .registry import CfgNode

_SLICE = 256          # output columns per tensor-core GEMM launch (the conv kernel's N limit)


def _need_cuda(t, who):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f'{who} (B200) runs on CUDA tensors only; there is no CPU fallback')


def _pack_slices(owner, key, weight):
    """fp16 (h, l) packings of the (n_out, K) matrix `weight` in column slices of <= 256 outputs, cached on `owner` under
    `_ptb_packed_tc` (dropped by layers.invalidate_packed)."""
    cache = getattr(owner, '_ptb_packed_tc', None)
    if cache is None or cache[0] != key:
        w = weight.detach().float().contiguous()
        owner._ptb_packed_tc = (key, [ops.conv_tc_pack_weight_f16(w[s:s + _SLICE].contiguous(), 1) for s in range(0, w.shape[0], _SLICE)])
    return owner._ptb_packed_tc[1]


def _wkey(*params):
    return tuple((p.data_ptr(), p._version, str(p.device)) for p in params)


class SingleRoIExtractor(nn.Module):
    """single_level_roi_extractor.py:8-100.  roi_layer = dict(type='RoIAlign', output_size, sampling_ratio=0, pool_mode='avg',
    aligned=True); pool_mode='max' and roi_scale_factor are not implemented."""

    def __init__(self, roi_layer, out_channels, featmap_strides, finest_scale=56, init_cfg=None):
        super().__init__()
        cfg = dict(roi_layer)
        if cfg.pop('type', 'RoIAlign') != 'RoIAlign':
            raise NotImplementedError('SingleRoIExtractor: only roi_layer type RoIAlign is implemented')
        if cfg.pop('pool_mode', 'avg') != 'avg':
            raise NotImplementedError("RoIAlign(pool_mode='max')")
        cfg.pop('use_torchvision', None)
        os_ = cfg.pop('output_size')
        self.output_size = (int(os_), int(os_)) if np.isscalar(os_) else tuple(int(v) for v in os_)
        self.sampling_ratio = int(cfg.pop('sampling_ratio', 0))
        self.aligned = bool(cfg.pop('aligned', True))
        if cfg:
            raise TypeError(f'RoIAlign: unexpected arguments {sorted(cfg)}')
        if not 1 <= len(featmap_strides) <= 5:
            raise NotImplementedError('SingleRoIExtractor: 1 to 5 feature levels')
        self.out_channels = out_channels
        self.featmap_strides = list(featmap_strides)
        self.finest_scale = finest_scale
        self.fp16_enabled = False

    @property
    def num_inputs(self):
        return len(self.featmap_strides)

    def _levels(self, feats):
        if len(feats) != self.num_inputs:
            raise ValueError(f'{len(feats)} feature maps for {self.num_inputs} strides')
        for f in feats:
            _need_cuda(f, 'SingleRoIExtractor')
        return [ops.to_nhwc(f.float()).contiguous() for f in feats], [1.0 / s for s in self.featmap_strides]

    def map_roi_levels(self, rois, num_levels):
        """(k,) int64 level per RoI, bit-exact with the reference's fp32 torch arithmetic (computed by ptb_roi_align)."""
        _need_cuda(rois, 'SingleRoIExtractor')
        dummy = [torch.zeros((1, 1, 1, 32), device=rois.device) for _ in range(num_levels)]
        _, lvl = ops.roi_align(dummy, rois.float().contiguous(), (1, 1), [1.0] * num_levels, 1, self.aligned, self.finest_scale,
                               want_levels=True)
        return lvl.long()

    def forward(self, feats, rois, roi_scale_factor=None):
        """(M, C, oh, ow) fp32: a view of the kernel's channels-last (M, oh, ow, C) result."""
        if roi_scale_factor is not None:
            raise NotImplementedError('SingleRoIExtractor: roi_scale_factor')
        _need_cuda(rois, 'SingleRoIExtractor')
        maps, scales = self._levels(feats)
        out = ops.roi_align(maps, rois.float().contiguous(), self.output_size, scales, self.sampling_ratio, self.aligned, self.finest_scale)
        return out.permute(0, 3, 1, 2)

    def forward_f16_pair(self, feats, rois):
        """the same features as the (h, l, dev_inv_scale) fp16 operand pair of the box head's first GEMM, rows padded to 16."""
        maps, scales = self._levels(feats)
        return ops.roi_align(maps, rois.float().contiguous(), self.output_size, scales, self.sampling_ratio, self.aligned, self.finest_scale,
                             f16_pair=True)


class Shared2FCBBoxHead(PackedWeightsMixin, nn.Module):
    """convfc_bbox_head.py:193-207 (num_shared_fcs=2, no convs, no branch fcs) with the BBoxHead keywords of bbox_head.py:16-95."""

    def __init__(self, fc_out_channels=1024, with_avg_pool=False, with_cls=True, with_reg=True, roi_feat_size=7, in_channels=256,
                 num_classes=80, bbox_coder=dict(type='DeltaXYWHBBoxCoder', clip_border=True, target_means=[0., 0., 0., 0.],
                                                  target_stds=[0.1, 0.1, 0.2, 0.2]),
                 reg_class_agnostic=False, reg_decoded_bbox=False, reg_predictor_cfg=dict(type='Linear'), cls_predictor_cfg=dict(type='Linear'),
                 loss_cls=dict(type='CrossEntropyLoss', use_sigmoid=False, loss_weight=1.0),
                 loss_bbox=dict(type='SmoothL1Loss', beta=1.0, loss_weight=1.0), init_cfg=None, **kwargs):
        super().__init__()
        extra = {k: v for k, v in kwargs.items() if k not in ('conv_cfg', 'norm_cfg')}
        if extra:
            raise NotImplementedError(f'Shared2FCBBoxHead: unsupported arguments {sorted(extra)}')
        if with_avg_pool or not (with_cls and with_reg) or reg_class_agnostic or reg_decoded_bbox:
            raise NotImplementedError('Shared2FCBBoxHead: with_avg_pool / without cls or reg / reg_class_agnostic / reg_decoded_bbox')
        if dict(reg_predictor_cfg).get('type', 'Linear') != 'Linear' or dict(cls_predictor_cfg).get('type', 'Linear') != 'Linear':
            raise NotImplementedError('Shared2FCBBoxHead: only Linear predictors')
        if dict(loss_cls).get('use_sigmoid', False) or dict(loss_cls).get('type', 'CrossEntropyLoss') != 'CrossEntropyLoss':
            raise NotImplementedError('Shared2FCBBoxHead: softmax cross-entropy classification only')
        bc = dict(bbox_coder)
        if bc.pop('type', 'DeltaXYWHBBoxCoder') != 'DeltaXYWHBBoxCoder' or not bc.get('clip_border', True) or bc.get('add_ctr_clamp', False):
            raise NotImplementedError('Shared2FCBBoxHead: DeltaXYWHBBoxCoder(clip_border=True) only')
        self.means = tuple(float(v) for v in bc.get('target_means', (0., 0., 0., 0.)))
        self.stds = tuple(float(v) for v in bc.get('target_stds', (1., 1., 1., 1.)))
        self.wh_ratio_clip = 16 / 1000                     # DeltaXYWHBBoxCoder.decode default (delta_xywh_bbox_coder.py:66)
        self.roi_feat_size = (roi_feat_size, roi_feat_size) if np.isscalar(roi_feat_size) else tuple(roi_feat_size)
        self.roi_feat_area = self.roi_feat_size[0] * self.roi_feat_size[1]
        self.in_channels, self.num_classes, self.fc_out_channels = in_channels, num_classes, fc_out_channels
        self.reg_class_agnostic, self.reg_decoded_bbox = reg_class_agnostic, reg_decoded_bbox
        self.loss_cls_cfg, self.loss_bbox_cfg = loss_cls, loss_bbox
        self.fp16_enabled = False
        self.shared_fcs = nn.ModuleList([nn.Linear(in_channels * self.roi_feat_area, fc_out_channels),
                                         nn.Linear(fc_out_channels, fc_out_channels)])
        self.fc_cls = nn.Linear(fc_out_channels, num_classes + 1)
        self.fc_reg = nn.Linear(fc_out_channels, 4 * num_classes)
        # reference init_cfg: Xavier-uniform shared fcs, Normal(0.01) fc_cls, Normal(0.001) fc_reg, zero biases
        for fcl in self.shared_fcs:
            nn.init.xavier_uniform_(fcl.weight)
            nn.init.zeros_(fcl.bias)
        nn.init.normal_(self.fc_cls.weight, 0, 0.01)
        nn.init.normal_(self.fc_reg.weight, 0, 0.001)
        nn.init.zeros_(self.fc_cls.bias)
        nn.init.zeros_(self.fc_reg.bias)
        self._init_packed_hooks()

    # ---- packed weights ----
    def _packs(self):
        fc6, fc7 = self.shared_fcs
        C, (oh, ow) = self.in_channels, self.roi_feat_size
        # the reference flattens RoI features as (C, oh, ow); the kernel's rows are channels-last (oh, ow, C): permute fc6's columns once
        p6 = _pack_slices(fc6, _wkey(fc6.weight) + ('fc6_hwc', C),
                          fc6.weight.detach().view(-1, C, oh, ow).permute(0, 2, 3, 1).reshape(fc6.weight.shape[0], -1))
        p7 = _pack_slices(fc7, _wkey(fc7.weight) + ('fc7',), fc7.weight)
        pout = _pack_slices(self.fc_cls, _wkey(self.fc_cls.weight, self.fc_reg.weight) + ('cls|reg',),
                            torch.cat([self.fc_cls.weight.detach(), self.fc_reg.weight.detach()]))
        return p6, p7, pout

    def _forward_pair(self, x_h, x_l, dev_inv_scale, overflow_flag=None):
        """GEMM chain on fp16 operand rows (M_pad, C*oh*ow) -> (M_pad, ldy) logits | deltas (columns [0, N+1) | [N+1, 5N+1))."""
        p6, p7, pout = self._packs()
        fc6, fc7 = self.shared_fcs
        n = self.fc_out_channels
        y = ops.linear_tc_f16(x_h, x_l, p6, n, fc6.bias.detach(), dev_inv_scale)
        h, l = ops.relu_split_f16(y, n, overflow_flag)
        y = ops.linear_tc_f16(h, l, p7, n, fc7.bias.detach())
        h, l = ops.relu_split_f16(y, n, overflow_flag)
        n_out = 5 * self.num_classes + 1
        bias = torch.cat([self.fc_cls.bias.detach(), self.fc_reg.bias.detach()])
        return ops.linear_tc_f16(h, l, pout, n_out, bias)

    def _split_out(self, y, M):
        N = self.num_classes
        return y[:M, :N + 1], y[:M, N + 1:5 * N + 1]

    def forward(self, x):
        """x (M, C, oh, ow) fp32 CUDA -> cls_score (M, N+1), bbox_pred (M, 4N) (inference; no autograd graph)."""
        _need_cuda(x, 'Shared2FCBBoxHead')
        M = x.shape[0]
        rows = x.detach().float().permute(0, 2, 3, 1).reshape(M, -1)
        Mp = (M + 15) // 16 * 16
        buf = torch.zeros((Mp, rows.shape[1]), dtype=torch.float32, device=x.device)
        buf[:M] = rows
        h, l, inv = ops.split_f16(buf, auto_scale=True)
        return self._split_out(self._forward_pair(h, l, inv), M)

    def forward_train(self, *a, **k):
        raise NotImplementedError('Shared2FCBBoxHead: the R-CNN training path (RoIAlign backward, sampler, losses) is not implemented')

    loss = forward_train

    def _nms_args(self, cfg):
        nms = dict(cfg.get('nms', dict(type='nms', iou_threshold=0.5)))
        if nms.pop('type', 'nms') != 'nms' or nms.pop('class_agnostic', False):
            raise NotImplementedError('R-CNN test: only class-aware nms is implemented')
        max_per_img = int(cfg.get('max_per_img', -1))
        if max_per_img > 1024:
            raise NotImplementedError('max_per_img must be <= 1024')
        return float(cfg.get('score_thr', 0.05)), float(nms.get('iou_threshold', nms.get('iou_thr', 0.5))), max_per_img

    def _decode_nms(self, rois, n, cls, reg, img_shapes, scale_factors, rescale, cfg, mask_padding):
        """decode (+ padding mask) for B images of n RoIs each, then one NMS launch; returns per-image (dets, labels) lists."""
        B = len(img_shapes)
        dev = rois.device
        N = self.num_classes
        if cfg is not None and n * N > 4096:
            raise NotImplementedError(f'R-CNN test: {n} RoIs x {N} classes > 4096 NMS candidates per image')
        img_hw = torch.tensor([[int(s[0]), int(s[1])] for s in img_shapes], dtype=torch.int32).to(dev)
        sf = None
        if rescale and n > 0:
            sf = torch.tensor(np.stack([np.broadcast_to(np.asarray(s, dtype=np.float32).reshape(-1), 4) for s in scale_factors]),
                              dtype=torch.float32).to(dev)
        boxes, scores, cand = ops.rcnn_bbox_decode(rois, n, cls, reg, N, self.means, self.stds, img_hw, sf, mask_padding, self.wh_ratio_clip,
                                                   want_scores=cfg is None, want_candidates=cfg is not None)
        if cfg is None:
            return [boxes.view(B, n, -1)[b] for b in range(B)], [scores.view(B, n, -1)[b] for b in range(B)]
        score_thr, iou, max_per_img = self._nms_args(cfg)
        if n == 0:
            return ([boxes.new_zeros((0, 5)) for _ in range(B)], [torch.zeros(0, dtype=torch.long, device=dev) for _ in range(B)])
        kmax = 1024 if max_per_img <= 0 else max_per_img
        cnt, det, lab, _, _ = ops.multiclass_nms_boxes(boxes.view(B, n * N, 4), cand, score_thr, iou, kmax)
        return cnt, det, lab, max_per_img

    def get_bboxes(self, rois, cls_score, bbox_pred, img_shape, scale_factor, rescale=False, cfg=None):
        """bbox_head.py:310-435, 2-D (one image, returns (dets, labels)) and batch mode (rois (B, n, 5); returns two lists)."""
        _need_cuda(rois, 'Shared2FCBBoxHead.get_bboxes')
        if bbox_pred is None or cls_score is None or img_shape is None:
            raise NotImplementedError('get_bboxes without cls_score / bbox_pred / img_shape')
        batch_mode = rois.dim() == 3
        if rois.dim() == 2:
            rois, cls_score, bbox_pred = rois[None], cls_score[None], bbox_pred[None]
            img_shape, scale_factor = [img_shape], (scale_factor,)
        elif rois.dim() != 3:
            raise NotImplementedError(f'Unexpect shape of roi {tuple(rois.shape)}')
        B, n = rois.shape[:2]
        cfg = CfgNode(cfg) if cfg is not None else None
        res = self._decode_nms(rois.float().reshape(B * n, 5).contiguous(), n, cls_score.float().reshape(B * n, -1),
                               bbox_pred.float().reshape(B * n, -1), img_shape, scale_factor, rescale, cfg, mask_padding=False)
        dets, labels = _finish(res, B)
        return (dets, labels) if batch_mode else (dets[0], labels[0])


def _finish(res, B):
    if len(res) == 2:
        return res
    cnt, det, lab, max_per_img = res
    k = cnt.cpu().tolist()                              # the one device-to-host copy of the batch
    if max_per_img <= 0 and max(k) >= 1024:
        raise NotImplementedError('max_per_img=-1: more than 1023 detections survive the NMS (kernel limit 1024)')
    return [det[b, :k[b]] for b in range(B)], [lab[b, :k[b]].long() for b in range(B)]


class StandardRoIHead(PackedWeightsMixin, nn.Module):
    """standard_roi_head.py (test path) with the bbox branch only."""

    def __init__(self, bbox_roi_extractor=None, bbox_head=None, mask_roi_extractor=None, mask_head=None, shared_head=None, train_cfg=None,
                 test_cfg=None, pretrained=None, init_cfg=None):
        super().__init__()
        if mask_head is not None or mask_roi_extractor is not None or shared_head is not None:
            raise NotImplementedError('StandardRoIHead: mask heads and shared heads are not implemented')
        if bbox_head is None:
            raise NotImplementedError('StandardRoIHead: a bbox head is required')
        from .registry import build_head, build_roi_extractor
        self.bbox_roi_extractor = build_roi_extractor(bbox_roi_extractor) if isinstance(bbox_roi_extractor, dict) else bbox_roi_extractor
        self.bbox_head = build_head(bbox_head) if isinstance(bbox_head, dict) else bbox_head
        self.train_cfg = train_cfg
        self.test_cfg = CfgNode(test_cfg) if test_cfg is not None else None
        self._init_packed_hooks()

    with_bbox = property(lambda self: True)
    with_mask = property(lambda self: False)
    with_shared_head = property(lambda self: False)

    def forward_train(self, *a, **k):
        raise NotImplementedError('StandardRoIHead: the R-CNN training path is not implemented')

    def _bbox_forward(self, x, rois):
        """standard_roi_head.py:116-127: dict(cls_score, bbox_pred, bbox_feats) — bbox_feats is the fp16 operand pair (h, l, 1/scale)."""
        M = rois.shape[0]
        pair = self.bbox_roi_extractor.forward_f16_pair(x[:self.bbox_roi_extractor.num_inputs], rois)
        cls, reg = self.bbox_head._split_out(self.bbox_head._forward_pair(*pair), M)
        return dict(cls_score=cls, bbox_pred=reg, bbox_feats=pair)

    @torch.no_grad()
    def simple_test_bboxes(self, x, img_metas, proposals, rcnn_test_cfg, rescale=False):
        """test_mixins.py:50-155 for the whole batch: (list of (k, 5) dets, list of (k,) labels)."""
        for p in proposals:
            _need_cuda(p, 'StandardRoIHead')
        img_shapes = tuple(m['img_shape'] for m in img_metas)
        scale_factors = tuple(m['scale_factor'] for m in img_metas)
        B = len(proposals)
        n = max(p.size(0) for p in proposals)
        dev = proposals[0].device
        for i, p in enumerate(proposals):           # the reference pads the caller's list in place, zero rows first
            proposals[i] = torch.cat((p.new_zeros((n - p.size(0), p.size(1))), p), dim=0)
        rois = torch.zeros((B, n, 5), dtype=torch.float32, device=dev)
        rois[..., 0] = torch.arange(B, device=dev, dtype=torch.float32)[:, None]
        if n:
            rois[..., 1:] = torch.stack(proposals)[..., :4]
        rois = rois.view(B * n, 5)
        cfg = CfgNode(rcnn_test_cfg) if rcnn_test_cfg is not None else None
        if cfg is not None and n * self.bbox_head.num_classes > 4096:
            raise NotImplementedError(f'R-CNN test: {n} RoIs x {self.bbox_head.num_classes} classes > 4096 NMS candidates per image')
        if n == 0:
            cls = reg = rois.new_zeros((0, 5 * self.bbox_head.num_classes + 1))
        else:
            r = self._bbox_forward(x, rois)
            cls, reg = r['cls_score'], r['bbox_pred']
        res = self.bbox_head._decode_nms(rois, n, cls, reg, img_shapes, scale_factors, rescale, cfg, mask_padding=True)
        return _finish(res, B)

    def simple_test(self, x, proposal_list, img_metas, proposals=None, rescale=False):
        from .results import bbox2result
        det_bboxes, det_labels = self.simple_test_bboxes(x, img_metas, proposal_list, self.test_cfg, rescale=rescale)
        return [bbox2result(det_bboxes[i], det_labels[i], self.bbox_head.num_classes) for i in range(len(det_bboxes))]

    def aug_test(self, *a, **k):
        raise NotImplementedError('StandardRoIHead: test-time augmentation is not implemented')
