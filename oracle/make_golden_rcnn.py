"""Golden fixture of the R-CNN box stage (BASELINE.json config 4): runs the REAL reference SingleRoIExtractor, Shared2FCBBoxHead and
StandardRoIHead.simple_test_bboxes (TOV_mmdetection, mmcv stubbed by oracle/_mmcv_stub.py plus a RoIAlign wrapping
torchvision.ops.roi_align) on seeded inputs, asserts oracle/roi.py == reference and writes

  tests/golden/rcnn_box_stage.npz        detections, labels, levels and sampled features / logits per case
  tests/golden/rcnn_api_signatures.json  parameter names of the three classes' public methods and their state_dict shapes

Kept apart from make_golden.py so that regenerating it leaves every other fixture untouched:  python -m oracle.make_golden_rcnn
"""
import inspect
import json
import os
import sys

import numpy as np
import torch
import torch.nn as nn

from oracle import roi as orr
from oracle._mmcv_stub import install

GOLD = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden')


class AttrDict(dict):
    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError:
            raise AttributeError(k)


def wrap(x):
    if isinstance(x, dict):
        return AttrDict({k: wrap(v) for k, v in x.items()})
    return x


class RoIAlign(nn.Module):
    """mmcv.ops.RoIAlign (avg pooling) on torchvision.ops.roi_align: the same published kernel."""

    def __init__(self, output_size, spatial_scale=1.0, sampling_ratio=0, pool_mode='avg', aligned=True, use_torchvision=False):
        super().__init__()
        assert pool_mode == 'avg'
        self.output_size = (output_size, output_size) if np.isscalar(output_size) else tuple(output_size)
        self.spatial_scale, self.sampling_ratio, self.aligned = float(spatial_scale), int(sampling_ratio), aligned

    def forward(self, x, rois):
        import torchvision
        return torchvision.ops.roi_align(x, rois, self.output_size, self.spatial_scale, self.sampling_ratio, self.aligned)


def load():
    install()
    from oracle._mmcv_stub import Registry
    Registry.__contains__ = lambda self, key: self.get(key) is not None      # mmdet's build_linear_layer tests membership
    import mmcv.ops
    mmcv.ops.RoIAlign = RoIAlign
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        import mmdet.models  # noqa: F401
        from mmdet.models.roi_heads import StandardRoIHead
        from mmdet.models.roi_heads.bbox_heads import Shared2FCBBoxHead
        from mmdet.models.roi_heads.roi_extractors import SingleRoIExtractor
    return SingleRoIExtractor, Shared2FCBBoxHead, StandardRoIHead


def eq(a, b, what, tol=0.0):
    a, b = torch.as_tensor(a).float(), torch.as_tensor(b).float()
    assert a.shape == b.shape, f'{what}: shape {tuple(a.shape)} vs {tuple(b.shape)}'
    d = (a - b).abs().max().item() if a.numel() else 0.0
    assert d <= tol * max(1.0, b.abs().max().item() if b.numel() else 0.0), f'{what}: max diff {d}'


def main():
    torch.set_num_threads(os.cpu_count())
    SRE, S2FC, SRH = load()
    out = {}
    for case in orr.GOLDEN_CASES:
        name = case['name']
        inp = orr.synth_rcnn_inputs(**case)
        cfg = orr.roi_head_cfg(inp['C'])
        head = SRH(bbox_roi_extractor=cfg['bbox_roi_extractor'], bbox_head=cfg['bbox_head'], test_cfg=wrap(cfg['test_cfg']))
        sd = head.state_dict()
        sd.update({f'bbox_head.{k}': v for k, v in inp['weights'].items()})
        head.load_state_dict(sd)
        rois = torch.cat([torch.full((p.shape[0], 1), float(i)) for i, p in enumerate(inp['proposals'])]
                         + [torch.zeros(0, 1)], 0)
        rois = torch.cat([rois, torch.cat(inp['proposals'])[:, :4]], 1)
        with torch.no_grad():
            lv_ref = head.bbox_roi_extractor.map_roi_levels(rois, len(inp['feats']))
            eq(orr.map_roi_levels(rois, len(inp['feats'])), lv_ref, f'{name} levels')
            feats_ref = head.bbox_roi_extractor(inp['feats'], rois)
            feats_or = orr.roi_extract(inp['feats'], rois, inp['strides'])
            eq(feats_or, feats_ref, f'{name} roi feats')
            cls_ref, reg_ref = head.bbox_head(feats_ref)
            cls_or, reg_or = orr.bbox_head_forward(feats_ref, inp['weights'])
            eq(cls_or, cls_ref, f'{name} cls'); eq(reg_or, reg_ref, f'{name} reg')
            for rescale in (False, True):
                props = [p.clone() for p in inp['proposals']]
                dets, labels = head.simple_test_bboxes(inp['feats'], inp['img_metas'], props, wrap(cfg['test_cfg']['rcnn']), rescale=rescale)
                od, ol = orr.simple_test_bboxes(inp['feats'], inp['proposals'], inp['img_metas'], inp['weights'], cfg['test_cfg']['rcnn'],
                                                inp['strides'], orr.MEANS, orr.STDS, rescale=rescale)
                tag = f'{name}_r{int(rescale)}'
                for b in range(len(dets)):
                    eq(od[b], dets[b], f'{tag} dets {b}', 1e-6)
                    assert torch.equal(ol[b], labels[b]), f'{tag} labels {b}'
                    out[f'{tag}_dets{b}'] = dets[b].numpy().astype(np.float32)
                    out[f'{tag}_labels{b}'] = labels[b].numpy().astype(np.int16)
                s = dets[0][:, 4]
                print(f'[golden] {tag}: {[int(d.shape[0]) for d in dets]} dets, scores {s.min().item() if s.numel() else 0:.3f}'
                      f'..{s.max().item() if s.numel() else 0:.3f}')
        out[f'{name}_levels'] = lv_ref.numpy().astype(np.int8)
        out[f'{name}_feats_sub'] = feats_ref.reshape(-1)[::97].numpy()
        out[f'{name}_cls'] = cls_ref.numpy()
        out[f'{name}_reg'] = reg_ref.numpy()
    path = os.path.join(GOLD, 'rcnn_box_stage.npz')
    np.savez_compressed(path, **out)
    print(f'[golden] {path}: {os.path.getsize(path) / 1024:.0f} KiB')

    def names(f):
        return [p.name for p in inspect.signature(f).parameters.values()
                if p.name != 'self' and p.kind not in (p.VAR_KEYWORD, p.VAR_POSITIONAL)]
    sig = {}
    for cls, meths in [(SRE, ['__init__', 'map_roi_levels', 'forward']), (S2FC, ['__init__', 'forward', 'get_bboxes']),
                       (SRH, ['__init__', 'simple_test_bboxes', 'simple_test'])]:
        for m in meths:
            sig[f'{cls.__name__}.{m}'] = names(getattr(cls, m))
    sig['Shared2FCBBoxHead.__init__'] = names(S2FC.__init__) + [n for n in names(S2FC.__mro__[2].__init__) if n not in names(S2FC.__init__)]
    cfg = orr.roi_head_cfg(256)
    head = SRH(bbox_roi_extractor=cfg['bbox_roi_extractor'], bbox_head=cfg['bbox_head'], test_cfg=wrap(cfg['test_cfg']))
    sig['state_dict:StandardRoIHead'] = {k: list(v.shape) for k, v in head.state_dict().items()}
    path = os.path.join(GOLD, 'rcnn_api_signatures.json')
    json.dump(sig, open(path, 'w'), indent=1, sort_keys=True)
    print(f'[golden] {path}: {len(sig)} entries')


if __name__ == '__main__':
    sys.exit(main())
