"""CPU checks of the R-CNN box stage's oracle (oracle/roi.py) and of the mirror classes' surface (pointtinybenchmark_b200/roi_head.py):
RoIAlign vs torchvision, level mapping at the ulp edges, oracle vs the reference's golden detections, signatures and state_dict keys."""
import inspect
import json
import os

import numpy as np
import pytest
import torch
import torchvision

from oracle import roi as orr

GOLD = os.path.join(os.path.dirname(__file__), 'golden')


def edge_rois(seed=0, n=80, B=2, extent=(100, 120)):
    g = torch.Generator().manual_seed(seed)
    xy = torch.rand(n, 2, generator=g) * torch.tensor([extent[1] + 40., extent[0] + 40.]) - 20
    wh = torch.rand(n, 2, generator=g) * 60
    r = torch.cat([torch.randint(0, B, (n, 1), generator=g).float(), xy, xy + wh], 1)
    r[0, 1:] = 0                                               # the padding row of simple_test_bboxes
    r[1, 3:] = r[1, 1:3]                                       # zero-size
    r[2, 1:] = torch.tensor([extent[1] + 50., extent[0] + 50., extent[1] + 90., extent[0] + 70.])   # outside the map
    r[3, 1:] = torch.tensor([-30., -25., 10., 12.])            # straddling the top-left corner
    r[4, 1:] = torch.tensor([40., 40., 40.3, 40.2])            # tiny
    return r


@pytest.mark.parametrize('aligned', [True, False])
@pytest.mark.parametrize('sr', [0, 2])
def test_oracle_roi_align_matches_torchvision(aligned, sr):
    g = torch.Generator().manual_seed(1)
    f = torch.randn(2, 32, 25, 30, generator=g)
    rois = edge_rois()
    for scale in (0.25, 0.125):
        a = orr.roi_align(f, rois, (7, 7), scale, sr, aligned)
        b = torchvision.ops.roi_align(f, rois, (7, 7), scale, sr, aligned)
        assert torch.equal(a, b)
    if sr == 0 and aligned:                                    # zero-size RoIs have grid 0: zeros (the padding rows rely on it)
        assert torch.equal(orr.roi_align(f, rois[:2], (7, 7), 0.25, sr, aligned), torch.zeros(2, 32, 7, 7))


def test_oracle_roi_extract_one_level():
    g = torch.Generator().manual_seed(2)
    f = torch.randn(2, 32, 25, 30, generator=g)
    rois = edge_rois(3)
    assert torch.equal(orr.roi_extract([f], rois, [4]), torchvision.ops.roi_align(f, rois, (7, 7), 0.25, 0, True))


def planted_level_rois(finest=56):
    """square RoIs whose scale / 56 + 1e-6 lands within a few ulp of 2, 4 and 8 (searched with fp32 torch arithmetic)."""
    out = []
    for t in (2.0, 4.0, 8.0):
        s0 = torch.tensor(finest * (t - 1e-6), dtype=torch.float32)
        side = s0 * (1 + torch.arange(-400, 401, dtype=torch.float32) * 2.0 ** -24)
        v = torch.sqrt(side * side) / finest + 1e-6
        near = (v - t).abs() <= 8 * torch.finfo(torch.float32).eps * t
        out.append(side[near])
    side = torch.cat(out)
    z = torch.zeros_like(side)
    return torch.stack([z, z + 3, z + 5, side + 3, side + 5], 1)


def test_planted_levels_cross_the_boundary():
    rois = planted_level_rois()
    assert rois.shape[0] > 30
    lv = orr.map_roi_levels(rois, 5)
    v = torch.sqrt((rois[:, 3] - rois[:, 1]) * (rois[:, 4] - rois[:, 2])) / 56 + 1e-6
    assert set(lv.tolist()) >= {0, 1, 2, 3}
    assert bool(((v < 2) & (lv == 1)).any() or ((v >= 2) & (lv == 1)).any())


def test_oracle_matches_golden():
    gold = np.load(os.path.join(GOLD, 'rcnn_box_stage.npz'))
    for case in orr.GOLDEN_CASES:
        inp = orr.synth_rcnn_inputs(**case)
        cfg = orr.roi_head_cfg(inp['C'])['test_cfg']['rcnn']
        dets, labels = orr.simple_test_bboxes(inp['feats'], inp['proposals'], inp['img_metas'], inp['weights'], cfg, inp['strides'],
                                              orr.MEANS, orr.STDS, rescale=True)
        for b in range(len(dets)):
            np.testing.assert_allclose(dets[b].numpy(), gold[f"{case['name']}_r1_dets{b}"], rtol=0, atol=1e-5)
            assert np.array_equal(labels[b].numpy(), gold[f"{case['name']}_r1_labels{b}"])
        rois = torch.cat([torch.cat([torch.full((p.shape[0], 1), float(i)), p[:, :4]], 1) for i, p in enumerate(inp['proposals'])])
        assert np.array_equal(orr.map_roi_levels(rois, 4).numpy(), gold[f"{case['name']}_levels"])


def test_signatures_and_state_dict_keys():
    from pointtinybenchmark_b200 import roi_head as rh
    sig = json.load(open(os.path.join(GOLD, 'rcnn_api_signatures.json')))

    def names(f):
        return [p.name for p in inspect.signature(f).parameters.values()
                if p.name != 'self' and p.kind not in (p.VAR_KEYWORD, p.VAR_POSITIONAL)]
    for key, ref in sig.items():
        if key.startswith('state_dict:'):
            continue
        cls, meth = key.split('.')
        mine = names(getattr(getattr(rh, cls), meth))
        assert [n for n in mine if n in ref] == [n for n in ref if n in mine] and set(ref) <= set(mine), (key, ref, mine)
    cfg = orr.roi_head_cfg(256)
    head = rh.StandardRoIHead(bbox_roi_extractor=rh.SingleRoIExtractor(**{k: v for k, v in cfg['bbox_roi_extractor'].items() if k != 'type'}),
                              bbox_head=rh.Shared2FCBBoxHead(**{k: v for k, v in cfg['bbox_head'].items() if k != 'type'}),
                              test_cfg=cfg['test_cfg'])
    assert {k: list(v.shape) for k, v in head.state_dict().items()} == sig['state_dict:StandardRoIHead']


def test_registry_builds_the_shipped_config():
    from pointtinybenchmark_b200 import registry
    registry.register_roi_heads()
    cfg = orr.roi_head_cfg(256)
    head = registry.build_head(dict(type='StandardRoIHead', **cfg))
    assert type(head.bbox_head).__name__ == 'Shared2FCBBoxHead' and type(head.bbox_roi_extractor).__name__ == 'SingleRoIExtractor'
    with pytest.raises(NotImplementedError):
        registry.build_head(dict(type='StandardRoIHead', mask_head=dict(type='FCNMaskHead'), **cfg))
    with pytest.raises(NotImplementedError):
        registry.build_roi_extractor(dict(cfg['bbox_roi_extractor'], roi_layer=dict(type='RoIAlign', output_size=7, pool_mode='max')))
