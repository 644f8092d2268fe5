"""HEADS registry: the drop-in boundary of this package (SURVEY.md §8b).

If mmdet is importable, CPRHead/P2PHead register into mmdet's own `HEADS` (= MODELS) registry with `force=True`, so a
reference config (`bbox_head=dict(type='CPRHead', ...)`) builds this implementation unchanged.  Otherwise a minimal
registry with the same `register_module` / `build` surface is used (mmcv/mmdet cannot be installed offline here).
"""


class Registry:
    def __init__(self, name):
        self.name = name
        self.module_dict = {}

    def register_module(self, name=None, force=False, module=None):
        def _reg(cls):
            key = name or cls.__name__
            if key in self.module_dict and not force:
                raise KeyError(f'{key} is already registered in {self.name}')
            self.module_dict[key] = cls
            return cls
        return _reg(module) if module is not None else _reg

    def get(self, key):
        return self.module_dict.get(key)

    def build(self, cfg, default_args=None):
        args = dict(cfg)
        for k, v in (default_args or {}).items():
            args.setdefault(k, v)
        t = args.pop('type')
        cls = self.get(t) if isinstance(t, str) else t
        if cls is None:
            raise KeyError(f'{t} is not in the {self.name} registry')
        return cls(**args)


try:   # pragma: no cover - mmdet is not installable in the offline build container
    from mmdet.models.builder import HEADS as _MMDET_HEADS
    HEADS = _MMDET_HEADS
    USING_MMDET = True
except Exception:
    HEADS = Registry('head')
    USING_MMDET = False


def register_head(cls):
    HEADS.register_module(name=cls.__name__, force=True, module=cls)
    return cls


def build_head(cfg, default_args=None):
    return HEADS.build(cfg, default_args)


class CfgNode(dict):
    """attribute-style dict (stand-in for mmcv.Config nodes in train_cfg / test_cfg)."""
    __getattr__ = dict.get


# ---- assigners / samplers / anchor generators (mmdet/core/bbox/builder.py:4-6, mmdet/core/anchor/builder.py:3): same pattern
try:   # pragma: no cover
    from mmdet.core.bbox.builder import BBOX_ASSIGNERS as _A, BBOX_SAMPLERS as _S
    from mmdet.core.anchor.builder import ANCHOR_GENERATORS as _G
    BBOX_ASSIGNERS, BBOX_SAMPLERS, ANCHOR_GENERATORS = _A, _S, _G
except Exception:
    BBOX_ASSIGNERS, BBOX_SAMPLERS, ANCHOR_GENERATORS = Registry('bbox_assigner'), Registry('bbox_sampler'), Registry('Anchor generator')


def register_core():
    """register the assigner / sampler / anchor-generator mirrors (force=True over the reference classes when mmdet is importable)."""
    from .assigners import HungarianAssignerV2, MaxIoUAssigner, PointAssigner, PseudoSampler
    from .rpn import AnchorGenerator
    for c in (HungarianAssignerV2, MaxIoUAssigner, PointAssigner):
        BBOX_ASSIGNERS.register_module(name=c.__name__, force=True, module=c)
    BBOX_SAMPLERS.register_module(name='PseudoSampler', force=True, module=PseudoSampler)
    ANCHOR_GENERATORS.register_module(name='AnchorGenerator', force=True, module=AnchorGenerator)


def build_assigner(cfg, **default_args):
    return BBOX_ASSIGNERS.build(cfg, default_args)


def build_sampler(cfg, **default_args):
    return BBOX_SAMPLERS.build(cfg, default_args)


def build_anchor_generator(cfg, default_args=None):
    return ANCHOR_GENERATORS.build(cfg, default_args)


# ---- R-CNN box stage (roi_head.py): RoI extractors have their own registry in mmdet (mmdet/models/builder.py)
try:   # pragma: no cover
    from mmdet.models.builder import ROI_EXTRACTORS as _R
    ROI_EXTRACTORS = _R
except Exception:
    ROI_EXTRACTORS = Registry('roi_extractor')


def register_roi_heads():
    """register SingleRoIExtractor into ROI_EXTRACTORS and Shared2FCBBoxHead / StandardRoIHead into HEADS (force=True over the reference
    classes when mmdet is importable)."""
    from .roi_head import Shared2FCBBoxHead, SingleRoIExtractor, StandardRoIHead
    ROI_EXTRACTORS.register_module(name='SingleRoIExtractor', force=True, module=SingleRoIExtractor)
    for c in (Shared2FCBBoxHead, StandardRoIHead):
        HEADS.register_module(name=c.__name__, force=True, module=c)


def build_roi_extractor(cfg, default_args=None):
    return ROI_EXTRACTORS.build(cfg, default_args)
