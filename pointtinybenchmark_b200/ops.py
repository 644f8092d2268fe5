"""Thin torch-tensor wrappers over the C ABI (include/ptb_b200.h).  Device memory, streams and autograd plumbing
only — all math happens in libptb_b200.so.  Every op raises if the library is missing or a tensor is not on CUDA.
"""
import ctypes
import math

import torch

from . import _lib
from ._lib import RefineCfg, check


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _chk(t, dtype, name):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f'{name}: expected a CUDA tensor (pointtinybenchmark_b200 has no CPU path)')
    if t.dtype != dtype:
        raise TypeError(f'{name}: expected {dtype}, got {t.dtype}')
    if not t.is_contiguous():
        raise ValueError(f'{name}: must be contiguous')
    return t


def to_nhwc(x):
    """(B,C,H,W) tensor -> contiguous (B,H,W,C) view (no copy when x is already channels_last)."""
    if x.dim() != 4:
        raise ValueError('expected (B,C,H,W)')
    return x.contiguous(memory_format=torch.channels_last).permute(0, 2, 3, 1)


def circle_offsets(radius, stride, start_angle=0, base_num_point=8, same_num_all_radius=False, append_center=True):
    """Bag offset table, computed once on the host with the reference's exact torch-CPU op sequence
    (cpr_head.py:484-497) so the sample coordinates are bit-identical.  (K,2) fp32 CPU tensor, centre LAST."""
    out = []
    for i in range(radius):
        r = (i + 1) * stride
        m = base_num_point if same_num_all_radius else base_num_point * (i + 1)
        ang = torch.arange(m).float() / m * 360 + start_angle
        ang = ang / 360 * math.pi * 2
        out.append(torch.stack([r * torch.cos(ang), r * torch.sin(ang)], dim=-1))
    off = torch.cat(out) if out else torch.zeros(0, 2)
    if append_center:
        off = torch.cat([off, torch.zeros(1, 2)])
    return off.float().contiguous()


# ----------------------------------------------------------------------------------------------------------------------
def bag_gather(map_nhwc, centers, bag_img, offsets, stride, pad_hw, feats=True, pts=True, valid=True, C=None):
    """ptb_cpr_bag_gather. map_nhwc (B,H,W,ld) fp32; centers (G,2); bag_img (G,) int32; offsets (K,2); pad_hw (B,2) int32.
    returns (feats (G,K,C) | None, pts (G,K,3) | None, valid (G,K) bool | None)."""
    lib = _lib.load()
    _chk(map_nhwc, torch.float32, 'map'); _chk(centers, torch.float32, 'centers'); _chk(bag_img, torch.int32, 'bag_img')
    _chk(offsets, torch.float32, 'offsets'); _chk(pad_hw, torch.int32, 'pad_hw')
    B, H, W, ld = map_nhwc.shape
    C = ld if C is None else C
    G, K = centers.shape[0], offsets.shape[0]
    dev = map_nhwc.device
    o_f = torch.empty((G, K, C), dtype=torch.float32, device=dev) if feats else None
    o_p = torch.empty((G, K, 3), dtype=torch.float32, device=dev) if pts else None
    o_v = torch.empty((G, K), dtype=torch.uint8, device=dev) if valid else None
    check(lib.ptb_cpr_bag_gather(_ptr(map_nhwc), B, H, W, C, ld, _ptr(centers), _ptr(bag_img), G, _ptr(offsets), K,
                                 float(stride), float(offsets_reach(offsets)) if feats else 0.0, _ptr(pad_hw), _ptr(o_f), _ptr(o_p), _ptr(o_v),
                                 _stream()),
          'ptb_cpr_bag_gather')
    return o_f, o_p, (o_v.bool() if o_v is not None else None)


def bag_gather_bwd(grad_out, map_shape, centers, bag_img, offsets, stride):
    lib = _lib.load()
    _chk(grad_out, torch.float32, 'grad_out')
    B, H, W, ld = map_shape
    G, K, C = grad_out.shape
    gm = torch.zeros(map_shape, dtype=torch.float32, device=grad_out.device)
    check(lib.ptb_cpr_bag_gather_bwd(_ptr(grad_out), B, H, W, C, ld, _ptr(centers), _ptr(bag_img), G, _ptr(offsets), K,
                                     float(stride), _ptr(gm), _stream()), 'ptb_cpr_bag_gather_bwd')
    return gm


def grid_circles_max_pos_num(radius, max_pos_num=-1):
    """GridCirclesPtFeatGenerator.get_max_pos_num (cpr_head.py:440-444)."""
    return 2 * (2 * radius) ** 2 if max_pos_num <= 0 else max_pos_num


def grid_bag(map_nhwc, centers, bag_img, stride, radius, max_pos_num=-1, feats=True, pts=True, valid=True, cell=True, C=None,
             check_overflow=True):
    """ptb_cpr_grid_bag: grid-cell bags of GridCirclesPtFeatGenerator (cpr_head.py:296-350, 418-444).
    returns (feats (G,Kt,C) | None, pts (G,Kt,3) | None, valid (G,Kt) bool | None, cell (G,Kt) int32 | None), Kt = max_pos_num + 2."""
    lib = _lib.load()
    _chk(map_nhwc, torch.float32, 'map'); _chk(centers, torch.float32, 'centers'); _chk(bag_img, torch.int32, 'bag_img')
    mp = grid_circles_max_pos_num(radius, max_pos_num)
    if not isinstance(mp, int):
        # the reference passes this straight to torch.zeros(n, max_pos_num + R, ...) which rejects floats
        raise TypeError(f'max_pos_num must be an int, got {mp!r} (use an int radius or set max_pos_num)')
    B, H, W, ld = map_nhwc.shape
    C = ld if C is None else C
    G = centers.shape[0]
    Kt = mp + 2
    dev = map_nhwc.device
    o_f = torch.empty((G, Kt, C), dtype=torch.float32, device=dev) if feats else None
    o_p = torch.empty((G, Kt, 3), dtype=torch.float32, device=dev) if pts else None
    o_v = torch.empty((G, Kt), dtype=torch.uint8, device=dev) if valid else None
    o_c = torch.empty((G, Kt), dtype=torch.int32, device=dev) if cell else None
    ovf = torch.zeros(1, dtype=torch.int32, device=dev)
    radius_px = float(torch.tensor(radius * stride, dtype=torch.float32))      # the comparison scalar is cast to fp32
    check(lib.ptb_cpr_grid_bag(_ptr(map_nhwc), B, H, W, C, ld, _ptr(centers), _ptr(bag_img), G, float(stride), radius_px, mp,
                               _ptr(o_f), _ptr(o_p), _ptr(o_v), _ptr(o_c), _ptr(ovf), _stream()), 'ptb_cpr_grid_bag')
    if check_overflow and int(ovf.item()):
        raise RuntimeError(f'GridCirclesPtFeatGenerator: a GT has more than max_pos_num + num_refine = {mp + 1} cells within '
                           f'radius {radius}*{stride}; the reference fails here too (cpr_head.py:334)')
    return o_f, o_p, (o_v.bool() if valid else None), o_c


def grid_bag_bwd(grad_out, map_shape, centers, bag_img, cell, stride):
    lib = _lib.load()
    _chk(grad_out, torch.float32, 'grad_out'); _chk(cell, torch.int32, 'cell')
    B, H, W, ld = map_shape
    G, Kt, C = grad_out.shape
    gm = torch.zeros(map_shape, dtype=torch.float32, device=grad_out.device)
    check(lib.ptb_cpr_grid_bag_bwd(_ptr(grad_out), B, H, W, C, ld, _ptr(centers), _ptr(bag_img), _ptr(cell), G, Kt, float(stride),
                                   _ptr(gm), _stream()), 'ptb_cpr_grid_bag_bwd')
    return gm


def linear_rows(x2d, weight, bias=None, out=None):
    """y = x2d @ weight.T + bias with the library's fp32 FFMA GEMM. x2d (M,Cin) view with row stride ldx."""
    lib = _lib.load()
    if x2d.dim() != 2 or x2d.stride(1) != 1:
        raise ValueError('x2d must be 2-D with unit inner stride')
    if x2d.dtype != torch.float32 or not x2d.is_cuda:
        raise RuntimeError('x2d: expected a CUDA fp32 tensor')
    _chk(weight, torch.float32, 'weight')
    M, Cin = x2d.shape
    N = weight.shape[0]
    if out is None:
        out = torch.empty((M, N), dtype=torch.float32, device=x2d.device)
    ldx = x2d.stride(0) if M > 1 else Cin
    check(lib.ptb_linear_rows(_ptr(x2d), M, Cin, ldx, _ptr(weight), _ptr(bias), N, _ptr(out), out.stride(0), _stream()),
          'ptb_linear_rows')
    return out


def linear_rows_bwd_x(dy, weight, accumulate_into=None):
    lib = _lib.load()
    _chk(dy, torch.float32, 'dy'); _chk(weight, torch.float32, 'weight')
    M, N = dy.shape
    Cin = weight.shape[1]
    dx = accumulate_into if accumulate_into is not None else torch.empty((M, Cin), dtype=torch.float32, device=dy.device)
    check(lib.ptb_linear_rows_bwd_x(_ptr(dy), M, N, dy.stride(0), _ptr(weight), Cin, _ptr(dx), dx.stride(0),
                                    1 if accumulate_into is not None else 0, _stream()), 'ptb_linear_rows_bwd_x')
    return dx


def linear_rows_bwd_w(dy, x2d):
    lib = _lib.load()
    _chk(dy, torch.float32, 'dy')
    M, N = dy.shape
    Cin = x2d.shape[1]
    ldx = x2d.stride(0) if M > 1 else Cin
    nbytes = lib.ptb_linear_rows_bwd_w_workspace(M, N, Cin)
    ws = torch.empty(nbytes // 4, dtype=torch.float32, device=dy.device)
    dw = torch.empty((N, Cin), dtype=torch.float32, device=dy.device)
    db = torch.empty((N,), dtype=torch.float32, device=dy.device)
    check(lib.ptb_linear_rows_bwd_w(_ptr(dy), M, N, dy.stride(0), _ptr(x2d), Cin, ldx, _ptr(dw), _ptr(db), _ptr(ws),
                                    nbytes, _stream()), 'ptb_linear_rows_bwd_w')
    return dw, db


def neg_mask(B, H, W, stride, pad_hw, centers, labels, img_ptr, thresh, num_classes, class_wise=True, as_bool=True):
    """ptb_cpr_neg_mask -> bool (or uint8 0/1) (B,H,W,num_classes)."""
    lib = _lib.load()
    _chk(pad_hw, torch.int32, 'pad_hw'); _chk(centers, torch.float32, 'centers'); _chk(labels, torch.int32, 'labels')
    _chk(img_ptr, torch.int32, 'img_ptr')
    out = torch.empty((B, H, W, num_classes), dtype=torch.uint8, device=centers.device)
    check(lib.ptb_cpr_neg_mask(B, H, W, float(stride), _ptr(pad_hw), _ptr(centers), _ptr(labels), _ptr(img_ptr),
                               centers.shape[0], float(thresh), num_classes, 1 if class_wise else 0, _ptr(out), _stream()),
          'ptb_cpr_neg_mask')
    return out.bool() if as_bool else out


def label_groups(bag_img, labels, num_classes):
    """CSR of same-(image,label) GT groups, built on the device without a host sync (replaces group_by_label,
    cpr_head.py:64-70, which forces labels.cpu()).  returns grp_of (G,), grp_ptr (G+1,), grp_idx (G,) int32."""
    G = labels.shape[0]
    key = bag_img.long() * num_classes + labels.long()
    order = torch.argsort(key, stable=True)
    ks = key[order]
    change = torch.ones(G, dtype=torch.long, device=key.device)
    if G > 1:
        change[1:] = (ks[1:] != ks[:-1]).long()
    gid = torch.cumsum(change, 0) - 1
    pos = torch.arange(G, device=key.device)
    grp_ptr = torch.full((G + 1,), G, dtype=torch.long, device=key.device)
    grp_ptr.scatter_reduce_(0, gid, pos, reduce='amin', include_self=True)
    grp_of = torch.empty(G, dtype=torch.long, device=key.device)
    grp_of[order] = gid
    return grp_of.int().contiguous(), grp_ptr.int().contiguous(), order.int().contiguous()


def label_groups_csr(labels, img_ptr, num_classes, max_per_image):
    """ptb_label_groups: same result as label_groups() (tested against it) in one ~10 us launch instead of a torch sort + scans."""
    lib = _lib.load()
    _chk(labels, torch.int32, 'labels'); _chk(img_ptr, torch.int32, 'img_ptr')
    G = labels.shape[0]
    dev = labels.device
    grp_of = torch.empty(G, dtype=torch.int32, device=dev)
    grp_ptr = torch.empty(G + 1, dtype=torch.int32, device=dev)
    grp_idx = torch.empty(G, dtype=torch.int32, device=dev)
    check(lib.ptb_label_groups(_ptr(labels), _ptr(img_ptr), img_ptr.shape[0] - 1, G, int(num_classes), int(max_per_image),
                               _ptr(grp_of), _ptr(grp_ptr), _ptr(grp_idx), _stream()), 'ptb_label_groups')
    return grp_of, grp_ptr, grp_idx


def _refine_cfg(merge_th, gt_alpha, refine_th, nearest_filter, classify_filter, score_max):
    return RefineCfg(float(merge_th), float(gt_alpha), float(refine_th),
                     (1 if nearest_filter else 0) | (2 if classify_filter else 0) | (4 if score_max else 0))


def refine(bag_prob, bag_pts, bag_valid, K, labels, bag_img, img_hw, groups, cfg, not_refine=None, want_masks=True):
    """ptb_cpr_refine (stage form).  bag_prob (G,Kt,C), bag_pts (G,Kt,3), bag_valid (G,Kt) bool/uint8."""
    lib = _lib.load()
    _chk(bag_prob, torch.float32, 'bag_prob'); _chk(bag_pts, torch.float32, 'bag_pts')
    bv = bag_valid.to(torch.uint8).contiguous()
    G, Kt, C = bag_prob.shape
    dev = bag_prob.device
    grp_of, grp_ptr, grp_idx = groups
    o_pts = torch.empty((G, 2), dtype=torch.float32, device=dev)
    o_sc = torch.empty((G,), dtype=torch.float32, device=dev)
    o_nr = torch.empty((G,), dtype=torch.uint8, device=dev)
    o_ch = torch.empty((G, Kt), dtype=torch.uint8, device=dev) if want_masks else None
    o_mv = torch.empty((G, Kt), dtype=torch.uint8, device=dev) if want_masks else None
    nr_in = not_refine.to(torch.uint8).contiguous() if not_refine is not None else None
    check(lib.ptb_cpr_refine(_ptr(bag_prob), _ptr(bag_pts), _ptr(bv), G, Kt, K, C, _ptr(labels), _ptr(bag_img), _ptr(img_hw),
                             _ptr(grp_of), _ptr(grp_ptr), _ptr(grp_idx), _ptr(nr_in), cfg, _ptr(o_pts), _ptr(o_sc),
                             _ptr(o_nr), _ptr(o_ch), _ptr(o_mv), _stream()), 'ptb_cpr_refine')
    return o_pts, o_sc, o_nr.bool(), (o_ch.bool() if want_masks else None), (o_mv.bool() if want_masks else None)


_REACH_CACHE = {}


def offsets_reach(offsets):
    """max |offset| of a bag offset table in pixels (= radius * stride for ring bags): sizes the shared-memory window the fused refine
    kernel stages per GT.  Read back from the device ONCE per table (cached by storage), never on the steady-state path."""
    key = (offsets.data_ptr(), offsets.numel(), str(offsets.device))
    r = _REACH_CACHE.get(key)
    if r is None:
        r = float(offsets.detach().abs().max()) if offsets.numel() else 0.0
        if len(_REACH_CACHE) > 64:
            _REACH_CACHE.clear()
        _REACH_CACHE[key] = r
    return r


def refine_fused(logit_map, num_classes, centers, labels, bag_img, offsets, stride, pad_hw, img_hw, groups, cfg,
                 not_refine=None, want_chosen=False, reach_px=None):
    """ptb_cpr_refine_fused.  logit_map (B,H,W,ld) fp32 class logits (channels-last)."""
    lib = _lib.load()
    if reach_px is None:
        reach_px = offsets_reach(offsets)
    _chk(logit_map, torch.float32, 'logit_map'); _chk(centers, torch.float32, 'centers')
    _chk(labels, torch.int32, 'labels'); _chk(bag_img, torch.int32, 'bag_img'); _chk(offsets, torch.float32, 'offsets')
    B, H, W, ld = logit_map.shape
    G, K = centers.shape[0], offsets.shape[0]
    dev = logit_map.device
    grp_of, grp_ptr, grp_idx = groups
    o_pts = torch.empty((G, 2), dtype=torch.float32, device=dev)
    o_sc = torch.empty((G,), dtype=torch.float32, device=dev)
    o_nr = torch.empty((G,), dtype=torch.uint8, device=dev)
    o_ch = torch.empty((G, K), dtype=torch.uint8, device=dev) if want_chosen else None
    nr_in = not_refine.to(torch.uint8).contiguous() if not_refine is not None else None
    check(lib.ptb_cpr_refine_fused(_ptr(logit_map), B, H, W, num_classes, ld, _ptr(centers), _ptr(labels), _ptr(bag_img), G,
                                   _ptr(offsets), K, float(stride), float(reach_px), _ptr(pad_hw), _ptr(img_hw), _ptr(grp_of),
                                   _ptr(grp_ptr), _ptr(grp_idx), _ptr(nr_in), cfg, _ptr(o_pts), _ptr(o_sc), _ptr(o_nr), _ptr(o_ch),
                                   _stream()), 'ptb_cpr_refine_fused')
    return o_pts, o_sc, o_nr.bool(), (o_ch.bool() if want_chosen else None)


def launch_count():
    return int(_lib.load().ptb_launch_count())


# ----------------------------------------------------------------------------------------------------------------------
# losses
# ----------------------------------------------------------------------------------------------------------------------
def mil_loss_fwd(logits, num_classes, ins_off, weight, labels, eps, want_aux=False):
    """ptb_mil_loss_fwd.  logits (G,Kt,ld) [cls | ins]; weight (G,Kt) fp32; labels (G,) int32.
    returns bag_prob (G,C), loss_sum (1,), stats (2,) = [#bags with weight, #top-1 hits]."""
    lib = _lib.load()
    _chk(logits, torch.float32, 'logits'); _chk(weight, torch.float32, 'weight'); _chk(labels, torch.int32, 'labels')
    G, Kt, ld = logits.shape
    buf = torch.empty(G * num_classes + 3 * G, dtype=torch.float32, device=logits.device)
    loss = torch.zeros(1, dtype=torch.float32, device=logits.device)
    stats = torch.zeros(2, dtype=torch.float32, device=logits.device)
    mt = torch.empty((G, num_classes, 2), dtype=torch.float32, device=logits.device) if want_aux else None
    check(lib.ptb_mil_loss_fwd(_ptr(logits), G, Kt, num_classes, ld, ins_off, _ptr(weight), _ptr(labels), float(eps),
                               _ptr(buf), _ptr(loss), _ptr(stats), _ptr(mt), _stream()), 'ptb_mil_loss_fwd')
    bag_prob = buf[:G * num_classes].view(G, num_classes)
    if want_aux:         # (max ins, 1/T) per (bag, class) and the per-bag label weight: inputs of ptb_cpr_loss_bwd_map
        return bag_prob, loss, stats, mt, buf[G * num_classes + G:G * num_classes + 2 * G]
    return bag_prob, loss, stats


def bag_mil_fwd(lmap, num_classes, ins_off, centers, bag_img, offsets, stride, pad_hw, labels, eps):
    """ptb_cpr_bag_mil_fwd: fused ring-bag gather of the [cls | ins] logit map + MIL forward.
    returns bag_logits (G,K,ld), weight (G,K) fp32 0/1, bag_prob (G,N), loss_sum (1,), stats (2,), mt (G,N,2), label_weight (G,)."""
    lib = _lib.load()
    _chk(lmap, torch.float32, 'lmap'); _chk(centers, torch.float32, 'centers'); _chk(labels, torch.int32, 'labels')
    B, H, W, ld = lmap.shape
    G, K = centers.shape[0], offsets.shape[0]
    dev = lmap.device
    bl = torch.empty((G, K, ld), dtype=torch.float32, device=dev)
    if ld > ins_off + (num_classes + 3) // 4 * 4 or ins_off > (num_classes + 3) // 4 * 4:
        bl.zero_()                               # pad columns the kernel does not write
    weight = torch.empty((G, K), dtype=torch.float32, device=dev)
    buf = torch.empty(G * num_classes + 3 * G, dtype=torch.float32, device=dev)
    loss = torch.zeros(1, dtype=torch.float32, device=dev)
    stats = torch.zeros(2, dtype=torch.float32, device=dev)
    mt = torch.empty((G, num_classes, 2), dtype=torch.float32, device=dev)
    check(lib.ptb_cpr_bag_mil_fwd(_ptr(lmap), B, H, W, ld, num_classes, ins_off, _ptr(centers), _ptr(bag_img), G, _ptr(offsets), K, float(stride),
                                  _ptr(pad_hw), _ptr(labels), float(eps), _ptr(bl), _ptr(weight), _ptr(buf), _ptr(loss), _ptr(stats), _ptr(mt),
                                  _stream()), 'ptb_cpr_bag_mil_fwd')
    return (bl, weight, buf[:G * num_classes].view(G, num_classes), loss, stats, mt, buf[G * num_classes + G:G * num_classes + 2 * G])


def mil_loss_bwd(logits, num_classes, ins_off, weight, labels, eps, bag_prob, scale, grad_out=None):
    lib = _lib.load()
    G, Kt, ld = logits.shape
    grad = grad_out if grad_out is not None else torch.zeros_like(logits)
    _chk(scale, torch.float32, 'scale')
    bp = bag_prob.contiguous()
    check(lib.ptb_mil_loss_bwd(_ptr(logits), G, Kt, num_classes, ld, ins_off, _ptr(weight), _ptr(labels), float(eps), _ptr(bp),
                               _ptr(scale), _ptr(grad), _stream()), 'ptb_mil_loss_bwd')
    return grad


def cpr_loss_bwd_map(bag_logits, weight, mil_mt, bag_prob, label_weight, labels, centers, img_ptr, offsets, map_shape, num_classes, ins_off,
                     stride, reach_px, eps, scale_mil=None, scale_gt=None, valid_center=None, logit_map=None, neg_mask=None, scale_neg=None,
                     out=None):
    """ptb_cpr_loss_bwd_map: d loss / d logit map (B,H,W,ld), deterministic, every element written (into `out` when given)."""
    lib = _lib.load()
    _chk(bag_logits, torch.float32, 'bag_logits'); _chk(weight, torch.float32, 'weight'); _chk(centers, torch.float32, 'centers')
    B, H, W, ld = map_shape
    G, K, _ = bag_logits.shape
    if out is None:
        out = torch.empty((B, H, W, ld), dtype=torch.float32, device=bag_logits.device)
    elif tuple(_chk(out, torch.float32, 'out').shape) != (B, H, W, ld):
        raise ValueError(f'out: expected shape {(B, H, W, ld)}, got {tuple(out.shape)}')
    ws = torch.empty(int(lib.ptb_cpr_loss_bwd_map_workspace(G, num_classes)) // 4, dtype=torch.float32, device=bag_logits.device)
    check(lib.ptb_cpr_loss_bwd_map(_ptr(bag_logits), _ptr(weight), _ptr(mil_mt), _ptr(bag_prob), _ptr(label_weight), _ptr(labels),
                                   _ptr(centers), _ptr(img_ptr), _ptr(offsets), B, H, W, G, K, num_classes, ins_off, ld, float(stride),
                                   float(reach_px), float(eps), _ptr(scale_mil), _ptr(scale_gt), _ptr(valid_center), _ptr(logit_map),
                                   _ptr(neg_mask), _ptr(scale_neg), _ptr(ws), _ptr(out), _stream()), 'ptb_cpr_loss_bwd_map')
    return out


def cpr_loss_bwd_scatter(bag_logits, weight, mil_mt, bag_prob, label_weight, labels, centers, bag_img, offsets, grad_map, num_classes, ins_off,
                         stride, eps, scale_mil=None, scale_gt=None, valid_center=None):
    """ptb_cpr_loss_bwd_scatter: adds the MIL + gt part of d loss / d logit map into grad_map (B,H,W,ld) with fp32 vector atomics."""
    lib = _lib.load()
    _chk(bag_logits, torch.float32, 'bag_logits'); _chk(weight, torch.float32, 'weight'); _chk(grad_map, torch.float32, 'grad_map')
    B, H, W, ld = grad_map.shape
    G, K, _ = bag_logits.shape
    ws = torch.empty(int(lib.ptb_cpr_loss_bwd_map_workspace(G, num_classes)) // 4, dtype=torch.float32, device=bag_logits.device)
    check(lib.ptb_cpr_loss_bwd_scatter(_ptr(bag_logits), _ptr(weight), _ptr(mil_mt), _ptr(bag_prob), _ptr(label_weight), _ptr(labels),
                                       _ptr(centers), _ptr(bag_img), _ptr(offsets), B, H, W, G, K, num_classes, ins_off, ld, float(stride),
                                       float(eps), _ptr(scale_mil), _ptr(scale_gt), _ptr(valid_center), _ptr(ws), _ptr(grad_map),
                                       _stream()), 'ptb_cpr_loss_bwd_scatter')
    return grad_map


def gfocal_fwd(logits, M, num_classes, row_stride, target_label, weight, eps, loss_sum=None):
    """sum of gfocal(sigmoid(logits[m, :C]), onehot(target_label[m]) or 0) * weight.  weight: uint8 (M,C) | float (M,) | None."""
    lib = _lib.load()
    if loss_sum is None:
        loss_sum = torch.zeros(1, dtype=torch.float32, device=logits.device)
    wmode = 0 if (weight is not None and weight.dtype == torch.uint8) else 1
    check(lib.ptb_gfocal_sigmoid_fwd(_ptr(logits), M, num_classes, row_stride, _ptr(target_label), _ptr(weight), wmode,
                                     float(eps), _ptr(loss_sum), _stream()), 'ptb_gfocal_sigmoid_fwd')
    return loss_sum


def gfocal_bwd(logits, M, num_classes, row_stride, target_label, weight, eps, scale, grad, grad_row_stride, accumulate):
    lib = _lib.load()
    wmode = 0 if (weight is not None and weight.dtype == torch.uint8) else 1
    check(lib.ptb_gfocal_sigmoid_bwd(_ptr(logits), M, num_classes, row_stride, _ptr(target_label), _ptr(weight), wmode,
                                     float(eps), _ptr(scale), _ptr(grad), grad_row_stride, 1 if accumulate else 0, _stream()),
          'ptb_gfocal_sigmoid_bwd')
    return grad


# ----------------------------------------------------------------------------------------------------------------------
# P2P
# ----------------------------------------------------------------------------------------------------------------------
def p2p_decode_topk(cls_map, reg_map, num_classes, k, point_anchor, stride, pts_gamma, img_hw, nms_pre, scale_xy=None):
    """ptb_p2p_decode_topk. cls_map (B,H,W,k*C), reg_map (B,H,W,2k) channels-last logits.
    returns topk_idx (B,P) int32, pts (B,P,2), scores (B,P,C)."""
    lib = _lib.load()
    _chk(cls_map, torch.float32, 'cls_map'); _chk(reg_map, torch.float32, 'reg_map'); _chk(point_anchor, torch.float32, 'anchor')
    _chk(img_hw, torch.int32, 'img_hw')
    B, H, W, _ = cls_map.shape
    Q = H * W * k
    P = nms_pre if 0 < nms_pre < Q else Q
    dev = cls_map.device
    idx = torch.empty((B, P), dtype=torch.int32, device=dev)
    pts = torch.empty((B, P, 2), dtype=torch.float32, device=dev)
    sc = torch.empty((B, P, num_classes), dtype=torch.float32, device=dev)
    nbytes = lib.ptb_p2p_decode_topk_workspace(B, H, W, k)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    check(lib.ptb_p2p_decode_topk(_ptr(cls_map), _ptr(reg_map), B, H, W, num_classes, k, _ptr(point_anchor), float(stride),
                                  float(pts_gamma), _ptr(img_hw), _ptr(scale_xy), int(nms_pre), _ptr(idx), _ptr(pts), _ptr(sc),
                                  _ptr(ws), nbytes, _stream()), 'ptb_p2p_decode_topk')
    return idx, pts, sc


def multiclass_nms(pts, scores, pseudo_wh, score_thr, iou_thr, max_per_img):
    """ptb_multiclass_nms. pts (B,P,2), scores (B,P,C) -> count (B,), det (B,max,5), label (B,max), keep (B,max), cand_count (B,)"""
    lib = _lib.load()
    _chk(pts, torch.float32, 'pts'); _chk(scores, torch.float32, 'scores')
    B, P, C = scores.shape
    dev = pts.device
    cnt = torch.empty((B,), dtype=torch.int32, device=dev)
    det = torch.zeros((B, max_per_img, 5), dtype=torch.float32, device=dev)
    lab = torch.zeros((B, max_per_img), dtype=torch.int32, device=dev)
    keep = torch.zeros((B, max_per_img), dtype=torch.int32, device=dev)
    cc = torch.empty((B,), dtype=torch.int32, device=dev)
    nbytes = lib.ptb_multiclass_nms_workspace(B, P, C)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    check(lib.ptb_multiclass_nms(_ptr(pts), _ptr(scores), B, P, C, float(pseudo_wh[0]), float(pseudo_wh[1]), float(score_thr),
                                 float(iou_thr), int(max_per_img), _ptr(cnt), _ptr(det), _ptr(lab), _ptr(keep), _ptr(cc),
                                 _ptr(ws), nbytes, _stream()), 'ptb_multiclass_nms')
    return cnt, det, lab, keep, cc


def multiclass_nms_boxes(boxes, scores, score_thr, iou_thr, max_per_img):
    """ptb_multiclass_nms_boxes. boxes (B,P,4) xyxy, scores (B,P,C) -> count, det (B,max,5), label, keep, cand_count."""
    lib = _lib.load()
    _chk(boxes, torch.float32, 'boxes'); _chk(scores, torch.float32, 'scores')
    B, P, C = scores.shape
    dev = boxes.device
    cnt = torch.empty((B,), dtype=torch.int32, device=dev)
    det = torch.zeros((B, max_per_img, 5), dtype=torch.float32, device=dev)
    lab = torch.zeros((B, max_per_img), dtype=torch.int32, device=dev)
    keep = torch.zeros((B, max_per_img), dtype=torch.int32, device=dev)
    cc = torch.empty((B,), dtype=torch.int32, device=dev)
    nbytes = lib.ptb_multiclass_nms_workspace(B, P, C)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    check(lib.ptb_multiclass_nms_boxes(_ptr(boxes), _ptr(scores), B, P, C, float(score_thr), float(iou_thr), int(max_per_img),
                                       _ptr(cnt), _ptr(det), _ptr(lab), _ptr(keep), _ptr(cc), _ptr(ws), nbytes, _stream()),
          'ptb_multiclass_nms_boxes')
    return cnt, det, lab, keep, cc


SOFT_NMS_METHODS = {'naive': 0, 'linear': 1, 'gaussian': 2}


def multiclass_soft_nms(pts_or_boxes, scores, pseudo_wh, score_thr, iou_thr, max_per_img, sigma=0.5, min_score=1e-3, method='linear'):
    """ptb_multiclass_soft_nms.  pts_or_boxes: (B,P,2) points (pseudo boxes of pseudo_wh) or (B,P,4) boxes; scores (B,P,C).
    returns count (B,), det (B,max,5) with DECAYED scores, label, keep, cand_count."""
    lib = _lib.load()
    _chk(pts_or_boxes, torch.float32, 'pts_or_boxes'); _chk(scores, torch.float32, 'scores')
    if method not in SOFT_NMS_METHODS:
        raise KeyError(method)
    B, P, C = scores.shape
    dev = scores.device
    is_boxes = pts_or_boxes.shape[-1] == 4
    cnt = torch.empty((B,), dtype=torch.int32, device=dev)
    det = torch.zeros((B, max_per_img, 5), dtype=torch.float32, device=dev)
    lab = torch.zeros((B, max_per_img), dtype=torch.int32, device=dev)
    keep = torch.zeros((B, max_per_img), dtype=torch.int32, device=dev)
    cc = torch.empty((B,), dtype=torch.int32, device=dev)
    nbytes = lib.ptb_multiclass_soft_nms_workspace(B, P, C)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    wh = pseudo_wh if pseudo_wh is not None else (0.0, 0.0)
    check(lib.ptb_multiclass_soft_nms(None if is_boxes else _ptr(pts_or_boxes), _ptr(pts_or_boxes) if is_boxes else None, _ptr(scores),
                                      B, P, C, float(wh[0]), float(wh[1]), float(score_thr), float(iou_thr), float(sigma),
                                      float(min_score), SOFT_NMS_METHODS[method], int(max_per_img), _ptr(cnt), _ptr(det), _ptr(lab),
                                      _ptr(keep), _ptr(cc), _ptr(ws), nbytes, _stream()), 'ptb_multiclass_soft_nms')
    return cnt, det, lab, keep, cc


def p2p_cost_matrix(cls_logits, pts, row_idx, gts, gt_labels, w_cls, alpha, gamma, eps, w_dis, fx=1.0, fy=1.0, out=None):
    """ptb_p2p_cost_matrix -> (n_rows, n_gt) fp32 (written into `out`, a contiguous fp32 buffer of n_rows*n_gt elements, if given)."""
    lib = _lib.load()
    _chk(cls_logits, torch.float32, 'cls_logits'); _chk(gts, torch.float32, 'gts'); _chk(gt_labels, torch.int32, 'gt_labels')
    if pts.stride(-1) != 1 or pts.dtype != torch.float32:
        raise ValueError('pts must be fp32 with unit inner stride')
    n_rows = row_idx.shape[0] if row_idx is not None else cls_logits.shape[0]
    n_gt = gts.shape[0]
    if out is None:
        cost = torch.empty((n_rows, n_gt), dtype=torch.float32, device=cls_logits.device)
    else:
        _chk(out, torch.float32, 'out')
        if out.numel() != n_rows * n_gt:
            raise ValueError('out must hold n_rows*n_gt elements')
        cost = out.view(n_rows, n_gt)
    check(lib.ptb_p2p_cost_matrix(_ptr(cls_logits), _ptr(pts), pts.stride(0), _ptr(row_idx), n_rows, cls_logits.shape[1],
                                  _ptr(gts), _ptr(gt_labels), n_gt, float(w_cls), float(alpha), float(gamma), float(eps),
                                  float(w_dis), float(fx), float(fy), _ptr(cost), _stream()), 'ptb_p2p_cost_matrix')
    return cost


def rpn_proposals(cls_scores, bbox_preds, base_anchors, strides_wh, img_hw, means, stds, wh_ratio_clip, nms_pre, min_bbox_size, iou_thr,
                  max_per_img, want_candidates=False):
    """ptb_rpn_proposals.  cls_scores[l] (B,A,H,W) / bbox_preds[l] (B,4A,H,W) contiguous NCHW fp32 CUDA tensors, base_anchors (L,A,4),
    img_hw (B,2) int32 (h, w).  returns count (B,), det (B,max,5), level (B,max) [, dict(pos, cand_box, cand_score, cand_idx)]."""
    lib = _lib.load()
    L = len(cls_scores)
    if L == 0 or len(bbox_preds) != L:
        raise ValueError('cls_scores / bbox_preds: one tensor per level')
    for c, r in zip(cls_scores, bbox_preds):
        _chk(c, torch.float32, 'cls_score'); _chk(r, torch.float32, 'bbox_pred')
        if c.dim() != 4 or r.dim() != 4 or r.shape[1] != 4 * c.shape[1] or r.shape[-2:] != c.shape[-2:] or r.shape[0] != c.shape[0]:
            raise ValueError(f'level shapes {tuple(c.shape)} / {tuple(r.shape)}')
    _chk(base_anchors, torch.float32, 'base_anchors'); _chk(img_hw, torch.int32, 'img_hw')
    B, A = cls_scores[0].shape[:2]
    if tuple(base_anchors.shape) != (L, A, 4) or tuple(img_hw.shape) != (B, 2):
        raise ValueError('base_anchors must be (L, A, 4) and img_hw (B, 2)')
    dev = cls_scores[0].device
    hw = (ctypes.c_int32 * (2 * L))(*[int(v) for c in cls_scores for v in c.shape[-2:]])
    st = (ctypes.c_int32 * (2 * L))(*[int(v) for s in strides_wh for v in s])
    cp = (ctypes.c_void_p * L)(*[c.data_ptr() for c in cls_scores])
    bp = (ctypes.c_void_p * L)(*[r.data_ptr() for r in bbox_preds])
    mean = (ctypes.c_float * 4)(*[float(v) for v in means])
    std = (ctypes.c_float * 4)(*[float(v) for v in stds])
    Ptot = sum(min(nms_pre, c.shape[1] * c.shape[2] * c.shape[3]) if nms_pre > 0 else c.shape[1] * c.shape[2] * c.shape[3] for c in cls_scores)
    cnt = torch.empty((B,), dtype=torch.int32, device=dev)
    det = torch.zeros((B, max_per_img, 5), dtype=torch.float32, device=dev)
    lvl = torch.zeros((B, max_per_img), dtype=torch.int32, device=dev)
    extra = None
    if want_candidates:
        extra = dict(pos=torch.zeros((B, max_per_img), dtype=torch.int32, device=dev), cand_box=torch.empty((B, Ptot, 4), device=dev),
                     cand_score=torch.empty((B, Ptot), device=dev), cand_idx=torch.empty((B, Ptot), dtype=torch.int32, device=dev))
    nbytes = int(lib.ptb_rpn_proposals_workspace(hw, L, B, A, int(nms_pre), int(max_per_img)))
    if nbytes == 0:
        raise ValueError('ptb_rpn_proposals_workspace: unsupported shape')
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    e = extra or {}
    check(lib.ptb_rpn_proposals(cp, bp, hw, st, _ptr(base_anchors), L, B, A, _ptr(img_hw), mean, std, float(wh_ratio_clip), int(nms_pre),
                                float(min_bbox_size), float(iou_thr), int(max_per_img), _ptr(cnt), _ptr(det), _ptr(lvl), _ptr(e.get('pos')),
                                _ptr(e.get('cand_box')), _ptr(e.get('cand_score')), _ptr(e.get('cand_idx')), _ptr(ws), nbytes, _stream()),
          'ptb_rpn_proposals')
    return (cnt, det, lvl, extra) if want_candidates else (cnt, det, lvl)


def hungarian_v2_batch(cost_flat, shapes, topk_k, out, out_offsets, row_idx=None, row_idx_offsets=None):
    """ptb_hungarian_v2_batch: HungarianAssignerV2's matching for a batch of images, on the device.
    cost_flat      : fp32 CUDA buffer, image b = (N_b, n_b) row-major at element offset sum_{a<b} N_a*n_a
    shapes         : [(N_b, n_b)] host ints
    out            : int64 CUDA buffer, pre-zeroed; image b's assigned_gt_inds slice starts at out_offsets[b]
    row_idx        : optional int32 CUDA buffer (concatenated per image, offsets row_idx_offsets[b]): cost row -> slot in the slice
    returns status : int32 CUDA tensor (B,): 0 ok, 1 infeasible, 2 invalid entries (scipy raises ValueError for both), 3 internal."""
    lib = _lib.load()
    _chk(cost_flat, torch.float32, 'cost'); _chk(out, torch.int64, 'out')
    if row_idx is not None:
        _chk(row_idx, torch.int32, 'row_idx')
    dev = cost_flat.device
    B = len(shapes)
    status = torch.zeros((max(B, 1),), dtype=torch.int32, device=dev)
    if B == 0:
        return status[:0]
    desc, co, wo = [], 0, 0
    for b, (N, n) in enumerate(shapes):
        desc.append([co, wo, int(out_offsets[b]), int(row_idx_offsets[b]) if row_idx is not None else -1, int(N), int(n)])
        co += int(N) * int(n)
        wo += (int(lib.ptb_hungarian_v2_workspace(int(N), int(n))) + 7) // 8 * 8
    if co > cost_flat.numel():
        raise ValueError('cost buffer smaller than the shapes imply')
    max_N, max_n = max(s[0] for s in shapes), max(s[1] for s in shapes)
    d = torch.tensor(desc, dtype=torch.int64).pin_memory().to(dev, non_blocking=True)
    ws = torch.empty(max(wo, 64), dtype=torch.uint8, device=dev)
    check(lib.ptb_hungarian_v2_batch(_ptr(cost_flat), _ptr(d), B, int(max_N), int(max_n), int(topk_k), _ptr(row_idx), _ptr(out), _ptr(ws),
                                     _ptr(status), _stream()), 'ptb_hungarian_v2_batch')
    return status


def bbox_overlaps(boxes1, boxes2, mode='iou'):
    """ptb_bbox_overlaps: (m,4),(n,4) -> (m,n) IoU ('iou') or IoF w.r.t. boxes1 ('iof')  (BboxOverlaps2D, is_aligned=False)."""
    lib = _lib.load()
    _chk(boxes1, torch.float32, 'boxes1'); _chk(boxes2, torch.float32, 'boxes2')
    if mode not in ('iou', 'iof'):
        raise NotImplementedError(f'bbox_overlaps mode {mode}')
    m, n = boxes1.shape[0], boxes2.shape[0]
    out = torch.empty((m, n), dtype=torch.float32, device=boxes1.device)
    check(lib.ptb_bbox_overlaps(_ptr(boxes1), m, _ptr(boxes2), n, 1 if mode == 'iof' else 0, _ptr(out), _stream()), 'ptb_bbox_overlaps')
    return out


def max_iou_assign(bboxes, gt_bboxes, gt_labels=None, gt_bboxes_ignore=None, pos_iou_thr=0.5, neg_iou_thr=0.5, min_pos_iou=0.0,
                   gt_max_assign_all=True, ignore_iof_thr=-1, ignore_wrt_candidates=True, match_low_quality=True):
    """ptb_max_iou_assign.  returns gt_inds (N,) int64, max_overlaps (N,), labels (N,) int64 | None."""
    lib = _lib.load()
    _chk(bboxes, torch.float32, 'bboxes'); _chk(gt_bboxes, torch.float32, 'gt_bboxes')
    N, n = bboxes.shape[0], gt_bboxes.shape[0]
    dev = bboxes.device
    lo, hi = (0.0, float(neg_iou_thr)) if isinstance(neg_iou_thr, float) else (float(neg_iou_thr[0]), float(neg_iou_thr[1]))
    gt_inds = torch.empty((N,), dtype=torch.int64, device=dev)
    max_ov = torch.empty((N,), dtype=torch.float32, device=dev)
    labels = torch.empty((N,), dtype=torch.int64, device=dev) if gt_labels is not None else None
    gl = gt_labels.to(torch.int32).contiguous() if gt_labels is not None else None
    ign = gt_bboxes_ignore if (gt_bboxes_ignore is not None and gt_bboxes_ignore.numel() > 0) else None
    if ign is not None:
        _chk(ign, torch.float32, 'gt_bboxes_ignore')
    nbytes = int(lib.ptb_max_iou_assign_workspace(N, n))
    ws = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=dev)
    check(lib.ptb_max_iou_assign(_ptr(bboxes), N, _ptr(gt_bboxes), n, _ptr(gl), _ptr(ign), 0 if ign is None else ign.shape[0],
                                 float(pos_iou_thr), lo, hi, float(min_pos_iou), 1 if gt_max_assign_all else 0,
                                 1 if match_low_quality else 0, float(ignore_iof_thr), 1 if ignore_wrt_candidates else 0,
                                 _ptr(gt_inds), _ptr(max_ov), _ptr(labels), _ptr(ws), ws.numel(), _stream()), 'ptb_max_iou_assign')
    return gt_inds, max_ov, labels


def point_assigner(points, gt_bboxes, scale=4, pos_num=3):
    lib = _lib.load()
    _chk(points, torch.float32, 'points'); _chk(gt_bboxes, torch.float32, 'gt_bboxes')
    N, n = points.shape[0], gt_bboxes.shape[0]
    out = torch.zeros((N,), dtype=torch.int64, device=points.device)
    nbytes = lib.ptb_point_assigner_workspace(N, n)
    ws = torch.empty(max(nbytes, 8), dtype=torch.uint8, device=points.device)
    check(lib.ptb_point_assigner(_ptr(points), N, _ptr(gt_bboxes), n, float(scale), int(pos_num), _ptr(out), _ptr(ws), nbytes,
                                 _stream()), 'ptb_point_assigner')
    return out


def sigmoid_focal(logits, labels, weight, gamma, alpha, scale=None, want_grad=False):
    """sum_m,c focal(logits, labels) * weight[m]; optional grad = scale * d/dlogits."""
    lib = _lib.load()
    _chk(logits, torch.float32, 'logits'); _chk(labels, torch.int64, 'labels')
    M, C = logits.shape
    loss = torch.zeros(1, dtype=torch.float32, device=logits.device)
    grad = torch.empty_like(logits) if want_grad else None
    check(lib.ptb_sigmoid_focal_fwd_bwd(_ptr(logits), _ptr(labels), _ptr(weight), M, C, float(gamma), float(alpha),
                                        _ptr(loss) if not want_grad else None, _ptr(scale), _ptr(grad), _stream()),
          'ptb_sigmoid_focal_fwd_bwd')
    return grad if want_grad else loss


def smooth_l1(pred, target, weight, inv_norm, beta, scale=None, want_grad=False):
    lib = _lib.load()
    _chk(pred, torch.float32, 'pred'); _chk(target, torch.float32, 'target')
    M = pred.shape[0]
    loss = torch.zeros(1, dtype=torch.float32, device=pred.device)
    grad = torch.empty_like(pred) if want_grad else None
    check(lib.ptb_smooth_l1_fwd_bwd(_ptr(pred), _ptr(target), _ptr(weight), M, float(inv_norm), float(beta),
                                    _ptr(loss) if not want_grad else None, _ptr(scale), _ptr(grad), _stream()),
          'ptb_smooth_l1_fwd_bwd')
    return grad if want_grad else loss


# ----------------------------------------------------------------------------------------------------------------------
# conv towers on the tensor cores (3xTF32 implicit GEMM + GroupNorm + ReLU)
# ----------------------------------------------------------------------------------------------------------------------
def split_tf32(x):
    lib = _lib.load()
    _chk(x, torch.float32, 'x')
    hi, lo = torch.empty_like(x), torch.empty_like(x)
    check(lib.ptb_split_tf32(_ptr(x), x.numel(), _ptr(hi), _ptr(lo), _stream()), 'ptb_split_tf32')
    return hi, lo


def conv3x3_pack_weight(w):
    """nn.Conv2d weight (Cout,Cin,3,3) -> packed (Cout, 9*Cin) hi / lo."""
    lib = _lib.load()
    w = _chk(w.detach().contiguous(), torch.float32, 'w')
    Cout, Cin = w.shape[:2]
    hi = torch.empty((Cout, 9 * Cin), dtype=torch.float32, device=w.device)
    lo = torch.empty_like(hi)
    check(lib.ptb_conv3x3_pack_weight(_ptr(w), Cout, Cin, _ptr(hi), _ptr(lo), _stream()), 'ptb_conv3x3_pack_weight')
    return hi, lo


def conv3x3_c256(x_hi, x_lo, w_hi, w_lo, want_stats=True):
    """x_* (B,H,W,Cin) channels-last hi/lo; w_* packed (256, 9*Cin) -> y (B,H,W,256), stats (B,32,2) fp64 | None."""
    lib = _lib.load()
    _chk(x_hi, torch.float32, 'x_hi'); _chk(x_lo, torch.float32, 'x_lo'); _chk(w_hi, torch.float32, 'w_hi'); _chk(w_lo, torch.float32, 'w_lo')
    B, H, W, Cin = x_hi.shape
    if w_hi.shape != (256, 9 * Cin):
        raise ValueError('packed weight must be (256, 9*Cin)')
    y = torch.empty((B, H, W, 256), dtype=torch.float32, device=x_hi.device)
    stats = torch.zeros((B, 32, 2), dtype=torch.float64, device=x_hi.device) if want_stats else None
    check(lib.ptb_conv3x3_c256_tf32x3(_ptr(x_hi), _ptr(x_lo), _ptr(w_hi), _ptr(w_lo), B, H, W, Cin, _ptr(y), _ptr(stats), _stream()),
          'ptb_conv3x3_c256_tf32x3')
    return y, stats


def gn_relu_apply(y, stats, gamma, beta, groups=32, eps=1e-5, relu=True, split=False):
    """GroupNorm(+ReLU) from the conv epilogue's statistics; split=True returns the (hi, lo) pair for the next conv."""
    lib = _lib.load()
    _chk(y, torch.float32, 'y'); _chk(stats, torch.float64, 'stats'); _chk(gamma, torch.float32, 'gamma'); _chk(beta, torch.float32, 'beta')
    B, H, W, C = y.shape
    out_hi = torch.empty_like(y)
    out_lo = torch.empty_like(y) if split else None
    check(lib.ptb_gn_relu_apply(_ptr(y), _ptr(stats), _ptr(gamma), _ptr(beta), B, H * W, C, groups, float(eps), 1 if relu else 0,
                                _ptr(out_hi), _ptr(out_lo), _stream()), 'ptb_gn_relu_apply')
    return (out_hi, out_lo) if split else out_hi


# ---- fp16 two-term variant (half the tensor-pipe time of 3xTF32) ----
def split_f16(x, auto_scale=False):
    """x fp32 -> (h, l) fp16 with x*scale = h + l; returns (h, l, dev_inv_scale | None)."""
    lib = _lib.load()
    _chk(x, torch.float32, 'x')
    h = torch.empty(x.shape, dtype=torch.float16, device=x.device)
    l = torch.empty_like(h)
    inv = torch.empty(1, dtype=torch.float32, device=x.device) if auto_scale else None
    ws = torch.empty(1, dtype=torch.int32, device=x.device) if auto_scale else None
    check(lib.ptb_split_f16(_ptr(x), x.numel(), 1 if auto_scale else 0, _ptr(h), _ptr(l), _ptr(inv), _ptr(ws), _stream()), 'ptb_split_f16')
    return h, l, inv


def conv3x3_pack_weight_f16(w):
    """(Cout,Cin,3,3) -> packed fp16 (h, l) of w*scale and 1/scale; scale = power of two with max|w|*scale in [2^9, 2^10)."""
    lib = _lib.load()
    w = _chk(w.detach().contiguous(), torch.float32, 'w')
    Cout, Cin = w.shape[:2]
    amax = float(w.abs().max())
    scale = 1.0
    if amax > 0 and math.isfinite(amax):
        scale = 2.0 ** (10 - math.frexp(amax)[1])
    h = torch.empty((Cout, 9 * Cin), dtype=torch.float16, device=w.device)
    l = torch.empty_like(h)
    check(lib.ptb_conv3x3_pack_weight_f16(_ptr(w), Cout, Cin, float(scale), _ptr(h), _ptr(l), _stream()), 'ptb_conv3x3_pack_weight_f16')
    return h, l, 1.0 / scale


def conv3x3_c256_f16(x_h, x_l, w_h, w_l, out_scale, dev_out_scale=None, want_stats=True):
    lib = _lib.load()
    _chk(x_h, torch.float16, 'x_h'); _chk(x_l, torch.float16, 'x_l'); _chk(w_h, torch.float16, 'w_h'); _chk(w_l, torch.float16, 'w_l')
    B, H, W, Cin = x_h.shape
    if w_h.shape != (256, 9 * Cin):
        raise ValueError('packed weight must be (256, 9*Cin)')
    y = torch.empty((B, H, W, 256), dtype=torch.float32, device=x_h.device)
    stats = torch.zeros((B, 32, 2), dtype=torch.float64, device=x_h.device) if want_stats else None
    check(lib.ptb_conv3x3_c256_f16x2(_ptr(x_h), _ptr(x_l), _ptr(w_h), _ptr(w_l), B, H, W, Cin, float(out_scale), _ptr(dev_out_scale),
                                     _ptr(y), _ptr(stats), _stream()), 'ptb_conv3x3_c256_f16x2')
    return y, stats


def gn_relu_apply_f16(y, stats, gamma, beta, groups=32, eps=1e-5, relu=True, overflow_flag=None):
    lib = _lib.load()
    _chk(y, torch.float32, 'y'); _chk(stats, torch.float64, 'stats')
    B, H, W, C = y.shape
    h = torch.empty(y.shape, dtype=torch.float16, device=y.device)
    l = torch.empty_like(h)
    check(lib.ptb_gn_relu_apply_f16(_ptr(y), _ptr(stats), _ptr(gamma), _ptr(beta), B, H * W, C, groups, float(eps), 1 if relu else 0,
                                    _ptr(h), _ptr(l), _ptr(overflow_flag), _stream()), 'ptb_gn_relu_apply_f16')
    return h, l


def gn_relu_bwd(da, y, stats, gamma, beta, groups=32, eps=1e-5, relu=True, want_amax=True):
    """ptb_gn_relu_bwd: backward of GroupNorm(+ReLU) on channels-last (B,H,W,C) tensors.
    returns dy (B,H,W,C) fp32, dgamma (C,), dbeta (C,), amax_bits (1,) int32 device (float bits of max|dy|) | None."""
    lib = _lib.load()
    _chk(da, torch.float32, 'da'); _chk(y, torch.float32, 'y'); _chk(stats, torch.float64, 'stats')
    B, H, W, C = y.shape
    dev = y.device
    nbytes = int(lib.ptb_gn_relu_bwd_workspace(B, H * W, C, groups))
    if nbytes == 0:
        raise ValueError(f'ptb_gn_relu_bwd: unsupported shape C={C}, groups={groups}')
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    dy = torch.empty_like(y)
    dg = torch.empty(C, dtype=torch.float32, device=dev)
    db = torch.empty(C, dtype=torch.float32, device=dev)
    amax = torch.zeros(1, dtype=torch.int32, device=dev) if want_amax else None
    check(lib.ptb_gn_relu_bwd(_ptr(da), _ptr(y), _ptr(stats), _ptr(gamma), _ptr(beta), B, H * W, C, groups, float(eps),
                              1 if relu else 0, _ptr(ws), _ptr(dy), _ptr(dg), _ptr(db), _ptr(amax), _stream()), 'ptb_gn_relu_bwd')
    return dy, dg, db, amax


def split_f16_amax(x, amax_bits):
    """x fp32 -> (h, l, dev_inv_scale) with the power-of-two scale chosen on the device from amax_bits (float bits of max|x|)."""
    lib = _lib.load()
    _chk(x, torch.float32, 'x')
    h = torch.empty(x.shape, dtype=torch.float16, device=x.device)
    l = torch.empty_like(h)
    inv = torch.empty(1, dtype=torch.float32, device=x.device)
    check(lib.ptb_split_f16_amax(_ptr(x), x.numel(), _ptr(amax_bits), _ptr(h), _ptr(l), _ptr(inv), _stream()), 'ptb_split_f16_amax')
    return h, l, inv


def conv3x3_wgrad_f16(dy_h, dy_l, x_h, x_l, scale=1.0, dev_scale_dy=None, dev_scale_x=None, out=None, accumulate=False):
    """ptb_conv3x3_wgrad_f16x2: dW (Cout,Cin,3,3) = scale * s_dy * s_x * sum_pixels dy (x) x_shifted; operands are fp16 pairs
    (B,H,W,256) channels-last."""
    lib = _lib.load()
    _chk(dy_h, torch.float16, 'dy_h'); _chk(dy_l, torch.float16, 'dy_l'); _chk(x_h, torch.float16, 'x_h'); _chk(x_l, torch.float16, 'x_l')
    B, H, W, Cout = dy_h.shape
    Cin = x_h.shape[3]
    ws = torch.empty(int(lib.ptb_conv3x3_wgrad_workspace(B, H, W)), dtype=torch.uint8, device=dy_h.device)
    dw = out if out is not None else torch.empty((Cout, Cin, 3, 3), dtype=torch.float32, device=dy_h.device)
    check(lib.ptb_conv3x3_wgrad_f16x2(_ptr(dy_h), _ptr(dy_l), _ptr(x_h), _ptr(x_l), B, H, W, Cout, Cin, float(scale), _ptr(dev_scale_dy),
                                      _ptr(dev_scale_x), _ptr(ws), _ptr(dw), 1 if accumulate else 0, _stream()),
          'ptb_conv3x3_wgrad_f16x2')
    return dw


def conv_tc_wgrad_f16(dy_h, dy_l, x_h, x_l, taps, scale=1.0, dev_scale_dy=None, dev_scale_x=None):
    """ptb_conv_tc_wgrad_f16x2: dW (Cout, 256[, 3, 3]) of a conv3x3 (taps 9) / per-cell Linear (taps 1) from fp16 operand pairs
    (B,H,W,Cout) and (B,H,W,256); tensor cores with K = pixels, deterministic."""
    lib = _lib.load()
    _chk(dy_h, torch.float16, 'dy_h'); _chk(dy_l, torch.float16, 'dy_l'); _chk(x_h, torch.float16, 'x_h'); _chk(x_l, torch.float16, 'x_l')
    B, H, W, Cout = dy_h.shape
    Cin = x_h.shape[3]
    ws = torch.empty(int(lib.ptb_conv_tc_wgrad_workspace(B, H, W, taps)), dtype=torch.uint8, device=dy_h.device)
    dw = torch.empty((Cout, Cin, 3, 3) if taps == 9 else (Cout, Cin), dtype=torch.float32, device=dy_h.device)
    check(lib.ptb_conv_tc_wgrad_f16x2(_ptr(dy_h), _ptr(dy_l), _ptr(x_h), _ptr(x_l), B, H, W, Cout, Cin, taps, float(scale), _ptr(dev_scale_dy),
                                      _ptr(dev_scale_x), _ptr(ws), _ptr(dw), 0, _stream()), 'ptb_conv_tc_wgrad_f16x2')
    return dw


def col_sum(y2d):
    """ptb_col_sum: out[n] = sum_m y[m][n] of a contiguous fp32 (M, N) matrix, fixed order."""
    lib = _lib.load()
    _chk(y2d, torch.float32, 'y2d')
    M, N = y2d.shape
    ws = torch.empty(int(lib.ptb_col_sum_workspace(M, N)) // 4, dtype=torch.float32, device=y2d.device)
    out = torch.empty(N, dtype=torch.float32, device=y2d.device)
    check(lib.ptb_col_sum(_ptr(y2d), M, N, N, _ptr(ws), _ptr(out), _stream()), 'ptb_col_sum')
    return out


def conv_tc_pack_weight_f16(w, taps):
    """weights of a conv3x3 (n_out,Cin,3,3) or Linear / conv1x1 (n_out,Cin) -> packed fp16 (h, l), 1/scale, n_mma."""
    lib = _lib.load()
    w = _chk(w.detach().contiguous(), torch.float32, 'w')
    n_out, Cin = w.shape[0], w.shape[1]
    n_mma = (n_out + 15) // 16 * 16
    amax = float(w.abs().max())
    scale = 2.0 ** (10 - math.frexp(amax)[1]) if (amax > 0 and math.isfinite(amax)) else 1.0
    h = torch.empty((n_mma, taps * Cin), dtype=torch.float16, device=w.device)
    l = torch.empty_like(h)
    check(lib.ptb_conv_tc_pack_weight_f16(_ptr(w), n_out, n_mma, Cin, taps, float(scale), _ptr(h), _ptr(l), _stream()),
          'ptb_conv_tc_pack_weight_f16')
    return h, l, 1.0 / scale, n_mma


def conv_tc_f16(x_h, x_l, packed, taps, n_out, bias=None, dev_out_scale=None, ldy=None):
    """general tcgen05 conv (taps 1|9) on fp16 operand pairs -> (B,H,W,ldy) fp32 (+bias)."""
    lib = _lib.load()
    _chk(x_h, torch.float16, 'x_h'); _chk(x_l, torch.float16, 'x_l')
    w_h, w_l, inv_w, n_mma = packed
    B, H, W, Cin = x_h.shape
    ldy = ldy or (n_out + 3) // 4 * 4
    y = torch.empty((B, H, W, ldy), dtype=torch.float32, device=x_h.device)
    check(lib.ptb_conv_tc_f16x2(_ptr(x_h), _ptr(x_l), _ptr(w_h), _ptr(w_l), B, H, W, Cin, taps, n_out, n_mma, float(inv_w),
                                _ptr(dev_out_scale), _ptr(bias), _ptr(y), ldy, _stream()), 'ptb_conv_tc_f16x2')
    return y


# ----------------------------------------------------------------------------------------------------------------------
# R-CNN box stage (roi_head.py)
# ----------------------------------------------------------------------------------------------------------------------
def amax_abs(tensors):
    """ptb_amax_abs over several fp32 tensors -> (1,) int32 device tensor holding the float bits of max|x| (no host sync)."""
    lib = _lib.load()
    bits = torch.empty(1, dtype=torch.int32, device=tensors[0].device)
    for i, t in enumerate(tensors):
        _chk(t, torch.float32, 'x')
        check(lib.ptb_amax_abs(_ptr(t), t.numel(), _ptr(bits), 1 if i else 0, _stream()), 'ptb_amax_abs')
    return bits


def roi_align(feats_nhwc, rois, out_size=(7, 7), spatial_scales=None, sampling_ratio=0, aligned=True, finest_scale=56, f16_pair=False,
              row_multiple=16, want_levels=False):
    """ptb_roi_align.  feats_nhwc: list of (B,H,W,C) contiguous fp32 level maps; rois (M,5) fp32.
    returns fp32 (M, oh, ow, C) — or with f16_pair (h, l, dev_inv_scale), h / l (M_pad, oh*ow*C) fp16, M_pad = M rounded up to
    row_multiple — plus the (M,) int8 levels when want_levels."""
    lib = _lib.load()
    L = len(feats_nhwc)
    if not 1 <= L <= 5:
        raise ValueError(f'ptb_roi_align takes 1 to 5 levels, got {L}')
    for f in feats_nhwc:
        _chk(f, torch.float32, 'feat')
    _chk(rois, torch.float32, 'rois')
    if rois.dim() != 2 or rois.shape[1] != 5:
        raise ValueError('rois must be (M, 5)')
    B, _, _, C = feats_nhwc[0].shape
    if any(f.shape[0] != B or f.shape[3] != C for f in feats_nhwc):
        raise ValueError('level maps must share batch size and channels')
    if C % 32:
        raise ValueError(f'ptb_roi_align needs C % 32 == 0, got C = {C}')
    oh, ow = out_size
    M = rois.shape[0]
    dev = rois.device
    hw = (ctypes.c_int32 * (2 * L))(*[int(v) for f in feats_nhwc for v in f.shape[1:3]])
    fp = (ctypes.c_void_p * L)(*[f.data_ptr() for f in feats_nhwc])
    sc = (ctypes.c_float * L)(*[float(s) for s in spatial_scales])
    lvl = torch.empty(M, dtype=torch.int8, device=dev) if want_levels else None
    if f16_pair:
        Mp = (M + row_multiple - 1) // row_multiple * row_multiple
        bits = amax_abs(feats_nhwc)
        h = torch.empty((Mp, oh * ow * C), dtype=torch.float16, device=dev)
        l = torch.empty_like(h)
        inv = torch.empty(1, dtype=torch.float32, device=dev)
        check(lib.ptb_roi_align(_ptr(rois), M, Mp, fp, hw, sc, L, B, C, oh, ow, int(sampling_ratio), 1 if aligned else 0, float(finest_scale),
                                _ptr(bits), None, _ptr(h), _ptr(l), _ptr(inv), _ptr(lvl), _stream()), 'ptb_roi_align')
        out = (h, l, inv)
    else:
        out = torch.empty((M, oh, ow, C), dtype=torch.float32, device=dev)
        check(lib.ptb_roi_align(_ptr(rois), M, M, fp, hw, sc, L, B, C, oh, ow, int(sampling_ratio), 1 if aligned else 0, float(finest_scale),
                                None, _ptr(out), None, None, None, _ptr(lvl), _stream()), 'ptb_roi_align')
    return (out, lvl) if want_levels else out


def relu_split_f16(y, n=None, overflow_flag=None):
    """ptb_relu_split_f16: (rows, ld) fp32 -> fp16 pair (rows, n) of relu(y[:, :n]) at unit scale."""
    lib = _lib.load()
    _chk(y, torch.float32, 'y')
    rows, ld = y.shape
    n = ld if n is None else n
    h = torch.empty((rows, n), dtype=torch.float16, device=y.device)
    l = torch.empty_like(h)
    check(lib.ptb_relu_split_f16(_ptr(y), rows, n, ld, _ptr(h), _ptr(l), _ptr(overflow_flag), _stream()), 'ptb_relu_split_f16')
    return h, l


def linear_tc_f16(x_h, x_l, packs, n_out, bias=None, dev_in_scale=None):
    """y (M_pad, ldy) = x @ W.T + bias on ptb_conv_tc_f16x2 with 1 tap: the rows of x (M_pad, K) fp16 pair are the 'pixels' of a
    (1, M_pad/16, 16, K) operand; `packs` = [(h, l, inv_w, n_mma)] column slices of <= 256 outputs (conv_tc_pack_weight_f16)."""
    lib = _lib.load()
    _chk(x_h, torch.float16, 'x_h'); _chk(x_l, torch.float16, 'x_l')
    Mp, K = x_h.shape
    if Mp % 16 or K % 32:
        raise ValueError(f'linear_tc_f16: rows must be a multiple of 16 and K of 32, got {tuple(x_h.shape)}')
    ldy = (n_out + 3) // 4 * 4
    y = torch.empty((Mp, ldy), dtype=torch.float32, device=x_h.device)
    if Mp == 0:
        return y
    n0 = 0
    for (w_h, w_l, inv_w, n_mma) in packs:
        ns = min(n_mma, n_out - n0)
        check(lib.ptb_conv_tc_f16x2(_ptr(x_h), _ptr(x_l), _ptr(w_h), _ptr(w_l), 1, Mp // 16, 16, K, 1, ns, n_mma, float(inv_w),
                                    _ptr(dev_in_scale), _ptr(bias[n0:] if bias is not None else None), ctypes.c_void_p(y.data_ptr() + 4 * n0),
                                    ldy, _stream()), 'ptb_conv_tc_f16x2')
        n0 += ns
    return y


def rcnn_bbox_decode(rois, n_per_img, cls, reg, num_classes, means, stds, img_hw, scale_factor=None, mask_padding=False,
                     wh_ratio_clip=16 / 1000, want_scores=True, want_candidates=True):
    """ptb_rcnn_bbox_decode.  rois (B*n, 5); cls (B*n, >= N+1) / reg (B*n, >= 4N) row-strided views with unit inner stride.
    returns boxes (B*n, 4N), scores (B*n, N+1) | None, candidate scores (B, n*N, N) | None."""
    lib = _lib.load()
    _chk(rois, torch.float32, 'rois'); _chk(img_hw, torch.int32, 'img_hw')
    for t, nm in ((cls, 'cls'), (reg, 'reg')):
        if t.dtype != torch.float32 or not t.is_cuda or t.stride(-1) != 1:
            raise RuntimeError(f'{nm}: expected a CUDA fp32 matrix with unit inner stride')
    if scale_factor is not None:
        _chk(scale_factor, torch.float32, 'scale_factor')
    R = rois.shape[0]
    B = img_hw.shape[0]
    if R != B * n_per_img:
        raise ValueError('rois must hold n_per_img rows per image')
    N = int(num_classes)
    dev = rois.device
    boxes = torch.empty((R, 4 * N), dtype=torch.float32, device=dev)
    scores = torch.empty((R, N + 1), dtype=torch.float32, device=dev) if want_scores else None
    cand = torch.empty((B, n_per_img * N, N), dtype=torch.float32, device=dev) if want_candidates else None
    mean = (ctypes.c_float * 4)(*[float(v) for v in means])
    std = (ctypes.c_float * 4)(*[float(v) for v in stds])
    check(lib.ptb_rcnn_bbox_decode(_ptr(rois), B, n_per_img, _ptr(cls), cls.stride(0) if R > 1 else cls.shape[1], _ptr(reg),
                                   reg.stride(0) if R > 1 else reg.shape[1], N, 1 if mask_padding else 0, mean, std, float(wh_ratio_clip),
                                   _ptr(img_hw), _ptr(scale_factor), _ptr(boxes), _ptr(scores), _ptr(cand), _stream()),
          'ptb_rcnn_bbox_decode')
    return boxes, scores, cand
