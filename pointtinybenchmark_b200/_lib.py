"""ctypes binding of libptb_b200.so (the C ABI declared in include/ptb_b200.h).

There is NO fallback: if the CUDA library is missing or fails to load, every op raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libptb_b200.so')

_lib = None
MISSING = []

c_int, c_float, c_void_p, c_u64, c_i64 = ctypes.c_int, ctypes.c_float, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int64


class RefineCfg(ctypes.Structure):
    _fields_ = [('merge_th', c_float), ('gt_alpha', c_float), ('refine_th', c_float), ('flags', ctypes.c_int32)]


P = c_void_p
# name -> (restype, argtypes); must list every symbol of include/ptb_b200.h (tests/test_capi_symbols.py checks)
SIGNATURES = {
    'ptb_abi_version': (c_int, []),
    'ptb_last_error': (ctypes.c_char_p, []),
    'ptb_launch_count': (c_u64, []),
    'ptb_reset_stream_state': (c_int, [P]),
    'ptb_cpr_bag_gather': (c_int, [P, c_int, c_int, c_int, c_int, c_int, P, P, c_int, P, c_int, c_float, c_float, P, P, P, P, P]),
    'ptb_cpr_bag_gather_bwd': (c_int, [P, c_int, c_int, c_int, c_int, c_int, P, P, c_int, P, c_int, c_float, P, P]),
    'ptb_linear_rows': (c_int, [P, c_int, c_int, c_int, P, P, c_int, P, c_int, P]),
    'ptb_linear_rows_bwd_x': (c_int, [P, c_int, c_int, c_int, P, c_int, P, c_int, c_int, P]),
    'ptb_linear_rows_bwd_w': (c_int, [P, c_int, c_int, c_int, P, c_int, c_int, P, P, P, c_u64, P]),
    'ptb_linear_rows_bwd_w_workspace': (c_u64, [c_int, c_int, c_int]),
    'ptb_cpr_neg_mask': (c_int, [c_int, c_int, c_int, c_float, P, P, P, P, c_int, c_float, c_int, c_int, P, P]),
    'ptb_cpr_grid_bag': (c_int, [P, c_int, c_int, c_int, c_int, c_int, P, P, c_int, c_float, c_float, c_int, P, P, P, P, P, P]),
    'ptb_cpr_grid_bag_bwd': (c_int, [P, c_int, c_int, c_int, c_int, c_int, P, P, P, c_int, c_int, c_float, P, P]),
    'ptb_label_groups': (c_int, [P, P, c_int, c_int, c_int, c_int, P, P, P, P]),
    'ptb_cpr_refine': (c_int, [P, P, P, c_int, c_int, c_int, c_int, P, P, P, P, P, P, P, RefineCfg, P, P, P, P, P, P]),
    'ptb_cpr_refine_fused': (c_int, [P, c_int, c_int, c_int, c_int, c_int, P, P, P, c_int, P, c_int, c_float, c_float, P, P, P, P, P,
                                     P, RefineCfg, P, P, P, P, P]),
    'ptb_mil_loss_fwd': (c_int, [P, c_int, c_int, c_int, c_int, c_int, P, P, c_float, P, P, P, P, P]),
    'ptb_cpr_bag_mil_fwd': (c_int, [P, c_int, c_int, c_int, c_int, c_int, c_int, P, P, c_int, P, c_int, c_float, P, P, c_float, P, P, P, P, P, P, P]),
    'ptb_cpr_loss_bwd_map': (c_int, [P, P, P, P, P, P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_float, c_float,
                                     P, P, P, P, P, P, P, P, P]),
    'ptb_cpr_loss_bwd_map_workspace': (c_u64, [c_int, c_int]),
    'ptb_cpr_loss_bwd_scatter': (c_int, [P, P, P, P, P, P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_float,
                                         P, P, P, P, P, P]),
    'ptb_mil_loss_bwd': (c_int, [P, c_int, c_int, c_int, c_int, c_int, P, P, c_float, P, P, P, P]),
    'ptb_gfocal_sigmoid_fwd': (c_int, [P, c_i64, c_int, c_i64, P, P, c_int, c_float, P, P]),
    'ptb_gfocal_sigmoid_bwd': (c_int, [P, c_i64, c_int, c_i64, P, P, c_int, c_float, P, P, c_i64, c_int, P]),
    'ptb_p2p_decode_topk': (c_int, [P, P, c_int, c_int, c_int, c_int, c_int, P, c_float, c_float, P, P, c_int, P, P, P, P,
                                    c_u64, P]),
    'ptb_p2p_decode_topk_workspace': (c_u64, [c_int, c_int, c_int, c_int]),
    'ptb_multiclass_nms': (c_int, [P, P, c_int, c_int, c_int, c_float, c_float, c_float, c_float, c_int, P, P, P, P, P, P,
                                   c_u64, P]),
    'ptb_multiclass_nms_workspace': (c_u64, [c_int, c_int, c_int]),
    'ptb_multiclass_soft_nms': (c_int, [P, P, P, c_int, c_int, c_int, c_float, c_float, c_float, c_float, c_float, c_float, c_int, c_int,
                                        P, P, P, P, P, P, c_u64, P]),
    'ptb_multiclass_soft_nms_workspace': (c_u64, [c_int, c_int, c_int]),
    'ptb_multiclass_nms_boxes': (c_int, [P, P, c_int, c_int, c_int, c_float, c_float, c_int, P, P, P, P, P, P, c_u64, P]),
    'ptb_p2p_cost_matrix': (c_int, [P, P, c_int, P, c_int, c_int, P, P, c_int, c_float, c_float, c_float, c_float, c_float,
                                    c_float, c_float, P, P]),
    'ptb_rpn_proposals_workspace': (c_u64, [P, c_int, c_int, c_int, c_int, c_int]),
    'ptb_rpn_proposals': (c_int, [P, P, P, P, P, c_int, c_int, c_int, P, P, P, c_float, c_int, c_float, c_float, c_int, P, P, P, P, P, P, P, P, c_u64, P]),
    'ptb_hungarian_v2_workspace': (c_u64, [c_int, c_int]),
    'ptb_hungarian_v2_batch': (c_int, [P, P, c_int, c_int, c_int, c_int, P, P, P, P, P]),
    'ptb_point_assigner': (c_int, [P, c_int, P, c_int, c_float, c_int, P, P, c_u64, P]),
    'ptb_point_assigner_workspace': (c_u64, [c_int, c_int]),
    'ptb_sigmoid_focal_fwd_bwd': (c_int, [P, P, P, c_i64, c_int, c_float, c_float, P, P, P, P]),
    'ptb_smooth_l1_fwd_bwd': (c_int, [P, P, P, c_i64, c_float, c_float, P, P, P, P]),
    'ptb_split_tf32': (c_int, [P, c_i64, P, P, P]),
    'ptb_conv3x3_pack_weight': (c_int, [P, c_int, c_int, P, P, P]),
    'ptb_conv3x3_c256_tf32x3': (c_int, [P, P, P, P, c_int, c_int, c_int, c_int, P, P, P]),
    'ptb_gn_relu_apply': (c_int, [P, P, P, P, c_int, c_int, c_int, c_int, c_float, c_int, P, P, P]),
    'ptb_split_f16': (c_int, [P, c_i64, c_int, P, P, P, P, P]),
    'ptb_conv3x3_pack_weight_f16': (c_int, [P, c_int, c_int, c_float, P, P, P]),
    'ptb_conv3x3_c256_f16x2': (c_int, [P, P, P, P, c_int, c_int, c_int, c_int, c_float, P, P, P, P]),
    'ptb_conv_tc_pack_weight_f16': (c_int, [P, c_int, c_int, c_int, c_int, c_float, P, P, P]),
    'ptb_conv_tc_f16x2': (c_int, [P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float, P, P, P, c_int, P]),
    'ptb_gn_relu_apply_f16': (c_int, [P, P, P, P, c_int, c_int, c_int, c_int, c_float, c_int, P, P, P, P]),
    'ptb_max_iou_assign_workspace': (c_u64, [c_int, c_int]),
    'ptb_max_iou_assign': (c_int, [P, c_int, P, c_int, P, P, c_int, c_float, c_float, c_float, c_float, c_int, c_int, c_float, c_int,
                                   P, P, P, P, c_u64, P]),
    'ptb_bbox_overlaps': (c_int, [P, c_int, P, c_int, c_int, P, P]),
    'ptb_gn_relu_bwd_workspace': (c_u64, [c_int, c_int, c_int, c_int]),
    'ptb_gn_relu_bwd': (c_int, [P, P, P, P, P, c_int, c_int, c_int, c_int, c_float, c_int, P, P, P, P, P, P]),
    'ptb_split_f16_amax': (c_int, [P, c_i64, P, P, P, P, P]),
    'ptb_conv3x3_wgrad_workspace': (c_u64, [c_int, c_int, c_int]),
    'ptb_conv3x3_wgrad_f16x2': (c_int, [P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_float, P, P, P, P, c_int, P]),
    'ptb_conv_tc_wgrad_workspace': (c_u64, [c_int, c_int, c_int, c_int]),
    'ptb_conv_tc_wgrad_f16x2': (c_int, [P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_float, P, P, P, P, c_int, P]),
    'ptb_col_sum_workspace': (c_u64, [c_i64, c_int]),
    'ptb_col_sum': (c_int, [P, c_i64, c_int, c_int, P, P, P]),
    'ptb_amax_abs': (c_int, [P, c_i64, P, c_int, P]),
    'ptb_roi_align': (c_int, [P, c_int, c_int, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float, P, P, P, P, P, P, P]),
    'ptb_relu_split_f16': (c_int, [P, c_int, c_int, c_int, P, P, P, P]),
    'ptb_rcnn_bbox_decode': (c_int, [P, c_int, c_int, P, c_int, P, c_int, c_int, c_int, P, P, c_float, P, P, P, P, P, P]),
}


def load():
    """dlopen the in-tree library; raises (never falls back) when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f'{LIB_PATH} is missing: build it with `python -c "import __graft_entry__ as g; g.build()"` '
            '(nvcc, sm_100a). pointtinybenchmark_b200 has no CPU or PyTorch fallback.')
    lib = ctypes.CDLL(LIB_PATH)
    missing = []
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            missing.append(name)
            continue
        fn.restype = res
        fn.argtypes = args
    global MISSING
    MISSING = missing      # tests/test_capi_symbols.py requires this to be empty
    if lib.ptb_abi_version() != 1:
        raise RuntimeError('libptb_b200.so ABI version mismatch')
    _lib = lib
    return lib


def check(rc, name):
    if rc != 0:
        msg = load().ptb_last_error().decode(errors='replace')
        raise RuntimeError(f'{name} failed (rc={rc}): {msg}')
