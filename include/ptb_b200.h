/* ptb_b200.h — C ABI of libptb_b200.so: the B200 (sm_100a) CPR / P2P point-localization hot path.
 *
 * The reference (ucas-vg/PointTinyBenchmark, TOV_mmdetection) is pure Python: it has NO FFI for this path.  Its
 * "plugin boundary" is the mmdet dense-head protocol (HEADS registry).  This header is the C ABI that sits directly
 * under the Python head classes in pointtinybenchmark_b200/ (ctypes binding, see INTEGRATION.md); every entry point
 * names the reference code (file:line under TOV_mmdetection/) it replaces.
 *
 * Conventions
 *   - all pointers are DEVICE pointers (cudaMalloc'ed / torch CUDA storage) unless the name ends in _host;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); every call is asynchronous on it;
 *   - every function returns 0 on success, non-zero on error; ptb_last_error() gives the message of the last failure
 *     on the calling thread (argument validation errors and CUDA launch errors alike);
 *   - feature / logit maps are channels-last:  map[b][y][x][c], c fastest;  `ld` = floats per (b,y,x) cell;
 *   - point sets of a batch are concatenated over images ("CSR"): img_ptr[b]..img_ptr[b+1] are the GTs of image b;
 *   - bool outputs are uint8_t 0/1;  indices are int32_t unless stated.
 */
#ifndef PTB_B200_H_
#define PTB_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PTB_ABI_VERSION 1

int ptb_abi_version(void);
const char* ptb_last_error(void);
/* number of kernels launched by this library since load (all threads) — bench.py's `gpu_launches` claim */
uint64_t ptb_launch_count(void);
/* The dynamic chunk schedulers and the fixed-order block reductions keep their tickets / partials in a small scratch block owned by
 * the library PER (device, stream) — created on first use — so launches on different streams never share counters.  The counters reset
 * themselves at the end of every kernel; after an ABORTED launch (device fault, killed context) call this to zero the block of `stream`. */
int ptb_reset_stream_state(void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Neighbor gather  — replaces PtFeatGenerator.extract_point_feat + grid_sample
 *   (mmdet/models/point/dense_heads/cpr_head.py:182-199, 73-93) together with
 *   CirclePtFeatGenerator.generate / get_point_neighbours / get_point_valid (cpr_head.py:453-497, 172-180).
 * For every bag g (centre centers[g], image bag_img[g]) and every offset k:  p = centers[g] + offsets[k];
 *   out_pts[g][k]   = (p.x, p.y, stride)
 *   out_valid[g][k] = 0<=p.x<pad_w && 0<=p.y<pad_h                        (pad_hw[b] = {pad_h, pad_w})
 *   out_feats[g][k][0..C) = bilinear sample of map[b] at p/stride, align_corners=False, border padding,
 *                           using ATen's fp32 coordinate pipeline  ix = fma((2u+1)/W-1+1, W/2, -0.5).
 * C must be a multiple of 4 and ld >= C (ld multiple of 4).  Any of out_feats/out_pts/out_valid may be NULL.
 * The same entry point samples the 80-channel logit maps of the fused path (C = num classes).
 */
int ptb_cpr_bag_gather(const float* map, int B, int H, int W, int C, int ld,
                       const float* centers /*[G][2]*/, const int32_t* bag_img /*[G]*/, int G,
                       const float* offsets /*[K][2]*/, int K, float stride,
                       float reach_px /* max_k |offsets[k]| (radius * stride), 0 = unknown: with it and C % 32 == 0 the bag's window of
                                         2*ceil(reach/stride)+2 cells per side is staged per channel chunk by one TMA box */,
                       const int32_t* pad_hw /*[B][2]*/,
                       float* out_feats /*[G][K][C]*/, float* out_pts /*[G][K][3]*/, uint8_t* out_valid /*[G][K]*/,
                       void* stream);

/* backward of the gather w.r.t. the map (scatter-add of bilinear taps; grid_sampler_2d_backward semantics).
 * grad_map must be zero-initialised by the caller; accumulation uses fp32 atomics (red.global.add.v4.f32). */
int ptb_cpr_bag_gather_bwd(const float* grad_out /*[G][K][C]*/, int B, int H, int W, int C, int ld,
                           const float* centers, const int32_t* bag_img, int G,
                           const float* offsets, int K, float stride,
                           float* grad_map /*[B][H][W][ld]*/, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Per-cell linear classifier  y[m][n] = sum_c x[m][c] * w[n][c] + bias[n]   — replaces CPRHead.get_pts_outs
 *   (cpr_head.py:1045-1078: nn.Linear cls_out / ins_out) applied to every map cell (1x1 conv form).
 * x: [M][ldx] (first Cin used), w: [N][Cin] row-major (nn.Linear layout), y: [M][ldy].  Cin % 4 == 0.
 * fp32 FFMA accumulation (parity mode: no TF32).
 */
int ptb_linear_rows(const float* x, int M, int Cin, int ldx, const float* w, const float* bias, int N,
                    float* y, int ldy, void* stream);
/* dX[m][c] = sum_n dY[m][n] w[n][c]   (accumulate=0: overwrite, 1: add) */
int ptb_linear_rows_bwd_x(const float* dy, int M, int N, int ldy, const float* w, int Cin,
                          float* dx, int ldx, int accumulate, void* stream);
/* dW[n][c] = sum_m dY[m][n] x[m][c];  db[n] = sum_m dY[m][n]   (overwrite; fixed-order tree reduction) */
int ptb_linear_rows_bwd_w(const float* dy, int M, int N, int ldy, const float* x, int Cin, int ldx,
                          float* dw /*[N][Cin]*/, float* db /*[N]*/, float* workspace, uint64_t workspace_bytes,
                          void* stream);
uint64_t ptb_linear_rows_bwd_w_workspace(int M, int N, int Cin);

/* ------------------------------------------------------------------------------------------------------------------
 * Negative (out-of-circle) mask — replaces OutCirclePtFeatGenerator.generate (cpr_head.py:254-290) and
 * AnchorPtFeatGenerator.anchor_points (cpr_head.py:240-244) for one FPN level.
 *   grid point (x,y) of cell (i,j) = (j*stride + stride/2, i*stride + stride/2);  cell_valid = inside pad_hw[b];
 *   class_wise:  out[b][i][j][c] = cell_valid && min_{g in image b, labels[g]==c} dist(p, centers[g]) >= thresh
 *   otherwise :  out[b][i][j][c] = cell_valid && min_{g in image b} dist(p, centers[g]) >= thresh       (all c)
 * dist reproduces torch.cdist's matmul formulation in fp32 (the reference's integer mask is defined by it; DESIGN.md).
 */
int ptb_cpr_neg_mask(int B, int H, int W, float stride, const int32_t* pad_hw,
                     const float* centers /*[G][2]*/, const int32_t* labels /*[G]*/, const int32_t* img_ptr /*[B+1]*/,
                     int G, float thresh, int num_classes, int class_wise,
                     uint8_t* out /*[B][H][W][num_classes]*/, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Point refinement — replaces PointRefiner.refine_single with nearest_filter / classify_filter / inside_img
 *   (cpr_head.py:780-850, 711-756, 773-778).
 * Kt = num_refine * K samples per GT; the centre of refine 0 is sample `center_idx` (= K-1).
 * grp_ptr/grp_idx: CSR of same-(image,label) GT groups: members of GT g's group are
 *   grp_idx[grp_ptr[grp_of[g]] .. grp_ptr[grp_of[g]+1]) in ascending GT order (host builds it; it is the
 *   group_by_label of cpr_head.py:64-70 without the device->host sync).
 * flags: bit0 nearest_filter, bit1 classify_filter, bit2 return_score_type=='max'.
 */
typedef struct {
  float merge_th, gt_alpha, refine_th;
  int32_t flags;
} ptb_refine_cfg;

/* ---------------------------------------------------------------------------------------------------------
 * a8  grid-cell ("neighbour index") bags: GridPtFeatGenerator.generate + GridCirclesPtFeatGenerator.get_chosen_neighbours
 *     (cpr_head.py:296-350, 418-444), num_refine == 1.
 * Bag of GT g = [cells whose centre (j*stride + stride/2, i*stride + stride/2) lies within radius_px of the GT, row-major |
 *                zero padding up to max_pos_num + 1 slots | the GT centre], Kt = max_pos_num + 2 slots.
 *   out_feats [G][Kt][C]  exact copies of the map's cell vectors, zeros in the padding, bilinear sample for the centre
 *   out_pts   [G][Kt][3]  (x, y, stride); zeros in the padding
 *   out_valid [G][Kt]     1 for filled cell slots and the centre (not tested against pad_shape: cpr_head.py:329)
 *   out_cell  [G][Kt]     int32 linear cell index i*W + j of the slot (the neighbour index; bit-exact target),
 *                         -1 = padding, -2 = the centre sample
 *   overflow  device int32 set to 1 if some GT has more than max_pos_num + 1 chosen cells (the reference raises there)
 * Any output pointer may be NULL.  map is channels-last [B][H][W][ld], C % 4 == 0. */
int ptb_cpr_grid_bag(const float* map, int B, int H, int W, int C, int ld, const float* centers /*[G][2]*/,
                     const int32_t* bag_img /*[G]*/, int G, float stride, float radius_px, int max_pos_num,
                     float* out_feats, float* out_pts, uint8_t* out_valid, int32_t* out_cell, int32_t* overflow,
                     void* stream);
/* backward of the above w.r.t. the map: grad_map [B][H][W][ld] += scatter(grad_out [G][Kt][C]) (caller zero-fills) */
int ptb_cpr_grid_bag_bwd(const float* grad_out, int B, int H, int W, int C, int ld, const float* centers,
                         const int32_t* bag_img, const int32_t* cell_idx /*[G][Kt] from the forward*/, int G, int Kt,
                         float stride, float* grad_map, void* stream);

/* builds that CSR on the device (no host sync): groups numbered image-major / label-minor, members in ascending GT order.
 * grp_of [G], grp_ptr [G+1] (entries past the last group are filled with G), grp_idx [G].  max_per_image <= 8192. */
int ptb_label_groups(const int32_t* labels /*[G]*/, const int32_t* img_ptr /*[B+1]*/, int B, int G, int num_classes,
                     int max_per_image, int32_t* grp_of, int32_t* grp_ptr, int32_t* grp_idx, void* stream);

/* stage form: consumes materialised probabilities (bit-exact masks vs the oracle given the same probs) */
int ptb_cpr_refine(const float* bag_prob /*[G][Kt][num_classes]*/, const float* bag_pts /*[G][Kt][3]*/,
                   const uint8_t* bag_valid /*[G][Kt]*/, int G, int Kt, int K, int num_classes,
                   const int32_t* labels /*[G]*/, const int32_t* bag_img /*[G]*/, const int32_t* img_hw /*[B][2]*/,
                   const int32_t* grp_of /*[G]*/, const int32_t* grp_ptr, const int32_t* grp_idx,
                   const uint8_t* not_refine_in /*[G] or NULL*/, ptb_refine_cfg cfg,
                   float* out_pts /*[G][2]*/, float* out_score /*[G]*/, uint8_t* out_not_refine /*[G]*/,
                   uint8_t* out_chosen /*[G][Kt] or NULL*/, uint8_t* out_merge_valid /*[G][Kt] or NULL*/,
                   void* stream);

/* fused form (production): samples the class-logit map on the fly (bilinear), sigmoid, filters, merge — the
 * (G,K,num_classes) probability tensor is never written.  num_refine == 1.  Replaces CPRHead.get_bboxes'
 * extract -> get_pts_outs -> get_cls_prob -> PointRefiner chain (cpr_head.py:1248-1257). */
int ptb_cpr_refine_fused(const float* logit_map /*[B][H][W][ld]*/, int B, int H, int W, int num_classes, int ld,
                         const float* centers /*[G][2]*/, const int32_t* labels, const int32_t* bag_img, int G,
                         const float* offsets /*[K][2]*/, int K, float stride,
                         float reach_px /* max_k |offsets[k]| (e.g. radius*stride), 0 = unknown: selects the shared-memory window
                                           of 2*ceil(reach/stride)+2 cells per side that one TMA box stages per GT */,
                         const int32_t* pad_hw, const int32_t* img_hw,
                         const int32_t* grp_of, const int32_t* grp_ptr, const int32_t* grp_idx,
                         const uint8_t* not_refine_in, ptb_refine_cfg cfg,
                         float* out_pts, float* out_score, uint8_t* out_not_refine,
                         uint8_t* out_chosen /*[G][K] or NULL*/, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * MIL bag loss — replaces MILLoss.forward (mmdet/models/losses/multi_instance_learning_loss.py:153-203,
 * binary_ins=False, gfocal) on bags whose cls/ins logits are given as [G][Kt][ld] rows (cls at column 0,
 * ins at column ins_off).  weight[g][k] = valid * gt_weight (cpr_head.py:1211).
 *   out_bag_prob[g][c] = sum_k sigmoid(cls) * normalize_L1(softmax_k(ins) * weight)
 *       (the buffer must hold G*num_classes + 3*G floats: the trailing 3*G are per-bag loss / weight / hit scratch)
 *   out_loss_sum[0]   += sum_g gfocal(bag_prob[g], onehot(labels[g])) * (any_k weight>0)      (un-normalised)
 *   out_stats[0] += #bags with any weight>0 ; out_stats[1] += #bags whose argmax == label
 * bwd: d(loss_sum)/d(cls logits), d/d(ins logits) scaled by `scale` (= loss_weight / num_sample).
 */
int ptb_mil_loss_fwd(const float* logits /*[G][Kt][ld]*/, int G, int Kt, int num_classes, int ld, int ins_off,
                     const float* weight /*[G][Kt]*/, const int32_t* labels, float eps,
                     float* out_bag_prob /*[G][num_classes]*/, float* out_loss_sum /*[1]*/, float* out_stats /*[2]*/,
                     float* out_mt /*[G][num_classes][2] = (max_k ins, 1/T or 0 if the L1-normalisation clamp is active) or NULL:
                                     what ptb_cpr_loss_bwd_map needs of the forward*/,
                     void* stream);
int ptb_mil_loss_bwd(const float* logits, int G, int Kt, int num_classes, int ld, int ins_off,
                     const float* weight, const int32_t* labels, float eps, const float* bag_prob,
                     const float* scale /*[1] device scalar*/, float* grad_logits /*[G][Kt][ld], cls+ins columns written*/,
                     void* stream);

/* Fused bag gather + MIL forward (ring bags, num_classes <= 128): samples the [cls | ins] logit map (columns 0.. and ins_off..) at every
 * bag point like ptb_cpr_bag_gather, writes the sampled rows (out_bag_logits [G][K][ld], needed by the backward), the sample validity
 * as weights (out_weight [G][K] = 0/1), and evaluates ptb_mil_loss_fwd on the fly with online softmax accumulators: the (G,K,ld) tensor
 * is written once and never re-read by the forward.  out_bag_prob needs G*num_classes + 3*G floats like ptb_mil_loss_fwd. */
int ptb_cpr_bag_mil_fwd(const float* logit_map /*[B][H][W][ld]*/, int B, int H, int W, int ld, int num_classes, int ins_off,
                        const float* centers, const int32_t* bag_img, int G, const float* offsets, int K, float stride,
                        const int32_t* pad_hw, const int32_t* labels, float eps, float* out_bag_logits, float* out_weight,
                        float* out_bag_prob, float* out_loss_sum /*[1]*/, float* out_stats /*[2]*/, float* out_mt /*[G][N][2] or NULL*/,
                        void* stream);

/* Backward of the whole CPR training loss w.r.t. the LOGIT MAP in one deterministic kernel (gather formulation, no atomics on global
 * memory): replaces autograd of MILLoss (multi_instance_learning_loss.py:153-203), of the gt / neg gfocal terms (cpr_head.py:1159-1184,
 * 1219-1228) and of grid_sample (cpr_head.py:73-93) for ring bags.
 *   grad_map[b][y][x][ch] = sum_{bag g of image b, sample k, tap t on (y,x)} w_t * dLoss/d bag_logits[g][k][ch]
 *                         + [ch < num_classes] scale_neg * neg_mask * d gfocal(sigmoid(logit_map), 0)           (if logit_map != NULL)
 * with dLoss/d bag_logits from scale_mil (MIL term; needs bag_prob, mil_mt, label_weight = the trailing [G..2G) aux floats of
 * ptb_mil_loss_fwd's out_bag_prob buffer) and scale_gt * valid_center (gt term on the centre sample k = K-1).  Every element of
 * grad_map is written (no zero-init needed).  One CTA per 8x8-cell tile; every sum is formed by one thread in a fixed order, so the
 * result is bit-identical run to run.  ld must be a multiple of 32 and at most 160; K <= 320. */
int ptb_cpr_loss_bwd_map(const float* bag_logits /*[G][K][ld]*/, const float* weight /*[G][K]*/, const float* mil_mt /*[G][N][2]*/,
                         const float* bag_prob /*[G][N]*/, const float* label_weight /*[G]*/, const int32_t* labels,
                         const float* centers /*[G][2]*/, const int32_t* img_ptr /*[B+1]*/, const float* offsets /*[K][2]*/,
                         int B, int H, int W, int G, int K, int num_classes, int ins_off, int ld, float stride, float reach_px, float eps,
                         const float* scale_mil /*[1] or NULL*/, const float* scale_gt /*[1] or NULL*/,
                         const float* valid_center /*[G] or NULL*/, const float* logit_map /*[B][H][W][ld] or NULL*/,
                         const uint8_t* neg_mask /*[B][H][W][N]*/, const float* scale_neg /*[1]*/,
                         void* workspace /*ptb_cpr_loss_bwd_map_workspace(G, N) bytes, 16-byte aligned*/,
                         float* grad_map /*[B][H][W][ld]*/, void* stream);
uint64_t ptb_cpr_loss_bwd_map_workspace(int G, int num_classes);
/* Scatter form of the MIL + gt part of the same gradient (fastest; fp32 vector atomics, so NOT bit-reproducible): one CTA per bag adds
 * w_tap * dLoss/d bag_logits straight into grad_map, which the caller has initialised (zeros, or the neg-loss term written by
 * ptb_gfocal_sigmoid_bwd).  Same inputs as ptb_cpr_loss_bwd_map except bag_img [G] instead of img_ptr; workspace as above. */
int ptb_cpr_loss_bwd_scatter(const float* bag_logits, const float* weight, const float* mil_mt, const float* bag_prob,
                             const float* label_weight, const int32_t* labels, const float* centers, const int32_t* bag_img,
                             const float* offsets, int B, int H, int W, int G, int K, int num_classes, int ins_off, int ld,
                             float stride, float eps, const float* scale_mil, const float* scale_gt, const float* valid_center,
                             void* workspace, float* grad_map /*[B][H][W][ld], accumulated into*/, void* stream);

/* gfocal on sigmoid(logits) vs a one-hot / all-zero target with per-element weights — replaces
 * MILLoss.gfocal_loss (multi_instance_learning_loss.py:148-151) as used for gt_loss and neg_loss
 * (cpr_head.py:1159-1184, 1219-1228).  rows: logits[m*row_stride + c], c<num_classes;
 * target_label[m] in [0,num_classes) or -1 (all-zero target); weight is uint8 [M][num_classes] (wmode 0),
 * float [M] (wmode 1) or NULL (all ones).  loss_sum[0] += sum.   bwd: grad = scale[0] * dloss/dlogit (overwrite or add). */
int ptb_gfocal_sigmoid_fwd(const float* logits, int64_t M, int num_classes, int64_t row_stride,
                           const int32_t* target_label, const void* weight, int wmode, float eps,
                           float* loss_sum, void* stream);
int ptb_gfocal_sigmoid_bwd(const float* logits, int64_t M, int num_classes, int64_t row_stride,
                           const int32_t* target_label, const void* weight, int wmode, float eps,
                           const float* scale, float* grad, int64_t grad_row_stride, int accumulate, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * P2P decode + top-k — replaces P2PHead.get_pred_points (p2p_head.py:125-170) and the per-level
 * max-over-classes + topk(nms_pre) of _get_bboxes_single (p2p_head.py:362-376).
 * cls_map [B][H][W][k*C] logits, reg_map [B][H][W][2k]; proposal index q = (i*W+j)*k + a.
 *   out_topk_idx[b][r]  = index of the r-th largest max_c sigmoid(cls[q][c]) (ties: lower index first)
 *   out_pts[b][r]       = clamp(anchor + reg*gamma*stride, [0,img_w]x[0,img_h])   (optionally / scale_factor)
 *   out_scores[b][r][c] = sigmoid(cls[topk][c])
 * nms_pre >= number of proposals keeps every proposal in index order (reference skips top-k then).
 */
int ptb_p2p_decode_topk(const float* cls_map, const float* reg_map, int B, int H, int W, int num_classes, int k,
                        const float* point_anchor /*[k][2]*/, float stride, float pts_gamma,
                        const int32_t* img_hw, const float* scale_xy /*[B][2] or NULL*/, int nms_pre,
                        int32_t* out_topk_idx /*[B][P]*/, float* out_pts /*[B][P][2]*/, float* out_scores /*[B][P][C]*/,
                        void* workspace, uint64_t workspace_bytes, void* stream);
uint64_t ptb_p2p_decode_topk_workspace(int B, int H, int W, int k);

/* ------------------------------------------------------------------------------------------------------------------
 * multiclass NMS — replaces multiclass_nms (mmdet/core/post_processing/bbox_nms.py:7-94) and the third-party
 * mmcv.ops.nms.batched_nms it calls (mmcv-full 1.3.x, not vendored; semantics restated in oracle/p2p.py).
 * Per image b: candidates = (point p, class c) with scores[b][p][c] > score_thr, flat id = p*C+c, in flat order;
 * box = pts[p] -/+ pseudo_wh/2 offset by c*(max_coord+1);  greedy NMS by descending score (ties: lower flat id first),
 * suppress IoU > iou_thr;  keep the first max_per_img.
 *   out_count[b], out_det[b][r] = (x1,y1,x2,y2,score), out_label[b][r], out_keep[b][r] = index into the candidate list,
 *   out_cand_count[b] = number of candidates.
 */
int ptb_multiclass_nms(const float* pts /*[B][P][2]*/, const float* scores /*[B][P][C]*/, int B, int P, int num_classes,
                       float pseudo_w, float pseudo_h, float score_thr, float iou_thr, int max_per_img,
                       int32_t* out_count /*[B]*/, float* out_det /*[B][max][5]*/, int32_t* out_label /*[B][max]*/,
                       int32_t* out_keep /*[B][max]*/, int32_t* out_cand_count /*[B]*/,
                       void* workspace, uint64_t workspace_bytes, void* stream);
uint64_t ptb_multiclass_nms_workspace(int B, int P, int num_classes);
/* same with explicit boxes [B][P][4] (x1,y1,x2,y2) instead of point pseudo-boxes: the second NMS of the test-time-aug /
 * tile merge path (P2PHead.aug_test_bboxes, p2p_head.py:487-572; dense_test_mixins.py:173-204). */
int ptb_multiclass_nms_boxes(const float* boxes /*[B][P][4]*/, const float* scores /*[B][P][C]*/, int B, int P, int num_classes,
                             float score_thr, float iou_thr, int max_per_img,
                             int32_t* out_count, float* out_det, int32_t* out_label, int32_t* out_keep, int32_t* out_cand_count,
                             void* workspace, uint64_t workspace_bytes, void* stream);

/* soft-NMS variant (nms=dict(type='soft_nms', iou_threshold, sigma=0.5, min_score=1e-3, method='linear'|'gaussian'|'naive') through
 * batched_nms; mmcv.ops.nms.soft_nms is third-party (mmcv-full 1.3.x) — its published CPU kernel is restated in
 * oracle/p2p.py::soft_nms; no reference test pins it: parity unpinned).  Same candidate list, class offset and outputs as
 * ptb_multiclass_nms, but out_det[..][4] is the DECAYED score and the order is the soft-NMS selection order (non-increasing decayed
 * score).  Give either pts (pseudo boxes) or boxes.  method: 0 naive, 1 linear, 2 gaussian.
 * Images whose classes are not separated by the class offset (negative coordinates on near-square images) take an exact global
 * path, like ptb_multiclass_nms. */
int ptb_multiclass_soft_nms(const float* pts /*[B][P][2] or NULL*/, const float* boxes /*[B][P][4] or NULL*/,
                            const float* scores /*[B][P][C]*/, int B, int P, int num_classes, float pseudo_w, float pseudo_h,
                            float score_thr, float iou_thr, float sigma, float min_score, int method, int max_per_img,
                            int32_t* out_count, float* out_det, int32_t* out_label, int32_t* out_keep, int32_t* out_cand_count,
                            void* workspace, uint64_t workspace_bytes, void* stream);
uint64_t ptb_multiclass_soft_nms_workspace(int B, int P, int num_classes);

/* ------------------------------------------------------------------------------------------------------------------
 * Hungarian cost matrix — replaces FocalLossCost + DisCostV2 (mmdet/core/bbox/match_costs/match_cost.py:94-99,
 * 197-214) as summed by HungarianAssignerV2.assign (hungarian_assigner.py:222-227).
 *   cost[q][g] = w_cls*(pos(p)-neg(p)) at column labels[g] + w_dis * sum_d |pts[q][d]/f_d - gts[g][d]/f_d|
 * rows = the n_rows proposals listed in row_idx (the valid ones), written densely [n_rows][n_gt].
 */
int ptb_p2p_cost_matrix(const float* cls_logits /*[Q][C]*/, const float* pts /*[Q][ldp]*/, int ldp,
                        const int32_t* row_idx /*[n_rows] or NULL*/, int n_rows, int num_classes,
                        const float* gts /*[n_gt][2]*/, const int32_t* gt_labels, int n_gt,
                        float w_cls, float alpha, float gamma, float eps, float w_dis, float fx, float fy,
                        float* cost, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * RPN proposals for dense anchors — replaces RPNHead._get_bboxes (mmdet/models/dense_heads/rpn_head.py:78-186) with the grid
 * anchors of AnchorGenerator (mmdet/core/anchor/anchor_generator.py:207-270), DeltaXYWHBBoxCoder.decode
 * (mmdet/core/bbox/coder/delta_xywh_bbox_coder.py:144-270, clip_border=True) and mmcv batched_nms over level ids, for a batch.
 *   cls_scores[l] : device (B, A, H_l, W_l) NCHW logits (use_sigmoid_cls);  bbox_preds[l] : device (B, 4A, H_l, W_l)
 *   level_hw      : HOST [L][2] (H_l, W_l);  strides_wh : HOST [L][2] (stride_w, stride_h);  base_anchors : DEVICE [L][A][4]
 *   img_hw        : DEVICE [B][2] = img_shape (h, w) -> clip range;  means, stds : HOST [4]
 *   per level: sigmoid, top-nms_pre by (score desc, anchor index asc) when the level has more than nms_pre anchors (else all, in
 *   index order), decode, clip;  then drop boxes with w <= min_bbox_size or h <= min_bbox_size (min_bbox_size < 0: keep all),
 *   greedy NMS (IoU > iou_thr) per level on coordinates offset by level*(boxes.max()+1), merge by descending score, first max_per_img.
 *   out_det [B][max_per_img][5] (x1,y1,x2,y2,score), out_count[B], out_level[B][max_per_img];
 *   optional (may be NULL): out_pos [B][max_per_img] position in the candidate list, out_cand_box [B][Ptot][4] (16-byte aligned),
 *   out_cand_score [B][Ptot], out_cand_idx [B][Ptot] (anchor index q = (y*W+x)*A + a inside its level), Ptot = sum_l min(nms_pre, H_l*W_l*A).
 * Limits: L <= 8, nms_pre <= 4096 (every level keeps <= 4096 candidates), max_per_img <= 2048.
 */
uint64_t ptb_rpn_proposals_workspace(const int32_t* level_hw, int L, int B, int A, int nms_pre, int max_per_img);
int ptb_rpn_proposals(const float* const* cls_scores, const float* const* bbox_preds, const int32_t* level_hw,
                      const int32_t* strides_wh, const float* base_anchors, int L, int B, int A, const int32_t* img_hw,
                      const float* means, const float* stds, float wh_ratio_clip, int nms_pre, float min_bbox_size,
                      float iou_thr, int max_per_img, int32_t* out_count, float* out_det, int32_t* out_level,
                      int32_t* out_pos, float* out_cand_box, float* out_cand_score, int32_t* out_cand_idx,
                      void* workspace, uint64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * HungarianAssignerV2 matching — replaces `cost.detach().cpu()` + the <= topk_k scipy.optimize.linear_sum_assignment solves of
 * HungarianAssignerV2.assign (mmdet/core/bbox/assigners/hungarian_assigner.py:229-270) for a whole batch, without a host
 * round trip.  scipy's algorithm (rectangular_lsap: shortest augmenting paths, fp64 duals, transpose rule, tie rule) is
 * restated bit-for-bit (oracle/lsap.c is pinned to scipy; pointtinybenchmark_b200/csrc/lsap_core.cuh is the parallel form, one CTA per
 * image; csrc/lsap_cluster.cuh solves an image on a cluster of 8 / 6 / 5 CTAs — the default up to 17 600 columns x 1024 rows).
 *   cost      : concatenated per-image cost matrices, image b = [N_b][n_b] fp32 row-major (proposals x GTs, as the reference
 *               builds it) at element offset desc[b][0]
 *   desc      : DEVICE int64 [num_images][6] = {cost_off, workspace byte offset (multiple of 8), gt_inds element offset,
 *               row_idx element offset or -1, N_b, n_b}
 *   row_idx   : optional map from the cost row to the slot inside the image's gt_inds slice (the valid proposals)
 *   gt_inds   : int64, PRE-ZEROED by the caller; matched proposals receive gt index + 1 (`assigned_gt_inds`)
 *   workspace : >= sum of ptb_hungarian_v2_workspace(N_b, n_b) bytes
 *   status    : DEVICE int32 [num_images], PRE-ZEROED; 0 ok, 1 = scipy's "cost matrix is infeasible",
 *               2 = scipy's "matrix contains invalid numeric entries" (NaN / -inf), 3 = internal error
 *   topk_k    : 1 = one solve (any orientation); > 1 = rounds on the still-unassigned proposals while they are >= n_b
 */
uint64_t ptb_hungarian_v2_workspace(int N, int n);
int ptb_hungarian_v2_batch(const float* cost, const int64_t* desc, int num_images, int max_N, int max_n, int topk_k,
                           const int32_t* row_idx, int64_t* gt_inds, void* workspace, int32_t* status, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * PointAssigner — replaces PointAssigner.assign (mmdet/core/bbox/assigners/point_assigner.py:23-133).
 * points [N][3] (x,y,stride), gts [n][4];  out_gt_inds[N] (0 = background, j+1 = gt j), int64 like the reference.
 */
int ptb_point_assigner(const float* points, int N, const float* gt_bboxes, int n, float scale, int pos_num,
                       int64_t* out_gt_inds, void* workspace, uint64_t workspace_bytes, void* stream);
uint64_t ptb_point_assigner_workspace(int N, int n);

/* elementwise P2P losses — replace FocalLoss (mmdet/models/losses/focal_loss.py:11-56 formula) and SmoothL1Loss
 * (smooth_l1_loss.py:25-31) as used by P2PHead.loss_single (p2p_head.py:220-248). sums are atomically added. */
int ptb_sigmoid_focal_fwd_bwd(const float* logits /*[M][C]*/, const int64_t* labels /*[M], ==C: background*/,
                              const float* weight /*[M]*/, int64_t M, int num_classes, float gamma, float alpha,
                              float* loss_sum /*[1]*/, const float* scale /*[1] or NULL*/, float* grad /*[M][C] or NULL*/,
                              void* stream);
int ptb_smooth_l1_fwd_bwd(const float* pred /*[M][2]*/, const float* target, const float* weight /*[M][2]*/, int64_t M,
                          float inv_norm /* 1/(stride*reg_norm) */, float beta,
                          float* loss_sum, const float* scale, float* grad /*[M][2] or NULL*/, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Conv towers on the tensor cores — replace the cuDNN calls behind CPRHead.forward_single / P2PHead.forward_single
 * (cpr_head.py:983-995,1033-1043; p2p_head.py:82-97,113-123): ConvModule = conv3x3(256 out, no bias) + GroupNorm + ReLU.
 * fp32-accurate 3xTF32 implicit GEMM (tcgen05.mma kind::tf32, TMA-staged operands, TMEM accumulators).
 *   ptb_split_tf32           x -> hi (13 low mantissa bits cleared) + lo (= x - hi, exact)
 *   ptb_conv3x3_pack_weight  nn.Conv2d weight [Cout][Cin][3][3] -> [Cout][tap][Cin] as hi / lo
 *   ptb_conv3x3_c256_tf32x3  y[b][h][w][0..256) = sum_{tap,ci} x[b][h+kh-1][w+kw-1][ci] * w[co][tap][ci]  (zero padding);
 *                            gn_stats (optional, zero-initialised by the caller) [B][32][2] fp64 += per-(image, group of 8
 *                            channels) sum / sum of squares of y
 *   ptb_gn_relu_apply        out = relu((y-mean)*rstd*gamma+beta) from those statistics, written as fp32 (out_lo == NULL)
 *                            or directly as the hi/lo pair the next conv consumes
 */
int ptb_split_tf32(const float* x, int64_t n, float* hi, float* lo, void* stream);
int ptb_conv3x3_pack_weight(const float* w_oihw, int Cout, int Cin, float* w_hi, float* w_lo, void* stream);
int ptb_conv3x3_c256_tf32x3(const float* x_hi, const float* x_lo /*[B][H][W][Cin]*/, const float* w_hi, const float* w_lo,
                            int B, int H, int W, int Cin, float* y /*[B][H][W][256]*/, double* gn_stats, void* stream);
int ptb_gn_relu_apply(const float* y, const double* gn_stats, const float* gamma, const float* beta, int B, int HW, int C,
                      int groups, float eps, int relu, float* out_hi, float* out_lo, void* stream);
/* Same tower at HALF the tensor-pipe time: two-term fp16 split  x*scale = h + l  (22 significant bits), three
 * tcgen05.mma.kind::f16 per k-step (h*h + l*h + h*l), fp32 accumulate.  Operands are IEEE fp16 arrays (void* = __half*).
 *   ptb_split_f16: auto_scale != 0 picks a power-of-two scale from max|x| ON THE DEVICE (workspace: 4 bytes) and writes
 *                  its inverse to dev_inv_scale (a device float), else scale = 1.
 *   ptb_conv3x3_pack_weight_f16: weights * scale (a power of two chosen by the caller) as h / l.
 *   ptb_conv3x3_c256_f16x2: y = conv * out_scale * (*dev_out_scale if given): undoes the operand scales exactly.
 *   ptb_gn_relu_apply_f16: GroupNorm(+ReLU) written as the (h, l) pair of the next conv (scale 1); |out| > 60000 is clamped
 *                  and *overflow_flag set (cannot happen for a GroupNorm output with sane affine parameters).
 */
int ptb_split_f16(const float* x, int64_t n, int auto_scale, void* hi, void* lo, float* dev_inv_scale, void* workspace, void* stream);
int ptb_conv3x3_pack_weight_f16(const float* w_oihw, int Cout, int Cin, float scale, void* w_h, void* w_l, void* stream);
int ptb_conv3x3_c256_f16x2(const void* x_h, const void* x_l, const void* w_h, const void* w_l, int B, int H, int W, int Cin,
                           float out_scale, const float* dev_out_scale, float* y, double* gn_stats, void* stream);
/* General form of the same kernel for the head's other GEMMs: taps = 1 (the per-cell Linear cls_out / ins_out of CPRHead,
 * cpr_head.py:1008-1014) or 9 (P2PHead's cls_out / reg_out conv3x3 WITH bias, p2p_head.py:98-102), n_out <= 256 output
 * channels, MMA N = n_mma (multiple of 16 >= n_out; the packed weight has zero rows beyond n_out), bias added in the
 * epilogue, output row stride ldy. */
int ptb_conv_tc_pack_weight_f16(const float* w /*[n_out][Cin][taps]*/, int n_out, int n_mma, int Cin, int taps, float scale,
                                void* w_h, void* w_l, void* stream);
int ptb_conv_tc_f16x2(const void* x_h, const void* x_l, const void* w_h, const void* w_l, int B, int H, int W, int Cin, int taps,
                      int n_out, int n_mma, float out_scale, const float* dev_out_scale, const float* bias, float* y, int ldy,
                      void* stream);
int ptb_gn_relu_apply_f16(const float* y, const double* gn_stats, const float* gamma, const float* beta, int B, int HW, int C,
                          int groups, float eps, int relu, void* out_h, void* out_l, int* overflow_flag, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Dense-anchor assignment (SURVEY.md §8f rank 4, BASELINE.json configs[3]): MaxIoUAssigner.assign
 * (mmdet/core/bbox/assigners/max_iou_assigner.py:60-212) over BboxOverlaps2D (iou_calculators/iou2d_calculator.py:211-256)
 * without materialising the (k, n) IoU matrix.  Boxes are [.][4] fp32 (x1,y1,x2,y2), 16-byte aligned.
 *   out_gt_inds[i]      int64: -1 ignored / between thresholds, 0 negative, g+1 assigned to GT g          (bit-exact target)
 *   out_max_overlaps[i] max IoU of anchor i over the GTs (-1 for anchors hit by gt_bboxes_ignore)
 *   out_labels[i]       int64 gt_labels[g] for positives, -1 otherwise (NULL to skip)
 * neg_iou_lo/hi: a float neg_iou_thr t is (0, t); a tuple (a, b) is (a, b).  ignore_iof_thr <= 0 or no ignore boxes: no ignoring;
 * ignore_wrt_candidates selects which box's area normalises the IoF (max_iou_assigner.py:109-116).
 * ptb_bbox_overlaps writes the matrix itself (mode_iof: 0 IoU, 1 IoF w.r.t. boxes1). */
uint64_t ptb_max_iou_assign_workspace(int N, int n_gt);
int ptb_max_iou_assign(const float* bboxes, int N, const float* gt_bboxes, int n_gt, const int32_t* gt_labels /*or NULL*/,
                       const float* gt_bboxes_ignore /*or NULL*/, int n_ignore, float pos_iou_thr, float neg_iou_lo, float neg_iou_hi,
                       float min_pos_iou, int gt_max_assign_all, int match_low_quality, float ignore_iof_thr, int ignore_wrt_candidates,
                       int64_t* out_gt_inds, float* out_max_overlaps, int64_t* out_labels, void* workspace, uint64_t workspace_bytes,
                       void* stream);
int ptb_bbox_overlaps(const float* boxes1, int m, const float* boxes2, int n, int mode_iof, float* out /*[m][n]*/, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Tower backward (autograd of CPRHead.forward_single / P2PHead.forward_single, cpr_head.py:1033-1043, p2p_head.py:113-123;
 * the reference gets it from ATen/cuDNN autograd).  Per ConvModule, in reverse order:
 *   ptb_gn_relu_bwd          da (grad of the ReLU output) + saved conv output y + epilogue statistics -> dy (fp32), dgamma, dbeta,
 *                            max|dy| as float bits (device) for the operand scale.  Deterministic (no fp atomics).
 *   ptb_split_f16_amax       dy -> fp16 (h, l) pair with the power-of-two scale derived from that device max; 1/scale -> dev_inv_scale
 *   ptb_conv_tc_f16x2        dgrad: the forward kernel on (dy pair, weights transposed + flipped and packed by the host layer)
 *   ptb_conv3x3_wgrad_f16x2  dW[co][ci][3][3] (+)= scale * s_dy * s_x * sum_pixels dy (x) x_shifted  on tcgen05 with MN-major operands
 * All tensors channels-last; C = 256 for the tensor-core kernels.
 */
uint64_t ptb_gn_relu_bwd_workspace(int B, int HW, int C, int groups);
int ptb_gn_relu_bwd(const float* da, const float* y, const double* gn_stats, const float* gamma, const float* beta, int B, int HW, int C,
                    int groups, float eps, int relu, void* workspace, float* dy, float* dgamma /*[C] or NULL*/,
                    float* dbeta /*[C] or NULL*/, unsigned int* amax_bits /*device, or NULL*/, void* stream);
int ptb_split_f16_amax(const float* x, int64_t n, const unsigned int* dev_amax_bits, void* hi, void* lo, float* dev_inv_scale,
                       void* stream);
uint64_t ptb_conv3x3_wgrad_workspace(int B, int H, int W);
int ptb_conv3x3_wgrad_f16x2(const void* dy_h, const void* dy_l, const void* x_h, const void* x_l, int B, int H, int W, int Cout, int Cin,
                            float scale, const float* dev_scale_dy /*or NULL*/, const float* dev_scale_x /*or NULL*/, void* workspace,
                            float* dw /*[Cout][Cin][3][3]*/, int accumulate, void* stream);

/* The same kernel for any channels-last GEMM with K = pixels:  dW[co][ci][tap] = scale * s_dy * s_x * sum_pixels dy[p][co] * x[p + tap][ci]
 * with taps = 9 (conv3x3, pad 1) or taps = 1 (conv1x1 / per-cell Linear: the weight gradient of CPRHead's cls_out / ins_out logit map,
 * cpr_head.py:1045-1078 under autograd), Cin = 256, Cout a multiple of 8 up to 256 (rows beyond Cout are never written).
 * dw is [Cout][256][taps] fp32.  Deterministic (fixed-order reduction of the pixel splits). */
uint64_t ptb_conv_tc_wgrad_workspace(int B, int H, int W, int taps);
int ptb_conv_tc_wgrad_f16x2(const void* dy_h, const void* dy_l /*[B][H][W][Cout] fp16*/, const void* x_h, const void* x_l /*[B][H][W][256] fp16*/,
                            int B, int H, int W, int Cout, int Cin, int taps, float scale, const float* dev_scale_dy,
                            const float* dev_scale_x, void* workspace, float* dw, int accumulate, void* stream);

/* column sums of a row-major fp32 matrix: out[n] = sum_m y[m][n] (bias gradient of the logit-map Linear); fixed-order, deterministic */
uint64_t ptb_col_sum_workspace(int64_t M, int N);
int ptb_col_sum(const float* y /*[M][ld]*/, int64_t M, int N, int ld, float* workspace, float* out /*[N]*/, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * R-CNN box stage (StandardRoIHead.simple_test_bboxes with SingleRoIExtractor + Shared2FCBBoxHead; roi_heads/test_mixins.py:50-130,
 * single_level_roi_extractor.py:34-100, bbox_head.py:310-435).
 *   ptb_amax_abs          max|x| of an fp32 tensor as float bits into *dev_amax_bits (atomicMax over non-negative floats); accumulate = 0
 *                         zeroes it first, 1 keeps the running max (several levels into one bound).
 *   ptb_roi_align         rois (M, 5) [batch_idx, x1, y1, x2, y2]; L <= 5 channels-last fp32 level maps (B, H_l, W_l, C), C % 32 == 0,
 *                         given as host arrays feats[L], hw[2L] (H, W), spatial_scales[L].  Level per RoI = map_roi_levels (finest_scale;
 *                         L == 1: level 0), mmcv RoIAlign avg pooling (aligned: offset 0.5, else roi size >= 1; sampling_ratio 0 = adaptive).
 *                         Exactly one output mode: out (M, out_h, out_w, C) fp32, or out_h16 / out_l16 (M_pad, out_h*out_w*C) fp16 pair of
 *                         x * s with s the power-of-two scale of ptb_split_f16_amax taken from *dev_amax_bits (1/s -> *dev_inv_scale;
 *                         rows M .. M_pad-1 are zero).  out_level (M,) int8 optional (-1: NaN scale, features zero).
 *   ptb_relu_split_f16    y (rows, ld) fp32 -> fp16 pair of relu(y[:, :n]) at unit scale; values above 60000 are clamped and raise
 *                         *overflow_flag (optional).
 *   ptb_rcnn_bbox_decode  rois (B * n_per_img, 5), logits cls (rows, ldc) with N + 1 columns, deltas reg (rows, ldr) with 4N columns:
 *                         mask_padding zeroes logits and deltas of all-zero RoIs (the batch padding of simple_test_bboxes); softmax;
 *                         class-specific delta2bbox (means, stds, wh_ratio_clip) clipped to img_hw (B, 2) int32 (h, w); rescale by
 *                         scale_factor (B, 4) when given.  out_boxes (rows, 4N); out_scores (rows, N + 1) and out_cand_scores
 *                         (rows * N, N): the candidate (RoI i, class k) has its score in column k and -inf elsewhere, the input of
 *                         ptb_multiclass_nms_boxes with P = n_per_img * N.  Both optional.
 */
int ptb_amax_abs(const float* x, int64_t n, unsigned int* dev_amax_bits, int accumulate, void* stream);
int ptb_roi_align(const float* rois, int M, int M_pad, const void* const* feats, const int32_t* hw, const float* spatial_scales, int L, int B,
                  int C, int out_h, int out_w, int sampling_ratio, int aligned, float finest_scale, const unsigned int* dev_amax_bits,
                  float* out, void* out_h16, void* out_l16, float* dev_inv_scale, int8_t* out_level, void* stream);
int ptb_relu_split_f16(const float* y, int rows, int n, int ld, void* out_h, void* out_l, int* overflow_flag, void* stream);
int ptb_rcnn_bbox_decode(const float* rois, int B, int n_per_img, const float* cls, int ldc, const float* reg, int ldr, int num_classes,
                         int mask_padding, const float* means /*host [4]*/, const float* stds /*host [4]*/, float wh_ratio_clip,
                         const int32_t* img_hw, const float* scale_factor /*or NULL*/, float* out_boxes, float* out_scores /*or NULL*/,
                         float* out_cand_scores /*or NULL*/, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PTB_B200_H_ */
