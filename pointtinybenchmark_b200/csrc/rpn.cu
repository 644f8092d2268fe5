// RPN proposal path for dense anchors (SURVEY.md §8f rank 4, BASELINE.json configs[3]) — replaces RPNHead._get_bboxes
// (mmdet/models/dense_heads/rpn_head.py:78-186) together with the anchors it is fed (AnchorGenerator.grid_anchors,
// mmdet/core/anchor/anchor_generator.py:207-270), DeltaXYWHBBoxCoder.decode (mmdet/core/bbox/coder/delta_xywh_bbox_coder.py:144-270)
// and the third-party mmcv batched_nms (restated in oracle/p2p.py).  One call per batch, all images and levels:
//
//   rpn_score_kernel      per level: key[b][q] = sigmoid(cls[b][a][y][x]),  q = (y*W + x)*A + a  (the reference's permute(0,2,3,1))
//   p2p_select_kernel     per level, CTA per image: exact top-nms_pre by (score desc, index asc)        (topk_select.cuh)
//   rpn_decode_kernel     per level, thread per candidate: grid anchor = base[a] + (x*sw, y*sh, x*sw, y*sh) computed on the fly (the
//                         81 840 x 4 anchor tensor is never materialised), delta2bbox in the reference's fp32 operation order,
//                         clip to img_shape; writes the concatenated candidate list [B][Ptot] (boxes, scores, anchor index)
//   rpn_nms_prepare_kernel CTA per image: min_bbox_size mask, boxes.max() over the surviving candidates (the batched_nms offset unit)
//   rpn_nms_level_kernel  CTA per (level, image): sort by (score desc, position asc), greedy IoU > thr suppression on the level-offset
//                         fp32 coordinates (bit-identical IoU to the reference), <= max_per_img kept per level
//                         (round 2: rpn_nms_level_bitmask_kernel — suppression bit matrix over the whole CTA + a find-first-set walk —
//                         whenever every level keeps <= 1024 candidates; the serial kernel remains for larger nms_pre)
//   rpn_nms_merge_rank_kernel CTA per image: output rank of every kept entry by binary searches in the other levels' sorted lists
//                         -> dets[:max_per_img] in descending score order
//
// Levels are disjoint after the level offset because every candidate box is clipped to [0, img_w] x [0, img_h] (>= 0), so the
// joint greedy NMS of the reference decomposes per level exactly.  Everything here is latency / HBM-scan work (1.3 MB of logits
// per image at configs[3]); the design goal is one pass over the logits and no intermediate anchor / IoU tensors.
#include "bbox_coder.cuh"
#include "ptb_common.cuh"
#include "topk_select.cuh"
#include <math_constants.h>
#include <stdlib.h>

namespace ptb {
namespace {

constexpr int RPN_MAX_LEVELS = 8;
constexpr int RPN_T = 256;

struct RpnLevels {                 // by-value kernel argument
  int L;
  int seg_off[RPN_MAX_LEVELS + 1]; // candidate segment of level l inside one image's list
};

struct RpnImg {
  float max_coord;
  int valid_count;
};

struct RBox {
  float x1, y1, x2, y2, area;
};
__device__ __forceinline__ bool rbox_iou_gt(const RBox& a, const RBox& b, float thr) {
  const float w = fmaxf(0.f, __fsub_rn(fminf(a.x2, b.x2), fmaxf(a.x1, b.x1)));
  const float h = fmaxf(0.f, __fsub_rn(fminf(a.y2, b.y2), fmaxf(a.y1, b.y1)));
  const float inter = __fmul_rn(w, h);
  if (inter == 0.f) return false;   // exact: 0 / union is +-0 or NaN, never > thr (thr >= 0 is required by the entry point); skips the
                                    // division for the disjoint pairs, which are almost all of them
  const float ovr = __fdiv_rn(inter, __fsub_rn(__fadd_rn(a.area, b.area), inter));
  return ovr > thr;
}
__device__ __forceinline__ RBox rbox_offset(const float4 r, float off) {
  RBox b;   // + level*(max_coord+1) on every coordinate (mmcv batched_nms)
  b.x1 = __fadd_rn(r.x, off); b.y1 = __fadd_rn(r.y, off); b.x2 = __fadd_rn(r.z, off); b.y2 = __fadd_rn(r.w, off);
  b.area = __fmul_rn(__fsub_rn(b.x2, b.x1), __fsub_rn(b.y2, b.y1));
  return b;
}

__global__ void __launch_bounds__(256)
rpn_score_kernel(const float* __restrict__ cls /*[B][A][H][W]*/, int B, int A, int HW, float* __restrict__ key /*[B][HW*A]*/) {
  const long long Q = (long long)HW * A;
  for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < (long long)B * Q; e += (long long)gridDim.x * 256) {
    const long long b = e / Q;
    const long long q = e - b * Q;
    const long long cell = q / A;
    const int a = (int)(q - cell * A);
    key[e] = sigmoidf_acc(cls[(b * A + a) * HW + cell]);
  }
}

__global__ void __launch_bounds__(256)
rpn_decode_kernel(const float* __restrict__ bbox /*[B][4A][H][W]*/, const float* __restrict__ key /*[B][Q]*/,
                  const int32_t* sel /*[B][Ptot] (level segment filled; may alias cand_idx)*/, int B, int A, int H, int W,
                  const float* __restrict__ base /*[A][4]*/, float sw, float sh, DecodeCfg dc, const int32_t* __restrict__ img_hw,
                  int P, int seg, int Ptot, int identity, float4* __restrict__ cand_box, float* __restrict__ cand_score,
                  int32_t* cand_idx) {
  const long long t = (long long)blockIdx.x * 256 + threadIdx.x;
  if (t >= (long long)B * P) return;
  const int b = (int)(t / P), r = (int)(t - (long long)b * P);
  const size_t o = (size_t)b * Ptot + seg + r;
  const int q = identity ? r : sel[o];
  const int HW = H * W;
  const int cell = q / A, a = q - cell * A;
  const int y = cell / W, x = cell - y * W;
  // anchor_generator.py:256-267: shift = arange * stride (integers), anchor = base + shift (one fp32 add per coordinate)
  const float fx = __fmul_rn((float)x, sw), fy = __fmul_rn((float)y, sh);
  const float ax1 = __fadd_rn(base[4 * a], fx), ay1 = __fadd_rn(base[4 * a + 1], fy);
  const float ax2 = __fadd_rn(base[4 * a + 2], fx), ay2 = __fadd_rn(base[4 * a + 3], fy);
  const float* d = bbox + ((size_t)b * 4 * A + 4 * a) * HW + cell;
  const float mw = (float)img_hw[2 * b + 1], mh = (float)img_hw[2 * b];      // max_shape = img_shape[:2] flipped -> (w, h)
  cand_box[o] = delta2bbox_clip(ax1, ay1, ax2, ay2, d[0], d[(size_t)HW], d[2 * (size_t)HW], d[3 * (size_t)HW], dc, mw, mh);
  cand_score[o] = key[(size_t)b * HW * A + q];
  cand_idx[o] = q;
}

// CTA per image: valid = (w > min_size) & (h > min_size) (rpn_head.py:171-182), max_coord = boxes.max() over the valid ones
__global__ void __launch_bounds__(RPN_T)
rpn_nms_prepare_kernel(const float4* __restrict__ cand_box, int Ptot, float min_size, uint8_t* __restrict__ valid, RpnImg* __restrict__ hdr) {
  __shared__ float s_max[RPN_T / 32];
  __shared__ int s_cnt[RPN_T / 32];
  const int b = blockIdx.x;
  float mx = -CUDART_INF_F;
  int cnt = 0;
  for (int p = threadIdx.x; p < Ptot; p += RPN_T) {
    const float4 r = cand_box[(size_t)b * Ptot + p];
    const bool v = min_size < 0.f || (__fsub_rn(r.z, r.x) > min_size && __fsub_rn(r.w, r.y) > min_size);
    valid[(size_t)b * Ptot + p] = v;
    if (v) { mx = fmaxf(mx, fmaxf(fmaxf(r.x, r.y), fmaxf(r.z, r.w))); ++cnt; }
  }
  mx = warp_max(mx);
  cnt = warp_sum_int(cnt);
  if ((threadIdx.x & 31) == 0) { s_max[threadIdx.x >> 5] = mx; s_cnt[threadIdx.x >> 5] = cnt; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float m = s_max[0];
    int c = s_cnt[0];
    for (int w = 1; w < RPN_T / 32; ++w) { m = fmaxf(m, s_max[w]); c += s_cnt[w]; }
    hdr[b].max_coord = m;
    hdr[b].valid_count = c;
  }
}

// CTA per (level, image): kept candidate positions of this level in descending score order (<= max_keep)
__global__ void __launch_bounds__(RPN_T)
rpn_nms_level_kernel(const float4* __restrict__ cand_box, const float* __restrict__ cand_score, const uint8_t* __restrict__ valid,
                     int Ptot, RpnLevels lv, float iou_thr, int max_keep, const RpnImg* __restrict__ hdr,
                     int32_t* __restrict__ lvl_cnt /*[B][L]*/, int32_t* __restrict__ lvl_list /*[B][L][max_keep]*/,
                     unsigned long long* __restrict__ lvl_key /*[B][L][max_keep]*/) {
  __shared__ unsigned long long keys[TOPK_MAX];
  __shared__ int s_n;
  __shared__ int s_wbase[RPN_T / 32];
  extern __shared__ float kept[];     // [max_keep][5]
  const int l = blockIdx.x, b = blockIdx.y;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int seg0 = lv.seg_off[l], segn = lv.seg_off[l + 1] - seg0;
  const float4* bx = cand_box + (size_t)b * Ptot;
  const float* sc = cand_score + (size_t)b * Ptot;
  const uint8_t* vd = valid + (size_t)b * Ptot;
  if (threadIdx.x == 0) s_n = 0;
  __syncthreads();
  for (int base0 = 0; base0 < segn; base0 += RPN_T) {
    const int p = seg0 + base0 + threadIdx.x;
    const bool is = (base0 + threadIdx.x) < segn && vd[p];
    const unsigned int bal = __ballot_sync(0xffffffffu, is);
    if (lane == 0) s_wbase[wid] = atomicAdd(&s_n, __popc(bal));
    __syncwarp();
    if (is) {
      const int slot = s_wbase[wid] + __popc(bal & ((1u << lane) - 1u));
      keys[slot] = ((unsigned long long)(~__float_as_uint(sc[p])) << 32) | (unsigned int)p;      // score desc, position asc
    }
    __syncwarp();
  }
  __syncthreads();
  const int n = s_n;
  int n2 = 1;
  while (n2 < n) n2 <<= 1;
  for (int i = n + threadIdx.x; i < n2; i += RPN_T) keys[i] = 0xFFFFFFFFFFFFFFFFull;
  bitonic_sort_u64(keys, n2);
  int nk = 0;
  if (wid == 0 && n > 0) {
    const float off = __fmul_rn((float)l, __fadd_rn(hdr[b].max_coord, 1.f));
    for (int base0 = 0; base0 < n && nk < max_keep; base0 += 32) {
      const int i = base0 + lane;
      const bool have = i < n;
      const int p = have ? (int)(keys[i] & 0xFFFFFFFFull) : seg0;
      const RBox me = rbox_offset(bx[p], off);
      bool alive = have;
      for (int t = 0; t < nk && alive; ++t) {
        RBox kb;
        kb.x1 = kept[5 * t]; kb.y1 = kept[5 * t + 1]; kb.x2 = kept[5 * t + 2]; kb.y2 = kept[5 * t + 3]; kb.area = kept[5 * t + 4];
        if (rbox_iou_gt(kb, me, iou_thr)) alive = false;
      }
      unsigned int alive_mask = __ballot_sync(0xffffffffu, alive);
      for (int jl = 0; jl < 32; ++jl) {
        if (!((alive_mask >> jl) & 1u)) continue;       // warp-uniform
        RBox ob;
        ob.x1 = __shfl_sync(0xffffffffu, me.x1, jl); ob.y1 = __shfl_sync(0xffffffffu, me.y1, jl);
        ob.x2 = __shfl_sync(0xffffffffu, me.x2, jl); ob.y2 = __shfl_sync(0xffffffffu, me.y2, jl);
        ob.area = __shfl_sync(0xffffffffu, me.area, jl);
        const int pj = __shfl_sync(0xffffffffu, p, jl);
        if (nk < max_keep) {
          if (lane == 0) {
            kept[5 * nk] = ob.x1; kept[5 * nk + 1] = ob.y1; kept[5 * nk + 2] = ob.x2; kept[5 * nk + 3] = ob.y2; kept[5 * nk + 4] = ob.area;
            lvl_list[((size_t)b * lv.L + l) * max_keep + nk] = pj;
            lvl_key[((size_t)b * lv.L + l) * max_keep + nk] = ((unsigned long long)(~__float_as_uint(sc[pj])) << 32) | (unsigned int)pj;
          }
          ++nk;
        }
        if (lane > jl && alive && rbox_iou_gt(ob, me, iou_thr)) alive = false;
        alive_mask = __ballot_sync(0xffffffffu, alive);
        if (nk >= max_keep) break;
      }
      __syncwarp();
    }
  }
  if (threadIdx.x == 0) lvl_cnt[(size_t)b * lv.L + l] = nk;
}

// ---- round 2: bitmask NMS (levels with <= RPN_BM_MAX candidates) -------------------------------------------------------------------
// CTA per (level, image), 1024 threads.  After the same compaction + sort as above:
//   * the sorted, level-offset boxes go to shared memory (SoA),
//   * every thread fills words of the suppression matrix  M[i][w] bit j = IoU(box_i, box_{64w+j}) > thr  for 64w+j > i  — n^2/2
//     independent IoU tests spread over the CTA (the serial kernel above ran them on ONE warp, kept-list against candidates:
//     3.55 ms per launch in ncu, the whole RPN path's critical kernel),
//   * one warp walks the candidates in order: lane w holds word w of the "removed" set, the next survivor is a find-first-set on
//     the current word, keeping it ORs its row of M into the set.  ~50 cycles per KEPT box instead of an IoU sweep per candidate.
// The greedy order and the IoU predicate (argument order: earlier box first) are those of the serial kernel: identical keep lists.
constexpr int RPN_BM_MAX = 1024;
constexpr int RPN_BT = 1024;

__device__ __forceinline__ unsigned long long shfl_u64(unsigned long long v, int src) {
  const unsigned int lo = __shfl_sync(0xffffffffu, (unsigned int)v, src);
  const unsigned int hi = __shfl_sync(0xffffffffu, (unsigned int)(v >> 32), src);
  return ((unsigned long long)hi << 32) | lo;
}

__global__ void __launch_bounds__(RPN_BT)
rpn_nms_level_bitmask_kernel(const float4* __restrict__ cand_box, const float* __restrict__ cand_score, const uint8_t* __restrict__ valid,
                             int Ptot, RpnLevels lv, float iou_thr, int max_keep, const RpnImg* __restrict__ hdr,
                             int32_t* __restrict__ lvl_cnt /*[B][L]*/, int32_t* __restrict__ lvl_list /*[B][L][max_keep]*/,
                             unsigned long long* __restrict__ lvl_key /*[B][L][max_keep]*/) {
  __shared__ unsigned long long keys[RPN_BM_MAX];
  __shared__ float s_x1[RPN_BM_MAX], s_y1[RPN_BM_MAX], s_x2[RPN_BM_MAX], s_y2[RPN_BM_MAX], s_ar[RPN_BM_MAX];
  __shared__ int s_n;
  __shared__ int s_wbase[RPN_BT / 32];
  extern __shared__ unsigned long long bm[];     // [n][nw]
  const int l = blockIdx.x, b = blockIdx.y;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int seg0 = lv.seg_off[l], segn = lv.seg_off[l + 1] - seg0;      // <= RPN_BM_MAX (checked by the host)
  const float4* bx = cand_box + (size_t)b * Ptot;
  const float* sc = cand_score + (size_t)b * Ptot;
  const uint8_t* vd = valid + (size_t)b * Ptot;
  if (threadIdx.x == 0) s_n = 0;
  __syncthreads();
  {
    const int p = seg0 + threadIdx.x;
    const bool is = (int)threadIdx.x < segn && vd[p];
    const unsigned int bal = __ballot_sync(0xffffffffu, is);
    if (lane == 0) s_wbase[wid] = atomicAdd(&s_n, __popc(bal));
    __syncwarp();
    if (is) keys[s_wbase[wid] + __popc(bal & ((1u << lane) - 1u))] = ((unsigned long long)(~__float_as_uint(sc[p])) << 32) | (unsigned int)p;
  }
  __syncthreads();
  const int n = s_n;
  int n2 = 1;
  while (n2 < n) n2 <<= 1;
  for (int i = n + threadIdx.x; i < n2; i += RPN_BT) keys[i] = 0xFFFFFFFFFFFFFFFFull;
  bitonic_sort_u64(keys, n2);      // (the slot order of the compaction above does not matter: the keys are unique)
  const float off = __fmul_rn((float)l, __fadd_rn(hdr[b].max_coord, 1.f));
  if ((int)threadIdx.x < n) {
    const RBox me = rbox_offset(bx[(int)(keys[threadIdx.x] & 0xFFFFFFFFull)], off);
    s_x1[threadIdx.x] = me.x1; s_y1[threadIdx.x] = me.y1; s_x2[threadIdx.x] = me.x2; s_y2[threadIdx.x] = me.y2; s_ar[threadIdx.x] = me.area;
  }
  __syncthreads();
  const int nw = (n + 63) >> 6;
  // e = w * n + i: the lanes of a warp take CONSECUTIVE rows i of one word column w, so box j is a shared-memory broadcast and box i is
  // conflict-free (with e = i * nw + w the 16 lanes of a row read boxes 64 apart: one bank, 16-way conflicts — 635 us per launch)
  for (int e = threadIdx.x; e < n * nw; e += RPN_BT) {
    const int w = e / n, i = e - w * n;
    unsigned long long word = 0;
    const int j0 = max(64 * w, i + 1), j1 = min(64 * w + 64, n);
    if (j0 < j1) {
      RBox a;
      a.x1 = s_x1[i]; a.y1 = s_y1[i]; a.x2 = s_x2[i]; a.y2 = s_y2[i]; a.area = s_ar[i];
      for (int j = j0; j < j1; ++j) {
        RBox c;
        c.x1 = s_x1[j]; c.y1 = s_y1[j]; c.x2 = s_x2[j]; c.y2 = s_y2[j]; c.area = s_ar[j];
        if (rbox_iou_gt(a, c, iou_thr)) word |= 1ull << (j - 64 * w);
      }
    }
    bm[i * nw + w] = word;
  }
  __syncthreads();
  if (wid == 0) {
    unsigned long long remv = 0;               // lane w: removed candidates of word w (nw <= 16)
    int nk = 0;
    int32_t* out_list = lvl_list + ((size_t)b * lv.L + l) * max_keep;
    unsigned long long* out_key = lvl_key + ((size_t)b * lv.L + l) * max_keep;
    for (int w = 0; w < nw && nk < max_keep; ++w) {
      const int cnt = min(64, n - 64 * w);
      unsigned long long live = ~shfl_u64(remv, w) & (cnt == 64 ? ~0ull : ((1ull << cnt) - 1ull));
      while (live != 0ull && nk < max_keep) {          // warp-uniform
        const int bit = __ffsll((long long)live) - 1;
        const int i = 64 * w + bit;
        if (lane == 0) {
          const unsigned long long k = keys[i];
          out_list[nk] = (int32_t)(k & 0xFFFFFFFFull);
          out_key[nk] = k;
        }
        ++nk;
        const unsigned long long row = lane < nw ? bm[i * nw + lane] : 0ull;
        remv |= row;
        live &= ~shfl_u64(row, w);
        live &= ~(1ull << bit);
      }
    }
    if (lane == 0) lvl_cnt[(size_t)b * lv.L + l] = nk;
  }
}

// CTA per image: every kept entry finds its output rank = number of kept entries (all levels) with a smaller key — its own position in
// its level's list plus one binary search per other level (the lists are sorted; keys are unique).  Replaces the L-way merge that one
// lane walked serially (max_per_img rounds of dependent global loads).
__global__ void __launch_bounds__(1024)
rpn_nms_merge_rank_kernel(const float4* __restrict__ cand_box, const float* __restrict__ cand_score, int Ptot, RpnLevels lv, int max_keep,
                          const int32_t* __restrict__ lvl_cnt, const unsigned long long* __restrict__ lvl_key,
                          int32_t* __restrict__ out_count, float* __restrict__ out_det /*[B][max_keep][5]*/,
                          int32_t* __restrict__ out_level, int32_t* __restrict__ out_pos) {
  extern __shared__ unsigned long long sk[];   // [L][max_keep]
  __shared__ int cnt[RPN_MAX_LEVELS];
  const int b = blockIdx.x;
  if ((int)threadIdx.x < lv.L) cnt[threadIdx.x] = lvl_cnt[(size_t)b * lv.L + threadIdx.x];
  __syncthreads();
  for (int e = threadIdx.x; e < lv.L * max_keep; e += 1024) {
    const int l = e / max_keep, k = e - l * max_keep;
    if (k < cnt[l]) sk[e] = lvl_key[(size_t)b * lv.L * max_keep + e];
  }
  __syncthreads();
  const float4* bx = cand_box + (size_t)b * Ptot;
  const float* sc = cand_score + (size_t)b * Ptot;
  for (int e = threadIdx.x; e < lv.L * max_keep; e += 1024) {
    const int l = e / max_keep, k = e - l * max_keep;
    if (k >= cnt[l]) continue;
    const unsigned long long key = sk[e];
    int rank = k;
    for (int o = 0; o < lv.L; ++o) {
      if (o == l) continue;
      const unsigned long long* a = sk + o * max_keep;
      int lo = 0, hi = cnt[o];                   // first index with a[idx] > key  (== number of smaller keys: no equal keys exist)
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (a[mid] < key) lo = mid + 1; else hi = mid;
      }
      rank += lo;
    }
    if (rank < max_keep) {
      const int p = (int)(key & 0xFFFFFFFFull);
      const float4 q = bx[p];
      float* d = out_det + ((size_t)b * max_keep + rank) * 5;
      d[0] = q.x; d[1] = q.y; d[2] = q.z; d[3] = q.w; d[4] = sc[p];
      out_level[(size_t)b * max_keep + rank] = l;
      out_pos[(size_t)b * max_keep + rank] = p;
    }
  }
  if (threadIdx.x == 0) {
    int tot = 0;
    for (int l = 0; l < lv.L; ++l) tot += cnt[l];
    out_count[b] = tot < max_keep ? tot : max_keep;
  }
}

struct RpnPlan {
  int P[RPN_MAX_LEVELS], Q[RPN_MAX_LEVELS];
  RpnLevels lv;
  int Ptot, maxQ;
};
int rpn_plan(const int32_t* level_hw, int L, int A, int nms_pre, RpnPlan* pl) {
  pl->lv.L = L;
  pl->Ptot = 0; pl->maxQ = 0;
  for (int l = 0; l < L; ++l) {
    const long long Q = (long long)level_hw[2 * l] * level_hw[2 * l + 1] * A;
    if (Q <= 0 || Q > (1ll << 30)) return 1;
    pl->Q[l] = (int)Q;
    pl->P[l] = (nms_pre > 0 && Q > nms_pre) ? nms_pre : (int)Q;     // rpn_head.py:139: top-k only when there are more than nms_pre
    pl->lv.seg_off[l] = pl->Ptot;
    pl->Ptot += pl->P[l];
    if (pl->Q[l] > pl->maxQ) pl->maxQ = pl->Q[l];
  }
  pl->lv.seg_off[L] = pl->Ptot;
  return 0;
}
inline size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }

}  // namespace
}  // namespace ptb

using namespace ptb;

extern "C" uint64_t ptb_rpn_proposals_workspace(const int32_t* level_hw, int L, int B, int A, int nms_pre, int max_per_img) {
  RpnPlan pl;
  if (!level_hw || L <= 0 || L > RPN_MAX_LEVELS || B <= 0 || A <= 0 || max_per_img <= 0 || rpn_plan(level_hw, L, A, nms_pre, &pl)) return 0;
  size_t b = 0;
  b += al256((size_t)B * pl.maxQ * 4);                 // key
  b += al256((size_t)B * pl.Ptot * 16);                // cand_box
  b += al256((size_t)B * pl.Ptot * 4) * 2;             // cand_score, cand_idx
  b += al256((size_t)B * pl.Ptot);                     // valid
  b += al256((size_t)B * sizeof(RpnImg));
  b += al256((size_t)B * L * 4);                       // lvl_cnt
  b += al256((size_t)B * L * max_per_img * 4);         // lvl_list
  b += al256((size_t)B * L * max_per_img * 8);         // lvl_key
  b += al256((size_t)B * max_per_img * 4);             // out_pos (when the caller does not ask for it)
  return (uint64_t)b + 256;
}

extern "C" int ptb_rpn_proposals(const float* const* cls_scores, const float* const* bbox_preds, const int32_t* level_hw,
                                 const int32_t* strides_wh, const float* base_anchors, int L, int B, int A, const int32_t* img_hw,
                                 const float* means, const float* stds, float wh_ratio_clip, int nms_pre, float min_bbox_size,
                                 float iou_thr, int max_per_img, int32_t* out_count, float* out_det, int32_t* out_level,
                                 int32_t* out_pos, float* out_cand_box, float* out_cand_score, int32_t* out_cand_idx,
                                 void* workspace, uint64_t workspace_bytes, void* stream) {
  PTB_REQUIRE(L > 0 && L <= RPN_MAX_LEVELS && B > 0 && A > 0, "shape");
  PTB_REQUIRE(cls_scores && bbox_preds && level_hw && strides_wh && base_anchors && img_hw && means && stds, "NULL input");
  PTB_REQUIRE(max_per_img > 0 && max_per_img <= 2048, "max_per_img must be in [1,2048]");
  PTB_REQUIRE(nms_pre <= TOPK_MAX, "nms_pre > 4096 not supported (<= 0 keeps every anchor: then every level must have <= 4096 anchors)");
  PTB_REQUIRE(iou_thr >= 0.f && wh_ratio_clip > 0.f, "iou_thr >= 0, wh_ratio_clip > 0");
  PTB_REQUIRE(out_count && out_det && out_level, "NULL output");
  RpnPlan pl;
  PTB_REQUIRE(rpn_plan(level_hw, L, A, nms_pre, &pl) == 0, "level shape");
  for (int l = 0; l < L; ++l) PTB_REQUIRE(pl.P[l] <= TOPK_MAX, "a level keeps more than 4096 candidates");
  PTB_REQUIRE(workspace && workspace_bytes >= ptb_rpn_proposals_workspace(level_hw, L, B, A, nms_pre, max_per_img), "workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  char* w = reinterpret_cast<char*>(workspace);
  w += (256 - (reinterpret_cast<uintptr_t>(w) & 255)) & 255;
  float* key = reinterpret_cast<float*>(w); w += al256((size_t)B * pl.maxQ * 4);
  float4* cbox = reinterpret_cast<float4*>(w); w += al256((size_t)B * pl.Ptot * 16);
  float* cscore = reinterpret_cast<float*>(w); w += al256((size_t)B * pl.Ptot * 4);
  int32_t* cidx = reinterpret_cast<int32_t*>(w); w += al256((size_t)B * pl.Ptot * 4);
  uint8_t* valid = reinterpret_cast<uint8_t*>(w); w += al256((size_t)B * pl.Ptot);
  RpnImg* hdr = reinterpret_cast<RpnImg*>(w); w += al256((size_t)B * sizeof(RpnImg));
  int32_t* lvl_cnt = reinterpret_cast<int32_t*>(w); w += al256((size_t)B * L * 4);
  int32_t* lvl_list = reinterpret_cast<int32_t*>(w); w += al256((size_t)B * L * max_per_img * 4);
  unsigned long long* lvl_key = reinterpret_cast<unsigned long long*>(w); w += al256((size_t)B * L * max_per_img * 8);
  int32_t* pos_ws = reinterpret_cast<int32_t*>(w);
  if (out_cand_box) { PTB_REQUIRE(((uintptr_t)out_cand_box & 15) == 0, "out_cand_box must be 16-byte aligned"); cbox = reinterpret_cast<float4*>(out_cand_box); }
  if (out_cand_score) cscore = out_cand_score;
  if (out_cand_idx) cidx = out_cand_idx;
  if (!out_pos) out_pos = pos_ws;
  DecodeCfg dc;
  for (int k = 0; k < 4; ++k) { dc.mean[k] = means[k]; dc.stdv[k] = stds[k]; }
  dc.max_ratio = (float)fabs(log((double)wh_ratio_clip));      // np.abs(np.log(wh_ratio_clip)) as a double, cast like ATen's clamp scalar
  int rc;
  const int cap = sm_count() * 8;
  for (int l = 0; l < L; ++l) {
    PTB_REQUIRE(cls_scores[l] && bbox_preds[l], "NULL level tensor");
    const int H = level_hw[2 * l], W = level_hw[2 * l + 1], Q = pl.Q[l], P = pl.P[l];
    long long blocks = ((long long)B * Q + 255) / 256;
    if (blocks > cap) blocks = cap;
    rpn_score_kernel<<<(unsigned)blocks, 256, 0, st>>>(cls_scores[l], B, A, H * W, key);
    if ((rc = check_launch("ptb_rpn_proposals/score"))) return rc;
    const int identity = P == Q;
    if (!identity) {
      p2p_select_kernel<<<B, SEL_THREADS, 0, st>>>(key, Q, P, cidx + pl.lv.seg_off[l], pl.Ptot);
      if ((rc = check_launch("ptb_rpn_proposals/select"))) return rc;
    }
    rpn_decode_kernel<<<(unsigned)(((long long)B * P + 255) / 256), 256, 0, st>>>(
        bbox_preds[l], key, cidx, B, A, H, W, base_anchors + (size_t)l * A * 4, (float)strides_wh[2 * l], (float)strides_wh[2 * l + 1], dc,
        img_hw, P, pl.lv.seg_off[l], pl.Ptot, identity, cbox, cscore, cidx);
    if ((rc = check_launch("ptb_rpn_proposals/decode"))) return rc;
  }
  rpn_nms_prepare_kernel<<<B, RPN_T, 0, st>>>(cbox, pl.Ptot, min_bbox_size, valid, hdr);
  if ((rc = check_launch("ptb_rpn_proposals/prepare"))) return rc;
  int maxP = 0;
  for (int l = 0; l < L; ++l) maxP = pl.P[l] > maxP ? pl.P[l] : maxP;
  const char* e_bm = getenv("PTB_RPN_NMS");                 // "serial": the round-1 one-warp kernel (debug / A-B timing)
  if (maxP <= RPN_BM_MAX && !(e_bm && e_bm[0] == 's')) {
    const size_t bm_bytes = (size_t)maxP * ((maxP + 63) / 64) * 8;      // <= 128 KB
    if (cudaFuncSetAttribute(rpn_nms_level_bitmask_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(RPN_BM_MAX * (RPN_BM_MAX / 64) * 8)) !=
        cudaSuccess)
      return fail("%s", "cudaFuncSetAttribute(MaxDynamicSharedMemorySize) failed for rpn_nms_level_bitmask_kernel");
    rpn_nms_level_bitmask_kernel<<<dim3(L, B), RPN_BT, bm_bytes, st>>>(cbox, cscore, valid, pl.Ptot, pl.lv, iou_thr, max_per_img, hdr, lvl_cnt,
                                                                       lvl_list, lvl_key);
    if ((rc = check_launch("ptb_rpn_proposals/nms_level_bitmask"))) return rc;
  } else {
    // keys (32 KB static) + kept list (dynamic, <= 40 KB) exceed the 48 KB default; per device and cheap: set on every call
    if (cudaFuncSetAttribute(rpn_nms_level_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 2048 * 5 * (int)sizeof(float)) != cudaSuccess)
      return fail("%s", "cudaFuncSetAttribute(MaxDynamicSharedMemorySize) failed for rpn_nms_level_kernel");
    rpn_nms_level_kernel<<<dim3(L, B), RPN_T, (size_t)max_per_img * 5 * sizeof(float), st>>>(cbox, cscore, valid, pl.Ptot, pl.lv, iou_thr,
                                                                                             max_per_img, hdr, lvl_cnt, lvl_list, lvl_key);
    if ((rc = check_launch("ptb_rpn_proposals/nms_level"))) return rc;
  }
  const size_t mk_bytes = (size_t)L * max_per_img * 8;        // <= 8 x 2048 x 8 = 128 KB
  if (cudaFuncSetAttribute(rpn_nms_merge_rank_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, RPN_MAX_LEVELS * 2048 * 8) != cudaSuccess)
    return fail("%s", "cudaFuncSetAttribute(MaxDynamicSharedMemorySize) failed for rpn_nms_merge_rank_kernel");
  rpn_nms_merge_rank_kernel<<<B, 1024, mk_bytes, st>>>(cbox, cscore, pl.Ptot, pl.lv, max_per_img, lvl_cnt, lvl_key, out_count, out_det, out_level,
                                                       out_pos);
  return check_launch("ptb_rpn_proposals/merge");
}
