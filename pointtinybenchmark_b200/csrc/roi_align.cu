// R-CNN box stage of the dense-anchor detector (BASELINE.json config 4: StandardRoIHead with SingleRoIExtractor + Shared2FCBBoxHead):
//   ptb_roi_align          SingleRoIExtractor.forward (single_level_roi_extractor.py:55-100): level choice map_roi_levels + mmcv
//                          RoIAlign (avg, aligned or not, any sampling_ratio) for every RoI of the batch and every level in one launch.
//                          Output either fp32 (M, oh, ow, C) channels-last, or directly the fp16 two-term operand pair (h, l) of the
//                          box head's first GEMM at a power-of-two scale taken on the device from max|feat| (ptb_amax_abs): every
//                          output is a convex combination of map values, so that bound holds before any sampling.
//   ptb_relu_split_f16     ReLU + fp16 (h, l) split of a GEMM output (fc6 -> fc7 -> predictors), unit scale.
//   ptb_rcnn_bbox_decode   per RoI: the padding mask of simple_test_bboxes (test_mixins.py:96-110), softmax over N+1 classes,
//                          class-specific delta2bbox with clip (shared with the RPN, bbox_coder.cuh), optional rescale
//                          (bbox_head.py:383-390), and the (box, class) candidate scores of multiclass_nms (bbox_nms.py:30-50).
// No float atomics anywhere: every output element is written by exactly one thread in a fixed order (run-to-run bit-identical).
#include "bbox_coder.cuh"
#include "tc_ptx.cuh"
#include <math_constants.h>

namespace ptb {
namespace {

constexpr int ROI_MAX_LEVELS = 5;
constexpr int ROI_T = 256;

struct RoiLevels {          // by-value kernel argument
  const float* feat[ROI_MAX_LEVELS];     // (B, H, W, C) channels-last, contiguous
  int H[ROI_MAX_LEVELS], W[ROI_MAX_LEVELS];
  float scale[ROI_MAX_LEVELS];           // spatial_scale = 1 / stride
  int L;
};

// map_roi_levels: floor(log2(sqrt(w*h) / finest_scale + 1e-6)) clamped to [0, L-1], fp32 with IEEE sqrt / division.  ATen's CPU
// log2 of an fp32 value equals (float)log2((double)x) on every input in [0.25, 16] (it rounds up to 3.0 at 7.9999995f and to 4.0
// at 15.999999f, where a floor of the exponent bits would not); the double log2 reproduces that.  A NaN scale (negative area)
// gives -1: the reference's NaN level matches no level there and the RoI's features stay zero.
__device__ __forceinline__ int roi_level(float x1, float y1, float x2, float y2, float finest_scale, int L) {
  if (L == 1) return 0;
  const float area = __fmul_rn(__fsub_rn(x2, x1), __fsub_rn(y2, y1));
  const float v = __fadd_rn(__fdiv_rn(__fsqrt_rn(area), finest_scale), 1e-6f);
  if (isnan(v)) return -1;
  const float lg = floorf((float)log2((double)v));
  return (int)fminf(fmaxf(lg, 0.f), (float)(L - 1));
}

// mmcv bilinear_interpolate (roi_align_cuda_kernel.cuh) in torchvision's CPU operation order (no contraction)
__device__ __forceinline__ float4 roi_tap(const float* __restrict__ f, int H, int W, int C, int c, float y, float x) {
  if (y < -1.f || y > (float)H || x < -1.f || x > (float)W) return make_float4(0.f, 0.f, 0.f, 0.f);
  if (y <= 0.f) y = 0.f;
  if (x <= 0.f) x = 0.f;
  int y_lo = (int)y, x_lo = (int)x, y_hi, x_hi;
  if (y_lo >= H - 1) { y_hi = y_lo = H - 1; y = (float)y_lo; } else y_hi = y_lo + 1;
  if (x_lo >= W - 1) { x_hi = x_lo = W - 1; x = (float)x_lo; } else x_hi = x_lo + 1;
  const float ly = __fsub_rn(y, (float)y_lo), lx = __fsub_rn(x, (float)x_lo);
  const float hy = __fsub_rn(1.f, ly), hx = __fsub_rn(1.f, lx);
  const float w1 = __fmul_rn(hy, hx), w2 = __fmul_rn(hy, lx), w3 = __fmul_rn(ly, hx), w4 = __fmul_rn(ly, lx);
  const float4 v1 = __ldg(reinterpret_cast<const float4*>(f + ((size_t)y_lo * W + x_lo) * C + c));
  const float4 v2 = __ldg(reinterpret_cast<const float4*>(f + ((size_t)y_lo * W + x_hi) * C + c));
  const float4 v3 = __ldg(reinterpret_cast<const float4*>(f + ((size_t)y_hi * W + x_lo) * C + c));
  const float4 v4 = __ldg(reinterpret_cast<const float4*>(f + ((size_t)y_hi * W + x_hi) * C + c));
  auto comb = [&](float a, float b, float cc, float d) {
    return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(w1, a), __fmul_rn(w2, b)), __fmul_rn(w3, cc)), __fmul_rn(w4, d));
  };
  return make_float4(comb(v1.x, v2.x, v3.x, v4.x), comb(v1.y, v2.y, v3.y, v4.y), comb(v1.z, v2.z, v3.z, v4.z), comb(v1.w, v2.w, v3.w, v4.w));
}

// one CTA per RoI (rows M .. M_pad-1 of the fp16 operand are zero padding of the GEMM's 16-row groups); thread item = (bin, 4 channels)
__global__ void __launch_bounds__(ROI_T)
roi_align_kernel(const float* __restrict__ rois, int M, RoiLevels lv, int B, int C, int oh, int ow, int sampling_ratio, float offset,
                 int aligned, float finest_scale, const unsigned int* __restrict__ amax_bits, float* __restrict__ out,
                 uint2* __restrict__ out_h, uint2* __restrict__ out_l, float* __restrict__ inv_scale_out, int8_t* __restrict__ out_level) {
  __shared__ const float* s_f;
  __shared__ int s_lvl, s_H, s_W, s_gh, s_gw;
  __shared__ float s_x0, s_y0, s_bw, s_bh, s_cnt;
  const int m = blockIdx.x;
  const int C4 = C >> 2;
  const int items = oh * ow * C4;
  const float scale = out_h ? pow2_scale_for(__uint_as_float(*amax_bits)) : 1.f;
  if (out_h && m == 0 && threadIdx.x == 0) *inv_scale_out = 1.f / scale;
  if (m >= M) {                                     // GEMM row padding
    for (int i = threadIdx.x; i < items; i += ROI_T) {
      out_h[(size_t)m * items + i] = make_uint2(0u, 0u);
      out_l[(size_t)m * items + i] = make_uint2(0u, 0u);
    }
    return;
  }
  if (threadIdx.x == 0) {
    const float* r = rois + (size_t)m * 5;
    const int b = (int)r[0];
    int lvl = roi_level(r[1], r[2], r[3], r[4], finest_scale, lv.L);
    if (out_level) out_level[m] = (int8_t)lvl;
    if (b < 0 || b >= B) lvl = -1;
    s_lvl = lvl;
    float s = 0.f;
#pragma unroll
    for (int l = 0; l < ROI_MAX_LEVELS; ++l)       // static indices: the level table stays in parameter space
      if (l == lvl) { s = lv.scale[l]; s_H = lv.H[l]; s_W = lv.W[l]; s_f = lv.feat[l] + (size_t)b * lv.H[l] * lv.W[l] * C; }
    if (lvl >= 0) {
      const float x0 = __fsub_rn(__fmul_rn(r[1], s), offset), y0 = __fsub_rn(__fmul_rn(r[2], s), offset);
      const float x1 = __fsub_rn(__fmul_rn(r[3], s), offset), y1 = __fsub_rn(__fmul_rn(r[4], s), offset);
      float rw = __fsub_rn(x1, x0), rh = __fsub_rn(y1, y0);
      if (!aligned) { rw = fmaxf(rw, 1.f); rh = fmaxf(rh, 1.f); }
      s_x0 = x0; s_y0 = y0;
      s_bw = __fdiv_rn(rw, (float)ow); s_bh = __fdiv_rn(rh, (float)oh);
      const int gh = sampling_ratio > 0 ? sampling_ratio : (int)ceilf(__fdiv_rn(rh, (float)oh));
      const int gw = sampling_ratio > 0 ? sampling_ratio : (int)ceilf(__fdiv_rn(rw, (float)ow));
      s_gh = gh; s_gw = gw;
      s_cnt = (float)max(gh * gw, 1);
    }
  }
  __syncthreads();
  const int lvl = s_lvl;
  for (int i = threadIdx.x; i < items; i += ROI_T) {
    const int bin = i / C4, c = (i - bin * C4) * 4;
    const int ph = bin / ow, pw = bin - ph * ow;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (lvl >= 0) {
      const int H = s_H, W = s_W;
      const float* f = s_f;
      const float gh = (float)s_gh, gw = (float)s_gw;
      for (int iy = 0; iy < s_gh; ++iy) {
        const float y = __fadd_rn(__fadd_rn(s_y0, __fmul_rn((float)ph, s_bh)), __fdiv_rn(__fmul_rn((float)iy + .5f, s_bh), gh));
        for (int ix = 0; ix < s_gw; ++ix) {
          const float x = __fadd_rn(__fadd_rn(s_x0, __fmul_rn((float)pw, s_bw)), __fdiv_rn(__fmul_rn((float)ix + .5f, s_bw), gw));
          const float4 v = roi_tap(f, H, W, C, c, y, x);
          acc.x = __fadd_rn(acc.x, v.x); acc.y = __fadd_rn(acc.y, v.y); acc.z = __fadd_rn(acc.z, v.z); acc.w = __fadd_rn(acc.w, v.w);
        }
      }
      const float cnt = s_cnt;
      acc = make_float4(__fdiv_rn(acc.x, cnt), __fdiv_rn(acc.y, cnt), __fdiv_rn(acc.z, cnt), __fdiv_rn(acc.w, cnt));
    }
    const size_t o = (size_t)m * items + i;
    if (out) __stcs(reinterpret_cast<float4*>(out) + o, acc);
    if (out_h) {
      __align__(8) __half h[4], l[4];
      split_h2(acc.x * scale, h[0], l[0]); split_h2(acc.y * scale, h[1], l[1]);
      split_h2(acc.z * scale, h[2], l[2]); split_h2(acc.w * scale, h[3], l[3]);
      out_h[o] = *reinterpret_cast<uint2*>(h);
      out_l[o] = *reinterpret_cast<uint2*>(l);
    }
  }
}

__global__ void __launch_bounds__(256)
relu_split_f16_kernel(const float4* __restrict__ y, int rows, int n4, int ld4, uint2* __restrict__ out_h, uint2* __restrict__ out_l,
                      int* __restrict__ overflow_flag) {
  const long long total = (long long)rows * n4;
  bool clamped = false;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const long long r = i / n4;
    const int c = (int)(i - r * n4);
    const float4 v = __ldcs(y + r * ld4 + c);
    float o[4] = {v.x, v.y, v.z, v.w};
    __align__(8) __half h[4], l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      o[j] = fmaxf(o[j], 0.f);
      if (o[j] > 60000.f) { o[j] = 60000.f; clamped = true; }
      split_h2(o[j], h[j], l[j]);
    }
    out_h[i] = *reinterpret_cast<uint2*>(h);
    out_l[i] = *reinterpret_cast<uint2*>(l);
  }
  if (clamped && overflow_flag) *overflow_flag = 1;
}

// thread per RoI.  Softmax in ATen's order (max, exp(x - max), sum, times 1/sum) with the Sleef exp of ATen's vectorised CPU path.
__global__ void __launch_bounds__(256)
rcnn_bbox_decode_kernel(const float* __restrict__ rois, int R, int n_per_img, const float* __restrict__ cls, int ldc,
                        const float* __restrict__ reg, int ldr, int N, int mask_padding, DecodeCfg dc, const int32_t* __restrict__ img_hw,
                        const float* __restrict__ scale_factor, float* __restrict__ out_boxes, float* __restrict__ out_scores,
                        float* __restrict__ out_cand_scores) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= R) return;
  const int b = i / n_per_img;
  const float* r = rois + (size_t)i * 5;
  const float x1 = r[1], y1 = r[2], x2 = r[3], y2 = r[4];
  const bool pad = mask_padding && __fadd_rn(__fadd_rn(__fadd_rn(fabsf(x1), fabsf(y1)), fabsf(x2)), fabsf(y2)) == 0.f;
  const float* lg = cls + (size_t)i * ldc;
  float mx = pad ? 0.f : lg[0];
  for (int k = 1; k <= N; ++k) mx = fmaxf(mx, pad ? 0.f : lg[k]);
  float sum = 0.f;
  for (int k = 0; k <= N; ++k) sum = __fadd_rn(sum, sleef_expf_u10(__fsub_rn(pad ? 0.f : lg[k], mx)));
  const float inv = __fdiv_rn(1.f, sum);
  const float mw = (float)img_hw[2 * b + 1], mh = (float)img_hw[2 * b];
  const float* d = reg + (size_t)i * ldr;
  for (int k = 0; k <= N; ++k) {
    const float p = __fmul_rn(sleef_expf_u10(__fsub_rn(pad ? 0.f : lg[k], mx)), inv);
    if (out_scores) out_scores[(size_t)i * (N + 1) + k] = p;
    if (k < N && out_cand_scores) {
      float* cs = out_cand_scores + ((size_t)i * N + k) * N;       // candidate (RoI i, class k): its score in its own class only
      for (int j = 0; j < N; ++j) cs[j] = j == k ? p : -CUDART_INF_F;
    }
  }
  for (int k = 0; k < N; ++k) {
    float4 bx = pad ? delta2bbox_clip(x1, y1, x2, y2, 0.f, 0.f, 0.f, 0.f, dc, mw, mh)
                    : delta2bbox_clip(x1, y1, x2, y2, d[4 * k], d[4 * k + 1], d[4 * k + 2], d[4 * k + 3], dc, mw, mh);
    if (scale_factor) {
      const float* sf = scale_factor + 4 * b;
      bx = make_float4(__fdiv_rn(bx.x, sf[0]), __fdiv_rn(bx.y, sf[1]), __fdiv_rn(bx.z, sf[2]), __fdiv_rn(bx.w, sf[3]));
    }
    reinterpret_cast<float4*>(out_boxes)[(size_t)i * N + k] = bx;
  }
}

}  // namespace
}  // namespace ptb

using namespace ptb;

extern "C" int ptb_roi_align(const float* rois, int M, int M_pad, const void* const* feats, const int32_t* hw, const float* spatial_scales,
                             int L, int B, int C, int out_h, int out_w, int sampling_ratio, int aligned, float finest_scale,
                             const unsigned int* dev_amax_bits, float* out, void* out_h16, void* out_l16, float* dev_inv_scale,
                             int8_t* out_level, void* stream) {
  PTB_REQUIRE(M >= 0 && B > 0 && L >= 1 && L <= ROI_MAX_LEVELS, "shape: 1 <= levels <= 5");
  PTB_REQUIRE(C > 0 && C % 32 == 0, "C must be a multiple of 32");
  PTB_REQUIRE(out_h > 0 && out_w > 0 && out_h * out_w <= 256 && sampling_ratio >= 0, "output size / sampling_ratio");
  PTB_REQUIRE(finest_scale > 0.f, "finest_scale > 0");
  PTB_REQUIRE((out != nullptr) != (out_h16 != nullptr), "exactly one of out (fp32) / out_h16, out_l16 (fp16 pair)");
  PTB_REQUIRE(!out_h16 || (out_l16 && dev_amax_bits && dev_inv_scale && M_pad >= M), "fp16 mode needs out_l16, dev_amax_bits, dev_inv_scale");
  PTB_REQUIRE(out_h16 || M_pad == M, "M_pad != M only in fp16 mode");
  PTB_REQUIRE(M == 0 || rois, "NULL rois");
  RoiLevels lv = {};
  lv.L = L;
  for (int l = 0; l < L; ++l) {
    PTB_REQUIRE(feats[l] && ((uintptr_t)feats[l] % 16) == 0 && hw[2 * l] > 0 && hw[2 * l + 1] > 0, "level map NULL / unaligned / empty");
    lv.feat[l] = reinterpret_cast<const float*>(feats[l]);
    lv.H[l] = hw[2 * l]; lv.W[l] = hw[2 * l + 1]; lv.scale[l] = spatial_scales[l];
  }
  const int grid = out_h16 ? M_pad : M;
  if (grid == 0) return 0;
  roi_align_kernel<<<grid, ROI_T, 0, (cudaStream_t)stream>>>(rois, M, lv, B, C, out_h, out_w, sampling_ratio, aligned ? 0.5f : 0.f, aligned,
                                                            finest_scale, dev_amax_bits, out, reinterpret_cast<uint2*>(out_h16),
                                                            reinterpret_cast<uint2*>(out_l16), dev_inv_scale, out_level);
  return check_launch("ptb_roi_align");
}

extern "C" int ptb_relu_split_f16(const float* y, int rows, int n, int ld, void* out_h, void* out_l, int* overflow_flag, void* stream) {
  PTB_REQUIRE(rows >= 0 && n > 0 && n % 4 == 0 && ld >= n && ld % 4 == 0, "n, ld multiples of 4, ld >= n");
  PTB_REQUIRE(y && out_h && out_l && ((uintptr_t)y % 16) == 0 && ((uintptr_t)out_h % 8) == 0 && ((uintptr_t)out_l % 8) == 0,
              "NULL / alignment");
  const long long total = (long long)rows * (n / 4);
  if (total == 0) return 0;
  long long blocks = (total + 255) / 256;
  const long long cap = (long long)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  relu_split_f16_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(y), rows, n / 4, ld / 4,
                                                                           reinterpret_cast<uint2*>(out_h), reinterpret_cast<uint2*>(out_l),
                                                                           overflow_flag);
  return check_launch("ptb_relu_split_f16");
}

extern "C" int ptb_rcnn_bbox_decode(const float* rois, int B, int n_per_img, const float* cls, int ldc, const float* reg, int ldr,
                                    int num_classes, int mask_padding, const float* means, const float* stds, float wh_ratio_clip,
                                    const int32_t* img_hw, const float* scale_factor, float* out_boxes, float* out_scores,
                                    float* out_cand_scores, void* stream) {
  PTB_REQUIRE(B > 0 && n_per_img >= 0 && num_classes > 0, "shape");
  PTB_REQUIRE(ldc >= num_classes + 1 && ldr >= 4 * num_classes, "row strides");
  PTB_REQUIRE(rois && cls && reg && img_hw && out_boxes && ((uintptr_t)out_boxes % 16) == 0, "NULL / alignment");
  PTB_REQUIRE(wh_ratio_clip > 0.f, "wh_ratio_clip > 0");
  DecodeCfg dc;
  for (int k = 0; k < 4; ++k) { dc.mean[k] = means[k]; dc.stdv[k] = stds[k]; }
  dc.max_ratio = (float)fabs(log((double)wh_ratio_clip));      // np.abs(np.log(wh_ratio_clip)) as a double, cast like ATen's clamp scalar
  const int R = B * n_per_img;
  if (R == 0) return 0;
  rcnn_bbox_decode_kernel<<<(R + 255) / 256, 256, 0, (cudaStream_t)stream>>>(rois, R, n_per_img, cls, ldc, reg, ldr, num_classes,
                                                                            mask_padding, dc, img_hw, scale_factor, out_boxes, out_scores,
                                                                            out_cand_scores);
  return check_launch("ptb_rcnn_bbox_decode");
}
