// DeltaXYWHBBoxCoder.decode (mmdet/core/bbox/coder/delta_xywh_bbox_coder.py:144-270) for one (box, delta) pair, shared by the
// RPN proposal decode (rpn.cu) and the R-CNN box decode (roi_align.cu).  fp32, one rounding per ATen operation, in the
// reference's order; boxes are clipped to [0, max_w] x [0, max_h] (clip_border=True, max_shape = img_shape).
#pragma once
#include "ptb_common.cuh"

namespace ptb {

struct DecodeCfg {
  float mean[4], stdv[4];
  float max_ratio;      // |log(wh_ratio_clip)|
};

__device__ __forceinline__ float4 delta2bbox_clip(float ax1, float ay1, float ax2, float ay2, float d0, float d1, float d2, float d3,
                                                  const DecodeCfg& dc, float mw, float mh) {
  // delta_xywh_bbox_coder.py:209-246 (fp32, separate multiply and add as ATen executes them)
  const float dx = __fadd_rn(__fmul_rn(d0, dc.stdv[0]), dc.mean[0]);
  const float dy = __fadd_rn(__fmul_rn(d1, dc.stdv[1]), dc.mean[1]);
  float dw = __fadd_rn(__fmul_rn(d2, dc.stdv[2]), dc.mean[2]);
  float dh = __fadd_rn(__fmul_rn(d3, dc.stdv[3]), dc.mean[3]);
  const float px = __fmul_rn(__fadd_rn(ax1, ax2), 0.5f), py = __fmul_rn(__fadd_rn(ay1, ay2), 0.5f);
  const float pw = __fsub_rn(ax2, ax1), ph = __fsub_rn(ay2, ay1);
  const float dxw = __fmul_rn(pw, dx), dyh = __fmul_rn(ph, dy);
  dw = fminf(fmaxf(dw, -dc.max_ratio), dc.max_ratio);
  dh = fminf(fmaxf(dh, -dc.max_ratio), dc.max_ratio);
  const float gw = __fmul_rn(pw, expf(dw)), gh = __fmul_rn(ph, expf(dh));
  const float gx = __fadd_rn(px, dxw), gy = __fadd_rn(py, dyh);
  const float hw2 = __fmul_rn(gw, 0.5f), hh2 = __fmul_rn(gh, 0.5f);
  float x1 = __fsub_rn(gx, hw2), y1 = __fsub_rn(gy, hh2), x2 = __fadd_rn(gx, hw2), y2 = __fadd_rn(gy, hh2);
  x1 = x1 < 0.f ? 0.f : x1; y1 = y1 < 0.f ? 0.f : y1; x2 = x2 < 0.f ? 0.f : x2; y2 = y2 < 0.f ? 0.f : y2;
  x1 = x1 > mw ? mw : x1; y1 = y1 > mh ? mh : y1; x2 = x2 > mw ? mw : x2; y2 = y2 > mh ? mh : y2;
  return make_float4(x1, y1, x2, y2);
}

}  // namespace ptb
