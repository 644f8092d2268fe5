// Backward of the CPR training loss w.r.t. the logit map, gather-formulated and DETERMINISTIC (round 2; replaces round 1's chain
// mil_bwd -> gfocal_bwd -> bag_gather_bwd (fp32 vector atomics into a zeroed map) -> gfocal_bwd(neg)).
//
//   d loss / d lmap[cell][ch] =   sum over (bag g, sample k, tap t on this cell)  w_t * d loss / d bag_logit[g][k][ch]      (grid_sample backward)
//                               + [ch < N] neg-loss term of the cell itself                                                (cpr_head.py:1219-1228)
//   d/d cls logit = gp * pi * sg (1 - sg)   [+ centre sample: gt-loss term, cpr_head.py:1159-1184]      gp = dLoss/dprob[g][c] (gfocal')
//   d/d ins logit = gp * pi * (sg - p)                                                                 pi = e w / T, e = exp(ins - m)
//   (MILLoss.forward, multi_instance_learning_loss.py:153-203; m, 1/T, p, gfocal'(p) per (bag, class) come from the forward kernel)
//
// One CTA owns a tile of 8 x 8 map cells and ALL channels of it; thread (cell, 32-channel group) keeps its 32 sums in registers.
//   A  the bags of the image whose sample window reaches the tile, in GT order (ordered ballot compaction);
//   B  bag by bag, warp w evaluates samples 32w .. 32w+31 (lane = sample: tap geometry, which taps land in the tile) and the samples
//      with a tap in the tile are appended to a record buffer in (bag, k) order;
//   C  rounds of min(64, blockDim.x / 4) records: (1) one warp per record, lanes = classes: two coalesced loads of the sampled logits,
//      the per-sample gradient row staged in shared memory; (2) the <= blockDim.x (record, tap) hits of the round are counting-sorted by
//      cell (stable), one thread per hit; (3) every
//      (cell, channel group) thread walks its cell's hits in order: acc += w * staged row.
// No atomics anywhere and every sum is evaluated by ONE thread in a FIXED order: bit-identical run to run, no zero-initialised gradient
// map, no materialised (G,K,2N) gradient tensor (740 MB written and re-read in round 1).  ncu history: a first version (one warp per
// (bag, chunk), per-(tap, channel) shared-memory atomics into 64-bit fixed point) took 3.1 ms with 64-bit CAS loops and 2.1 ms with
// hi/lo 32-bit atomics — 680 M warp instructions, a third of the time at the block barrier; this layout needs ~2.5x fewer.
// Samples whose taps straddle a tile border are evaluated by each tile they touch (~1.25x).
#include "ptb_common.cuh"
#include <math_constants.h>

namespace ptb {

constexpr int LB_T = 8;                       // tile side (cells)
constexpr int LB_CELLS = LB_T * LB_T;
constexpr int LB_MAXCAND = 1024;              // GT indices examined per pass
constexpr int LB_REC = 512;                   // record buffer (a bag contributes at most K <= 320 relevant samples per pass)
constexpr int LB_ROUND = 64;                  // records staged per round
constexpr int LB_NIT = 8;                     // class iterations per lane: up to 256 classes
constexpr int LB_MAXK = 320;                  // samples per bag handled by the 10 warps of the evaluation step

__device__ __forceinline__ float fast_sigmoid(float x) { return __fdividef(1.f, 1.f + __expf(-x)); }
__device__ __forceinline__ float gfocal_dp_f(float p, float q, float eps) {      // d/dp of -( (p-q)^2 (q log(p+eps) + (1-q) log(1-p+eps)) )
  const float d = p - q;
  const float L = q * __logf(p + eps) + (1.f - q) * __logf(1.f - p + eps);
  const float dL = __fdividef(q, p + eps) - __fdividef(1.f - q, 1.f - p + eps);
  return -(2.f * d * L + d * d * dL);
}

struct LossBwdArgs {
  const float* bl;          // [G][K][LD] sampled logits (cls at 0, ins at NP)
  const float* weight;      // [G][K]
  const float4* coef;       // [G][N]  (max ins, 1/T or 0, bag prob, label_weight * gfocal'(prob, onehot))
  const int32_t* labels;    // [G]
  const float* centers;     // [G][2]
  const int32_t* img_ptr;   // [B+1]
  const float* offsets;     // [K][2]
  const float* scale_mil;   // [1] or NULL (no MIL term)
  const float* scale_gt;    // [1] or NULL
  const float* wc;          // [G] validity of the centre sample (gt loss) or NULL
  const float* lmap;        // [B][H][W][LD] logit map (neg term) or NULL
  const uint8_t* neg_mask;  // [B][H][W][N]
  const float* scale_neg;   // [1]
  float* dlmap;             // [B][H][W][LD]
  int H, W, N, NP, LD, K;
  float stride, reach_px, eps;
};

struct LbRec {              // a sample with at least one tap in the tile
  int g, k;
  float wk;
  int cells;                // 4 x int8: local cell of tap t or -1
  float w[4];
};

__global__ void __launch_bounds__(320, 2)
cpr_loss_bwd_tile_kernel(const LossBwdArgs a) {
  extern __shared__ float st[];                        // [LB_ROUND][LDS] staged gradient rows (row stride LDS = LD + 4: bank spread)
  __shared__ LbRec s_rec[LB_REC];
  __shared__ int s_cand[LB_MAXCAND];
  __shared__ int s_ncand, s_nrec;
  __shared__ int s_wcnt[16];
  __shared__ int s_ccnt[LB_CELLS], s_cstart[LB_CELLS + 1];
  __shared__ unsigned short s_hit[LB_ROUND * 4];       // sorted hits: (record in round << 2) | tap
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  const int b = blockIdx.z;
  const int tx0 = blockIdx.x * LB_T, ty0 = blockIdx.y * LB_T;
  const int H = a.H, W = a.W, N = a.N, NP = a.NP, LD = a.LD, K = a.K;
  const int LDS = LD + 4;
  const int groups = LD >> 5;                          // 32-channel groups; blockDim.x == 64 * groups
  const int my_cell = tid / groups, my_grp = tid - my_cell * groups;
  const float hw = 0.5f * (float)W, hh = 0.5f * (float)H;
  const float s_mil = a.scale_mil ? a.scale_mil[0] : 0.f;
  const float s_gt = (a.scale_gt && a.wc) ? a.scale_gt[0] : 0.f;
  const int g_lo = a.img_ptr[b], g_hi = a.img_ptr[b + 1];
  const int nit = (N + 31) / 32;
  float acc[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) acc[i] = 0.f;
  for (int i = tid; i < LB_ROUND * LDS; i += blockDim.x) st[i] = 0.f;      // pad columns [N, NP) stay zero for the whole kernel
  if (tid == 0) s_nrec = 0;

  // ---- C: consume the record buffer in rounds of up to LB_ROUND records.  Step (2) ranks each (record, tap) hit on the thread of the
  // same index, so a round holds at most blockDim.x / 4 records: 64 at LD >= 128, 16 / 32 / 48 at LD 32 / 64 / 96
  const int per_round = min(LB_ROUND, (int)blockDim.x / 4);
  auto process = [&]() {
    const int nrec = s_nrec;                                               // (caller has synchronised)
    for (int r0 = 0; r0 < nrec; r0 += per_round) {
      const int nr = min(per_round, nrec - r0);
      // (1) gradient rows: one warp per record, lanes = classes
      for (int r = warp; r < nr; r += nwarps) {
        const LbRec rec = s_rec[r0 + r];
        const float* row = a.bl + ((size_t)rec.g * K + rec.k) * LD;
        const float4* cf = a.coef + (size_t)rec.g * N;
        const int lab = a.labels[rec.g];
        const float sgt = (s_gt != 0.f && rec.k == K - 1) ? s_gt * a.wc[rec.g] : 0.f;
        float* out = st + (size_t)r * LDS;
#pragma unroll
        for (int i = 0; i < LB_NIT; ++i) {
          const int c = lane + 32 * i;
          if (i < nit && c < N) {
            const float xc = __ldg(row + c), xi = __ldg(row + NP + c);
            const float4 q = __ldg(cf + c);                                // (m, 1/T, p, lw * gfocal'(p))
            const float sg = fast_sigmoid(xc);
            const float gpi = s_mil * q.w * (__expf(xi - q.x) * rec.wk * q.y);
            float dc = gpi * sg * (1.f - sg);
            if (sgt != 0.f) dc += sgt * gfocal_dp_f(sg, c == lab ? 1.f : 0.f, a.eps) * sg * (1.f - sg);
            out[c] = dc;
            out[NP + c] = gpi * (sg - q.z);
          }
        }
      }
      // (2) stable counting sort of the round's (record, tap) hits by cell
      if (tid < LB_CELLS) s_ccnt[tid] = 0;
      __syncthreads();
      int my_hit_cell = -1, my_rank = 0;
      if (tid < nr * 4) {
        my_hit_cell = (int)(signed char)((s_rec[r0 + (tid >> 2)].cells >> (8 * (tid & 3))) & 0xff);
        if (my_hit_cell >= 0) {
          for (int e = 0; e < tid; ++e) {                                  // rank among the earlier hits of the same cell (<= 255 broadcast reads)
            const int ce = (int)(signed char)((s_rec[r0 + (e >> 2)].cells >> (8 * (e & 3))) & 0xff);
            my_rank += (ce == my_hit_cell);
          }
          atomicAdd(&s_ccnt[my_hit_cell], 1);                              // integer count: order-independent
        }
      }
      __syncthreads();
      if (tid == 0) {
        int run = 0;
        for (int c = 0; c < LB_CELLS; ++c) { s_cstart[c] = run; run += s_ccnt[c]; }
        s_cstart[LB_CELLS] = run;
      }
      __syncthreads();
      if (my_hit_cell >= 0) s_hit[s_cstart[my_hit_cell] + my_rank] = (unsigned short)tid;
      __syncthreads();
      // (3) every (cell, channel group) thread adds its cell's hits in order
      {
        const int h0 = s_cstart[my_cell], h1 = s_cstart[my_cell + 1];
        for (int hix = h0; hix < h1; ++hix) {
          const int e = s_hit[hix];
          const float w = s_rec[r0 + (e >> 2)].w[e & 3];
          const float4* src = reinterpret_cast<const float4*>(st + (size_t)(e >> 2) * LDS + 32 * my_grp);
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const float4 v = src[q];
            acc[4 * q] = fmaf(w, v.x, acc[4 * q]); acc[4 * q + 1] = fmaf(w, v.y, acc[4 * q + 1]);
            acc[4 * q + 2] = fmaf(w, v.z, acc[4 * q + 2]); acc[4 * q + 3] = fmaf(w, v.w, acc[4 * q + 3]);
          }
        }
      }
      __syncthreads();                                                     // the staged rows / hit list are free again
    }
    if (tid == 0) s_nrec = 0;
    __syncthreads();
  };

  for (int seg = g_lo; seg < g_hi; seg += LB_MAXCAND) {
    // ---- A: bags of this image whose window reaches the tile, in GT order (warp 0, ordered ballot compaction)
    __syncthreads();
    if (warp == 0) {
      int n = 0;
      for (int g0 = seg; g0 < min(seg + LB_MAXCAND, g_hi); g0 += 32) {
        const int g = g0 + lane;
        bool hit = false;
        if (g < g_hi) {
          const float cx = a.centers[2 * g], cy = a.centers[2 * g + 1];
          const int x_lo = (int)floorf(sample_coord(__fadd_rn(-a.reach_px, cx), a.stride, (float)W, hw));
          const int x_hi = min((int)floorf(sample_coord(__fadd_rn(a.reach_px, cx), a.stride, (float)W, hw)) + 1, W - 1);
          const int y_lo = (int)floorf(sample_coord(__fadd_rn(-a.reach_px, cy), a.stride, (float)H, hh));
          const int y_hi = min((int)floorf(sample_coord(__fadd_rn(a.reach_px, cy), a.stride, (float)H, hh)) + 1, H - 1);
          hit = x_hi >= tx0 && x_lo < tx0 + LB_T && y_hi >= ty0 && y_lo < ty0 + LB_T;
        }
        const unsigned m = __ballot_sync(0xffffffffu, hit);
        if (hit) s_cand[n + __popc(m & ((1u << lane) - 1u))] = g;
        n += __popc(m);
      }
      if (lane == 0) s_ncand = n;
    }
    __syncthreads();
    const int ncand = s_ncand;
    // ---- B: bag by bag: warp w evaluates samples 32w..32w+31 (K <= 32 * nwarps per pass), relevant samples appended in k order
    for (int ci = 0; ci < ncand; ++ci) {
      const int g = s_cand[ci];
      for (int kb = 0; kb < K; kb += 32 * nwarps) {
        const int k = kb + 32 * warp + lane;
        int cells = -1;
        float tw[4] = {0.f, 0.f, 0.f, 0.f};
        bool rel = false;
        if (k < K) {
          const float px = __fadd_rn(a.offsets[2 * k], a.centers[2 * g]), py = __fadd_rn(a.offsets[2 * k + 1], a.centers[2 * g + 1]);
          const float ix = sample_coord(px, a.stride, (float)W, hw), iy = sample_coord(py, a.stride, (float)H, hh);
          const float x0f = floorf(ix), y0f = floorf(iy);
          const int x0 = (int)x0f, y0 = (int)y0f;
          const int x1 = min(x0 + 1, W - 1), y1 = min(y0 + 1, H - 1);
          const float ex = __fsub_rn(__fadd_rn(x0f, 1.f), ix), wx = __fsub_rn(ix, x0f);
          const float ey = __fsub_rn(__fadd_rn(y0f, 1.f), iy), wy = __fsub_rn(iy, y0f);
          tw[0] = __fmul_rn(ex, ey); tw[1] = __fmul_rn(wx, ey); tw[2] = __fmul_rn(ex, wy); tw[3] = __fmul_rn(wx, wy);
          const int lx0 = x0 - tx0, lx1 = x1 - tx0, ly0 = y0 - ty0, ly1 = y1 - ty0;
          const bool inx0 = (unsigned)lx0 < (unsigned)LB_T, inx1 = (unsigned)lx1 < (unsigned)LB_T;
          const bool iny0 = (unsigned)ly0 < (unsigned)LB_T, iny1 = (unsigned)ly1 < (unsigned)LB_T;
          const int c0 = (inx0 && iny0) ? ly0 * LB_T + lx0 : -1, c1 = (inx1 && iny0) ? ly0 * LB_T + lx1 : -1;
          const int c2 = (inx0 && iny1) ? ly1 * LB_T + lx0 : -1, c3 = (inx1 && iny1) ? ly1 * LB_T + lx1 : -1;
          // a clamped east / south tap repeats its neighbour's cell with weight 0: keep it (adds 0), the arithmetic matches the reference's
          cells = (c0 & 0xff) | ((c1 & 0xff) << 8) | ((c2 & 0xff) << 16) | ((c3 & 0xff) << 24);
          rel = (c0 >= 0) || (c1 >= 0) || (c2 >= 0) || (c3 >= 0);
        }
        const unsigned m = __ballot_sync(0xffffffffu, rel);
        if (lane == 0) s_wcnt[warp] = __popc(m);
        __syncthreads();
        int base = s_nrec, total = 0;
        for (int w = 0; w < nwarps; ++w) { if (w < warp) base += s_wcnt[w]; total += s_wcnt[w]; }
        if (s_nrec + total > LB_REC) {                                      // CTA-uniform: flush first, then append
          process();
          base -= 0;                                                        // s_nrec is 0 now
          base = 0;
          for (int w = 0; w < warp; ++w) base += s_wcnt[w];
        }
        if (rel) {
          LbRec rec;
          rec.g = g; rec.k = k; rec.wk = a.weight[(size_t)g * K + k]; rec.cells = cells;
          rec.w[0] = tw[0]; rec.w[1] = tw[1]; rec.w[2] = tw[2]; rec.w[3] = tw[3];
          s_rec[base + __popc(m & ((1u << lane) - 1u))] = rec;
        }
        __syncthreads();
        if (tid == 0) s_nrec += total;
        __syncthreads();
      }
    }
  }
  __syncthreads();
  process();
  // ---- D: + neg-loss term of the cell itself, write the tile (every channel of every in-map cell)
  const int y = ty0 + my_cell / LB_T, x = tx0 + my_cell % LB_T;
  if (y < H && x < W) {
    const float s_neg = (a.lmap && a.scale_neg) ? a.scale_neg[0] : 0.f;
    const size_t cellg = ((size_t)b * H + y) * W + x;
    float* dst = a.dlmap + cellg * LD + 32 * my_grp;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      float v[4] = {acc[4 * q], acc[4 * q + 1], acc[4 * q + 2], acc[4 * q + 3]};
      if (s_neg != 0.f) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int ch = 32 * my_grp + 4 * q + j;
          if (ch < N && a.neg_mask[cellg * N + ch]) {
            const float sg = fast_sigmoid(a.lmap[cellg * LD + ch]);
            v[j] += s_neg * gfocal_dp_f(sg, 0.f, a.eps) * sg * (1.f - sg);
          }
        }
      }
      *reinterpret_cast<float4*>(dst + 4 * q) = make_float4(v[0], v[1], v[2], v[3]);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------------------
// Scatter form of the same gradient (default: fastest; NOT bit-reproducible because the map accumulation uses fp32 vector atomics —
// the tile kernel above is the deterministic mode).  One CTA per bag: the bag's tap table goes to shared memory once, then thread
// (sample slice, 4-class group) loads the cls / ins float4 of its classes, forms the gradient from the forward's (m, 1/T, p, gfocal')
// and adds w_tap * gradient straight into the zero-initialised gradient map (red.global.add.v4.f32).  Compared with round 1's chain the
// (G,K,2N) gradient tensor is never written (740 MB + 740 MB) and the three latency-bound passes of mil_bwd (943 us) disappear.
// ---------------------------------------------------------------------------------------------------------------------------------
constexpr int LS_THREADS = 320;

struct LsTap { int o[4]; float w[4]; };

__global__ void __launch_bounds__(LS_THREADS)
cpr_loss_bwd_scatter_kernel(const LossBwdArgs a, const int32_t* __restrict__ bag_img) {
  extern __shared__ LsTap s_tap[];                     // [K]
  const int g = blockIdx.x;
  const int H = a.H, W = a.W, N = a.N, NP = a.NP, LD = a.LD, K = a.K;
  const int b = bag_img[g];
  const float cx = a.centers[2 * g], cy = a.centers[2 * g + 1];
  for (int k = threadIdx.x; k < K; k += LS_THREADS) {
    const Taps t = make_taps(__fadd_rn(a.offsets[2 * k], cx), __fadd_rn(a.offsets[2 * k + 1], cy), a.stride, H, W);
    LsTap r;
    r.o[0] = t.o00; r.o[1] = t.o01; r.o[2] = t.o10; r.o[3] = t.o11;
    r.w[0] = t.w00; r.w[1] = t.w01; r.w[2] = t.w10; r.w[3] = t.w11;
    s_tap[k] = r;
  }
  const int ng = (N + 3) >> 2;                         // 4-class groups
  const int slices = LS_THREADS / ng;
  const int q = threadIdx.x % ng, slice = threadIdx.x / ng;
  __syncthreads();
  if (slice >= slices) return;
  const float s_mil = a.scale_mil ? a.scale_mil[0] : 0.f;
  const float sgt = (a.scale_gt && a.wc) ? a.scale_gt[0] * a.wc[g] : 0.f;
  const int lab = a.labels[g];
  float cm[4], cit[4], cpb[4], cgd[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int c = 4 * q + j;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c < N) v = __ldg(a.coef + (size_t)g * N + c);
    cm[j] = v.x; cit[j] = v.y; cpb[j] = v.z; cgd[j] = s_mil * v.w;
  }
  float* map = a.dlmap + (size_t)b * H * W * LD;
  for (int k = slice; k < K; k += slices) {
    const float* row = a.bl + ((size_t)g * K + k) * LD;
    const float4 xc4 = __ldcs(reinterpret_cast<const float4*>(row + 4 * q));
    const float4 xi4 = __ldcs(reinterpret_cast<const float4*>(row + NP + 4 * q));
    const float wk = a.weight[(size_t)g * K + k];
    const float xc[4] = {xc4.x, xc4.y, xc4.z, xc4.w}, xi[4] = {xi4.x, xi4.y, xi4.z, xi4.w};
    float dc[4], di[4];
    const bool centre = (k == K - 1) && sgt != 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = 4 * q + j;
      const float sg = fast_sigmoid(xc[j]);
      const float gpi = cgd[j] * (__expf(xi[j] - cm[j]) * wk * cit[j]);
      dc[j] = gpi * sg * (1.f - sg);
      di[j] = gpi * (sg - cpb[j]);
      if (centre) dc[j] += sgt * gfocal_dp_f(sg, c == lab ? 1.f : 0.f, a.eps) * sg * (1.f - sg);
      if (c >= N) { dc[j] = 0.f; di[j] = 0.f; }
    }
    const LsTap t = s_tap[k];
#pragma unroll
    for (int tt = 0; tt < 4; ++tt) {
      const float w = t.w[tt];
      if (w != 0.f) {
        float* base = map + (size_t)t.o[tt] * LD;
        atomicAdd(reinterpret_cast<float4*>(base + 4 * q), make_float4(w * dc[0], w * dc[1], w * dc[2], w * dc[3]));
        atomicAdd(reinterpret_cast<float4*>(base + NP + 4 * q), make_float4(w * di[0], w * di[1], w * di[2], w * di[3]));
      }
    }
  }
}

// coef[g][c] = (max_k ins, 1/T or 0, bag prob, label_weight * gfocal'(prob, onehot(label)))  from the forward's outputs
__global__ void __launch_bounds__(256)
mil_coef_kernel(const float* __restrict__ mt, const float* __restrict__ bag_prob, const float* __restrict__ lw,
                const int32_t* __restrict__ labels, int G, int N, float eps, float4* __restrict__ coef) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= G * N) return;
  const int g = i / N, c = i - g * N;
  const float p = bag_prob[i];
  coef[i] = make_float4(mt[2 * i], mt[2 * i + 1], p, lw[g] * gfocal_dp_f(p, c == labels[g] ? 1.f : 0.f, eps));
}

}  // namespace ptb

using namespace ptb;

extern "C" uint64_t ptb_cpr_loss_bwd_map_workspace(int G, int num_classes) {
  return (uint64_t)(G > 0 ? G : 1) * (uint64_t)(num_classes > 0 ? num_classes : 1) * sizeof(float4);
}

extern "C" int ptb_cpr_loss_bwd_map(const float* bag_logits, const float* weight, const float* mil_mt, const float* bag_prob,
                                    const float* label_weight, const int32_t* labels, const float* centers, const int32_t* img_ptr,
                                    const float* offsets, int B, int H, int W, int G, int K, int num_classes, int ins_off, int ld,
                                    float stride, float reach_px, float eps, const float* scale_mil, const float* scale_gt,
                                    const float* valid_center, const float* logit_map, const uint8_t* neg_mask, const float* scale_neg,
                                    void* workspace, float* grad_map, void* stream) {
  PTB_REQUIRE(B > 0 && H > 0 && W > 0 && G >= 0 && K > 0 && num_classes > 0 && num_classes <= 32 * LB_NIT, "shape (num_classes <= 256)");
  PTB_REQUIRE(ld >= ins_off + num_classes && ins_off >= num_classes && stride > 0.f && reach_px >= 0.f, "ld / ins_off / stride");
  PTB_REQUIRE(ld % 32 == 0 && ld <= 512, "ld must be a multiple of 32 (32-channel register groups), at most 512");
  PTB_REQUIRE(K <= LB_MAXK, "at most 320 samples per bag");
  PTB_REQUIRE(img_ptr && grad_map && workspace &&
                  (G == 0 || (bag_logits && weight && mil_mt && bag_prob && label_weight && labels && centers && offsets)), "NULL input");
  PTB_REQUIRE(!logit_map || (neg_mask && scale_neg), "the neg term needs logit_map, neg_mask and scale_neg");
  PTB_REQUIRE(((uintptr_t)workspace % 16 == 0) && ((uintptr_t)grad_map % 16 == 0), "16-byte alignment");
  cudaStream_t st = (cudaStream_t)stream;
  float4* coef = reinterpret_cast<float4*>(workspace);
  if (G > 0) {
    mil_coef_kernel<<<(G * num_classes + 255) / 256, 256, 0, st>>>(mil_mt, bag_prob, label_weight, labels, G, num_classes, eps, coef);
    int rc = check_launch("ptb_cpr_loss_bwd_map/coef");
    if (rc) return rc;
  }
  LossBwdArgs a;
  a.bl = bag_logits; a.weight = weight; a.coef = coef; a.labels = labels;
  a.centers = centers; a.img_ptr = img_ptr; a.offsets = offsets; a.scale_mil = scale_mil; a.scale_gt = scale_gt; a.wc = valid_center;
  a.lmap = logit_map; a.neg_mask = neg_mask; a.scale_neg = scale_neg; a.dlmap = grad_map;
  a.H = H; a.W = W; a.N = num_classes; a.NP = ins_off; a.LD = ld; a.K = K; a.stride = stride; a.reach_px = reach_px; a.eps = eps;
  const size_t smem = (size_t)LB_ROUND * (ld + 4) * sizeof(float);
  const int threads = LB_CELLS * (ld / 32);
  PTB_REQUIRE(threads <= 320 || ld <= 512, "ld");
  if (threads > 320) return fail("%s", "ptb_cpr_loss_bwd_map: ld > 160 needs more than 320 threads per tile (not built)");
  // the kernel's static shared memory (record buffer, candidates, hit list: ~21 KB) counts against the 48 KB that need no opt-in
  static int static_smem = -1;
  if (static_smem < 0) {
    cudaFuncAttributes fa;
    if (cudaFuncGetAttributes(&fa, cpr_loss_bwd_tile_kernel) != cudaSuccess) return fail("%s", "ptb_cpr_loss_bwd_map: cudaFuncGetAttributes failed");
    static_smem = (int)fa.sharedSizeBytes;
  }
  if (static_smem + smem > 48 * 1024 &&
      cudaFuncSetAttribute(cpr_loss_bwd_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return fail("%s", "ptb_cpr_loss_bwd_map: shared memory opt-in failed");
  dim3 grid((W + LB_T - 1) / LB_T, (H + LB_T - 1) / LB_T, B);
  cpr_loss_bwd_tile_kernel<<<grid, threads, smem, st>>>(a);
  return check_launch("ptb_cpr_loss_bwd_map");
}

extern "C" int ptb_cpr_loss_bwd_scatter(const float* bag_logits, const float* weight, const float* mil_mt, const float* bag_prob,
                                        const float* label_weight, const int32_t* labels, const float* centers, const int32_t* bag_img,
                                        const float* offsets, int B, int H, int W, int G, int K, int num_classes, int ins_off, int ld,
                                        float stride, float eps, const float* scale_mil, const float* scale_gt, const float* valid_center,
                                        void* workspace, float* grad_map, void* stream) {
  PTB_REQUIRE(B > 0 && H > 0 && W > 0 && G >= 0 && K > 0 && num_classes > 0 && num_classes <= 4 * LS_THREADS, "shape");
  PTB_REQUIRE(ld >= ins_off + num_classes && ins_off >= num_classes && ins_off % 4 == 0 && ld % 4 == 0 && stride > 0.f, "ld / ins_off / stride");
  if (G == 0) return 0;
  PTB_REQUIRE(bag_logits && weight && mil_mt && bag_prob && label_weight && labels && centers && bag_img && offsets && workspace && grad_map,
              "NULL input");
  PTB_REQUIRE(((uintptr_t)workspace % 16 == 0) && ((uintptr_t)grad_map % 16 == 0) && ((uintptr_t)bag_logits % 16 == 0), "16-byte alignment");
  cudaStream_t st = (cudaStream_t)stream;
  float4* coef = reinterpret_cast<float4*>(workspace);
  mil_coef_kernel<<<(G * num_classes + 255) / 256, 256, 0, st>>>(mil_mt, bag_prob, label_weight, labels, G, num_classes, eps, coef);
  int rc = check_launch("ptb_cpr_loss_bwd_scatter/coef");
  if (rc) return rc;
  LossBwdArgs a;
  a.bl = bag_logits; a.weight = weight; a.coef = coef; a.labels = labels;
  a.centers = centers; a.img_ptr = nullptr; a.offsets = offsets; a.scale_mil = scale_mil; a.scale_gt = scale_gt; a.wc = valid_center;
  a.lmap = nullptr; a.neg_mask = nullptr; a.scale_neg = nullptr; a.dlmap = grad_map;
  a.H = H; a.W = W; a.N = num_classes; a.NP = ins_off; a.LD = ld; a.K = K; a.stride = stride; a.reach_px = 0.f; a.eps = eps;
  const size_t smem = (size_t)K * sizeof(LsTap);
  PTB_REQUIRE(smem <= 200 * 1024, "bag too large for shared memory");
  if (smem > 40 * 1024 &&
      cudaFuncSetAttribute(cpr_loss_bwd_scatter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return fail("%s", "ptb_cpr_loss_bwd_scatter: shared memory opt-in failed");
  cpr_loss_bwd_scatter_kernel<<<G, LS_THREADS, smem, st>>>(a, bag_img);
  return check_launch("ptb_cpr_loss_bwd_scatter");
}
