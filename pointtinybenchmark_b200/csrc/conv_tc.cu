// Dense convolutions of the head on the 5th-gen tensor cores (tcgen05 + TMEM + TMA), fp32-accurate by operand splitting:
// conv3x3 (stride 1, pad 1) and conv1x1 / per-cell Linear, Cin % 32 == 0 (fp16 mode) or Cin % 16 == 0 (TF32 mode), up to 256
// output channels, optional bias, optional GroupNorm statistics in the epilogue; GroupNorm-apply + ReLU + operand split is a
// second, HBM-bound kernel.  Replaces the cuDNN / cuBLAS calls behind CPRHead.forward_single / P2PHead.forward_single
// (cpr_head.py:1033-1043, p2p_head.py:113-123: 4 x ConvModule(conv3x3 + GN(32) + ReLU), 79.3 GFLOP per image), the
// per-sample cls_out / ins_out Linear of CPRHead.get_pts_outs (cpr_head.py:1045-1078, applied once per map cell here) and
// P2PHead's cls_out / reg_out conv3x3.
//
// Implicit GEMM:  M = output pixels (tile = 8 rows x 16 cols = 128 pixels of one image), N = n_mma <= 256 output channels,
//                 K = taps x Cin.  One K-block = (tap, 64 B of input channels) = one SWIZZLE_64B row.
//   * A operand: 4-D TMA box {64 B ch, 16 w, 8 h, 1 img} of the channels-last activation at the tap-shifted origin;
//     out-of-bounds (the zero padding of the conv and partial edge tiles) is zero-filled by the TMA unit.
//   * B operand: 2-D TMA box {64 B k, n_mma co} of the packed weights W2[co][tap*Cin + ci].
//   * fp32 accuracy (the head's logits must match the fp32 reference to 1e-4).  Every operand is split x = hi + lo and three
//     MMAs per k-step accumulate hi*hi + lo*hi + hi*lo (the lo*lo term is below 2^-22 |a||b|):
//       F16 = true  (default): hi = fp16(x*s), lo = fp16(x*s - hi) with one power-of-two scale s per tensor (undone exactly in
//                    the epilogue), kind::f16, 32 channels per K-block  -> 0.37 ms per 256->256 layer at the headline shape;
//       F16 = false: hi = x with the 13 low mantissa bits cleared (exact TF32), lo = x - hi (exact), kind::tf32, 16 channels
//                    per K-block (half the MMA rate)                    -> 0.62 ms per layer.
//   * TMEM: the tensor core adds into the fp32 accumulator with truncation, i.e. every accumulate step costs ~0.5 ulp of
//     the accumulator (measured with one accumulator: 2-5e-5 relative).  The two small correction products therefore go to
//     their OWN 256-column accumulator (their truncation is 2^-11 smaller in absolute terms); the epilogue adds the two in
//     fp32 (round-to-nearest).  512 columns = whole TMEM, so the epilogue of a tile cannot overlap the next tile's MMAs
//     beyond the early release below — measured cost 0.05 ms of 0.37 ms per layer.
//   * warp roles (192 threads, 1 CTA / SM, persistent over tiles): warp 0 = TMA producer, warp 1 = MMA issuer (+TMEM
//     allocator), warps 2-5 = epilogue.  Four 48 KB smem stages (mbarrier full/empty ring): with two 96 KB stages the tensor
//     pipe was only 62 % busy (ncu) because one K-block of loads could not hide behind one K-block of MMAs.
//   * epilogue: per 32-column chunk tcgen05.ld (main + correction) -> one tcgen05.wait::ld -> add, scale, bias -> staged in a
//     double-buffered SWIZZLE_128B smem tile -> cp.async.bulk.tensor.4d store (the TMA unit clips partial edge tiles);
//     GroupNorm sum / sum of squares per (image, group) by a halving butterfly over the 32 lanes + fp64 atomics; the TMEM
//     "empty" barrier is arrived right after the last tcgen05.ld so the next tile's MMAs start while the tail is stored.
#include "tc_ptx.cuh"
#include <stdlib.h>

namespace ptb {

constexpr int CV_TH = 8, CV_TW = 16;            // output tile (pixels)
constexpr int CV_BM = CV_TH * CV_TW;            // 128
constexpr int CV_N = 256;                       // output channels
constexpr int CV_KB = 16;                       // fp32/TF32 input channels per K-block (64 B = one SWIZZLE_64B row)
constexpr int CV_KB_F16 = 32;                   // fp16 input channels per K-block (also 64 B)
constexpr int CV_STAGES = 4;                    // 4 x 48 KB ring: 3 K-blocks of loads in flight behind the MMA
constexpr uint32_t CV_A_BYTES = CV_BM * CV_KB * 4;          // 8 KB
constexpr uint32_t CV_B_BYTES = CV_N * CV_KB * 4;           // 16 KB
constexpr uint32_t CV_STAGE_BYTES = 2 * CV_A_BYTES + 2 * CV_B_BYTES;   // 48 KB
constexpr uint32_t CV_OUT_BYTES = CV_BM * 32 * 4;              // one 128-row x 32-column fp32 output chunk (16 KB)
constexpr uint32_t CV_SMEM_BYTES = CV_STAGES * CV_STAGE_BYTES + 2 * CV_OUT_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
constexpr int CV_THREADS = 192;
// CTA-pair mode (CL = 3): each CTA stages half of the weight tile -> 32 KB stages, five of them, and the freed shared memory holds a
// second pair of output staging buffers for a second group of four epilogue warps (columns 128..255): the accumulators are read out
// twice as fast, and it is this read-out — not the stores — that keeps the tensor pipe waiting between tiles (TMEM is full).
constexpr int CV_STAGES_PAIR = 5;
constexpr uint32_t CV_STAGE_BYTES_PAIR = 2 * CV_A_BYTES + CV_B_BYTES;                                  // 32 KB
constexpr int CV_THREADS_PAIR = 64 + 8 * 32;                                                           // TMA + MMA + 8 epilogue warps
constexpr uint32_t CV_SMEM_BYTES_PAIR = CV_STAGES_PAIR * CV_STAGE_BYTES_PAIR + 4 * CV_OUT_BYTES + 1024 + 256;

// K-major, SWIZZLE_64B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): 8-row atoms of 64 B rows,
// atoms 512 B apart (SBO), version 1 (sm_100), layout type 4 (SWIZZLE_64B)
__device__ __forceinline__ uint64_t umma_desc_sw(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);            // start address  [0,14)
  d |= (uint64_t)1 << 16;                                  // leading byte offset (unused for swizzled K-major) = 1
  d |= (uint64_t)((8 * CV_KB * 4) >> 4) << 32;             // stride byte offset  [32,46): 8 rows x 64 B
  d |= (uint64_t)1 << 46;                                  // version = 1
  d |= (uint64_t)4 << 61;                                  // SWIZZLE_64B
  return d;
}
// cute::UMMA::InstrDescriptor for kind::tf32: D=f32, A=B=tf32, both K-major, M=128, N=256, dense, no negate
__host__ __device__ constexpr uint32_t umma_idesc_tf32_m128_n256() {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(CV_N >> 3) << 17) | ((uint32_t)(CV_BM >> 4) << 24);
}
// same for kind::f16 with fp16 operands (a_format = b_format = F16 = 0), fp32 accumulate
__host__ __device__ constexpr uint32_t umma_idesc_f16_m128_n256() {
  return (1u << 4) | ((uint32_t)(CV_N >> 3) << 17) | ((uint32_t)(CV_BM >> 4) << 24);
}

// Output tiling (round 2).  A tile is always 128 pixels (the UMMA M of one CTA); the main region uses 8 x 16 tiles and the two edge
// strips that 8 x 16 tiles would cover half-empty get their own shapes: a bottom strip of <= 4 rows is covered by 4 x 32 tiles, a right
// strip of <= 8 columns by 16 x 8 tiles.  At the headline 100 x 168 map that is 132 tiles per image instead of 143 (13 x 11 with the
// last tile row and column half outside the image): 7.7 % fewer MMAs, loads and epilogues for the same output.
//   shape 0: 8 h x 16 w (main)     shape 1: 4 h x 32 w (bottom strip, all columns)     shape 2: 16 h x 8 w (right strip, rows above the bottom strip)
struct ConvShape {
  int B, H, W, Cin;
  int tiles_h, tiles_w;   // main region, in 8 x 16 tiles
  int n_main, n_right, n_bottom, per_img, n_tiles;
  int right_w0, right_h;  // right strip: first column, number of rows it covers (rows below belong to the bottom strip)
  int bottom_h0;          // bottom strip: first row
  // Tail wave (pair mode): the n_groups tile pairs are dealt round-robin to the n_units CTA pairs, `q_full` full rounds and a last round
  // of `rem` pairs that used to leave most SMs idle for a whole tile time (528 = 7 x 74 + 10 at the headline shape).  The tail tiles are
  // therefore split into `tail_s` column slices (N = 256 / tail_s output channels each, independent outputs: no reduction), one slice per
  // unit: the last round takes ~1/tail_s of a tile time.  tail_s = 1: no split.
  int q_full, rem, tail_s;
  int taps;       // 9: conv3x3 (pad 1), 1: conv1x1 / per-cell Linear
  int n_mma;      // MMA N (multiple of 16, <= 256): output channels rounded up; weight rows beyond n_out are zero
  int n_out;      // output channels actually stored
  int ldy;        // floats per output pixel row
};

struct ConvMaps {          // by-value __grid_constant__ kernel argument (15 x 128 B)
  CUtensorMap x[3][2];     // activations (hi, lo) with the box of tile shape 0 / 1 / 2
  CUtensorMap y[3];        // output, same boxes (the right strip's map is clipped to right_h rows)
  CUtensorMap w[3][2];     // packed weights (hi, lo); box rows = n_mma/2, n_mma/4, n_mma/8 (full tile, half- and quarter-width tail slices)
};
struct TileAt {
  int b, h0, w0, shape, twl;     // image, origin, shape id, log2(tile width)
};
__device__ __forceinline__ TileAt tile_at(const ConvShape& cs, int tile) {
  TileAt t;
  t.b = tile / cs.per_img;
  const int r = tile - t.b * cs.per_img;
  if (r < cs.n_main) {
    t.shape = 0; t.twl = 4; t.h0 = (r / cs.tiles_w) * 8; t.w0 = (r % cs.tiles_w) * 16;
  } else if (r < cs.n_main + cs.n_right) {
    t.shape = 2; t.twl = 3; t.h0 = (r - cs.n_main) * 16; t.w0 = cs.right_w0;
  } else {
    t.shape = 1; t.twl = 5; t.h0 = cs.bottom_h0; t.w0 = (r - cs.n_main - cs.n_right) * 32;
  }
  return t;
}

struct WorkItem {
  int grp;        // tile group (pair of tiles in cluster modes)
  int n0, nn;     // output-channel slice [n0, n0 + nn) this unit computes for the group
  int kind;       // 0: full width, 1: half, 2: quarter (selects the weight map)
};
// k-th work item of `unit`; false when the unit is done.  Rounds 0 .. q_full-1: group unit + k*n_units, full width; round q_full: the
// tail (see ConvShape).  Every role of the CTA (producer, MMA issuer, epilogue) walks the same list.
__device__ __forceinline__ bool work_item(const ConvShape& cs, int unit, int n_units, int k, WorkItem& wi) {
  if (k < cs.q_full) { wi.grp = unit + k * n_units; wi.n0 = 0; wi.nn = cs.n_mma; wi.kind = 0; return true; }
  if (k > cs.q_full || unit >= cs.rem * cs.tail_s) return false;
  const int sl = unit / cs.rem;
  wi.grp = cs.q_full * n_units + (unit - sl * cs.rem);
  wi.nn = cs.n_mma / cs.tail_s;
  wi.n0 = sl * wi.nn;
  wi.kind = cs.tail_s == 4 ? 2 : (cs.tail_s == 2 ? 1 : 0);
  return true;
}

// CL = 3 (round 2, default for 256-channel outputs): CTA PAIRS issuing ONE tcgen05.mma.cta_group::2 per product over both SMs
// (M = 256 = the pair's two pixel tiles, N = 256): each CTA stages its own activation tile and only HALF of the weight tile, the
// tensor cores exchange the halves.  Per CTA and K-step the shared-memory traffic drops from 36 KB of MMA operand reads + 24 KB of TMA
// fill (160 B/clk at full tensor rate, above the 128 B/clk the SM has: ncu showed the tensor pipe 63 % active, l1tex 78 % busy) to
// 24 KB + 16 KB (107 B/clk).  The leader CTA's MMA thread issues for both; its "full" barrier collects both CTAs' TMA bytes
// (cp.async.bulk.tensor.cta_group::2 with the leader's barrier as completion target), tcgen05.commit.cta_group::2 multicasts the
// "stage free" / "accumulator ready" arrivals to both CTAs, and the peer's epilogue warps release the accumulators with remote
// mbarrier arrives.  Every CTA still stores its own 128-pixel tile and adds its own GroupNorm partial sums.
// CL = 1: independent CTAs.  CL = 2: clusters of two CTAs working on neighbouring tiles in lock-step; each CTA fetches
// its own activation tile and HALF of the weight tile, TMA-multicast into both CTAs' shared memory.  The weights are
// 2/3 of the operand bytes, and the kernel is bound by the L2->SM operand stream (41 B/clk/SM measured), so this cuts
// the stream per SM from 48 KB to 32 KB per K-block.
// F16 = false: 3xTF32 (operands fp32 hi/lo).  F16 = true: 2-term fp16 split (x = h + l, 22 significant bits):
// h*h + l*h + h*l with kind::f16 — the same three MMAs per k-step but K = 16 per MMA, i.e. HALF the tensor-pipe time
// (the 3xTF32 kernel is tensor bound) and half the operand bytes.  out_scale undoes the power-of-two scaling of the
// fp16 operands (exact).
template <int CL, bool F16>
__global__ void __launch_bounds__(CL == 3 ? CV_THREADS_PAIR : CV_THREADS, 1)
conv_tc_kernel(const __grid_constant__ ConvMaps mp, ConvShape cs, float* __restrict__ y, double* __restrict__ stats /*[B][32][2] or NULL*/,
                      float out_scale, const float* __restrict__ dev_out_scale, const float* __restrict__ bias) {
  constexpr int KBC = F16 ? CV_KB_F16 : CV_KB;      // channels per K-block
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;      // SWIZZLE_128B atoms need 1024 B alignment
  constexpr int NST = CL == 3 ? CV_STAGES_PAIR : CV_STAGES;              // smem ring depth
  constexpr uint32_t STB = CL == 3 ? CV_STAGE_BYTES_PAIR : CV_STAGE_BYTES;
  constexpr uint32_t BLO = CL == 3 ? CV_B_BYTES / 2 : CV_B_BYTES;        // offset of the weight lo tile behind the hi tile
  constexpr int NEG = CL == 3 ? 2 : 1;                                   // epilogue warp groups (4 warps each, 128 / 256 columns each)
  const uint32_t out_base = smem_base + NST * STB;                       // NEG x 2 x 16 KB output staging (SWIZZLE_128B rows)
  const uint32_t bar_base = out_base + NEG * 2 * CV_OUT_BYTES;
  // barriers: full[4] | empty[4] | tmem_full | tmem_empty | tmem_ptr
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 64u + 8u * s; };
  auto tfull_bar = [&](int s) { return bar_base + 128u + 8u * s; };
  auto tempty_bar = [&](int s) { return bar_base + 144u + 8u * s; };
  const uint32_t tmem_slot = bar_base + 160u;
  uint8_t* smem_aligned = smem_raw + (smem_base - smem_u32(smem_raw));
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_aligned + NST * STB + NEG * 2 * CV_OUT_BYTES + 160);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kblocks_per_tap = cs.Cin / KBC;
  const int n_kb = cs.taps * kblocks_per_tap;
  // work distribution: unit u = blockIdx.x / CL owns tile groups u, u + n_units, ...; CTA `rank` of the cluster takes
  // tile CL*group + rank (a group's missing last tile is a dummy: loads + MMAs run, nothing is stored)
  constexpr int CSZ = CL >= 2 ? 2 : 1;   // CTAs per cluster
  const uint32_t rank = (CL >= 2) ? cluster_ctarank() : 0u;
  const int unit = blockIdx.x / CSZ, n_units = gridDim.x / CSZ;
  const int n_groups = (cs.n_tiles + CSZ - 1) / CSZ;

  if (threadIdx.x == 0) {
    for (int s = 0; s < NST; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), CL == 2 ? 2 : 1);       // CL 2: one tcgen05.commit per CTA of the cluster; CL 3: the leader's commit, multicast
    }
    mbar_init(tfull_bar(0), 1);
    mbar_init(tempty_bar(0), CL == 3 ? 16 : 4);       // one arrive per epilogue warp (CL 3: 8 warps of BOTH CTAs, on the leader's barrier)
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {     // TMEM: 512 columns = 2 accumulators of 128 lanes x 256 fp32 columns
    if (CL == 3) {     // pair allocation: one warp of EACH CTA
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(512u) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(512u) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  if (CL >= 2) cluster_sync_all();       // the peer's barriers exist before any multicast / remote arrive can land
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // =============================== TMA producer ===============================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      WorkItem wi;
      for (int k = 0; work_item(cs, unit, n_units, k, wi); ++k) {
        const int grp = wi.grp;
        const uint32_t b_bytes = (uint32_t)wi.nn * 64u;            // one weight operand tile of this item: nn rows x 64 B
        const uint32_t stage_tx = 2 * CV_A_BYTES + 2 * b_bytes;
        const int w_half = wi.nn / 2;
        int tile = CSZ * grp + (int)rank;
        if (tile >= cs.n_tiles) tile = cs.n_tiles - 1;              // dummy: re-load a valid tile, never stored
        const TileAt ta = tile_at(cs, tile);
        const int b = ta.b, h0 = ta.h0, w0 = ta.w0;
        const CUtensorMap* tm_xhi_p = &mp.x[ta.shape][0];
        const CUtensorMap* tm_xlo_p = &mp.x[ta.shape][1];
        for (int kb = 0; kb < n_kb; ++kb) {
          const int tap = kb / kblocks_per_tap, cblk = kb - tap * kblocks_per_tap;
          const int kh = cs.taps == 9 ? tap / 3 : 1, kw = cs.taps == 9 ? tap - (tap / 3) * 3 : 1;
          mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t sA_hi = smem_base + stage * STB;
          const uint32_t sA_lo = sA_hi + CV_A_BYTES;
          const uint32_t sB_hi = sA_lo + CV_A_BYTES;
          const uint32_t sB_lo = sB_hi + BLO;
          const int kcol = tap * cs.Cin + cblk * KBC;
          if (CL == 3) {
            // pair mode: my activation tile + MY half of the weight tile into my shared memory; all bytes are counted on the LEADER's barrier
            const uint32_t lead_full = mapa_rank(full_bar(stage), 0u);
            if (rank == 0) mbar_expect_tx(full_bar(stage), 2u * (2 * CV_A_BYTES + b_bytes));      // both CTAs: 2 x (A hi + lo + half B hi + lo)
            tma_load_4d_pair(tm_xhi_p, lead_full, sA_hi, cblk * KBC, w0 + kw - 1, h0 + kh - 1, b);
            tma_load_4d_pair(tm_xlo_p, lead_full, sA_lo, cblk * KBC, w0 + kw - 1, h0 + kh - 1, b);
            tma_load_2d_pair(&mp.w[wi.kind][0], lead_full, sB_hi, kcol, wi.n0 + (int)rank * w_half);
            tma_load_2d_pair(&mp.w[wi.kind][1], lead_full, sB_lo, kcol, wi.n0 + (int)rank * w_half);
            if (++stage == NST) { stage = 0; phase ^= 1u; }
            continue;
          }
          mbar_expect_tx(full_bar(stage), stage_tx);
          tma_load_4d(tm_xhi_p, full_bar(stage), sA_hi, cblk * KBC, w0 + kw - 1, h0 + kh - 1, b);
          tma_load_4d(tm_xlo_p, full_bar(stage), sA_lo, cblk * KBC, w0 + kw - 1, h0 + kh - 1, b);
          if (CL == 2) {     // my 128-row half of the weight tile, delivered to both CTAs (and both full barriers)
            const uint32_t half = rank * (b_bytes / 2);
            tma_load_2d_mc(&mp.w[0][0], full_bar(stage), sB_hi + half, kcol, (int)rank * (cs.n_mma / 2), (uint16_t)0x3);
            tma_load_2d_mc(&mp.w[0][1], full_bar(stage), sB_lo + half, kcol, (int)rank * (cs.n_mma / 2), (uint16_t)0x3);
          } else {
            tma_load_2d(&mp.w[0][0], full_bar(stage), sB_hi, kcol, 0);
            tma_load_2d(&mp.w[0][0], full_bar(stage), sB_hi + b_bytes / 2, kcol, cs.n_mma / 2);
            tma_load_2d(&mp.w[0][1], full_bar(stage), sB_lo, kcol, 0);
            tma_load_2d(&mp.w[0][1], full_bar(stage), sB_lo + b_bytes / 2, kcol, cs.n_mma / 2);
          }
          if (++stage == NST) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // =============================== MMA issuer ===============================
    if (lane == 0 && (CL != 3 || rank == 0)) {          // pair mode: the leader's thread issues for both CTAs
      uint32_t idesc0 = (F16 ? umma_idesc_f16_m128_n256() : umma_idesc_tf32_m128_n256()) & ~(0x3Fu << 17);
      if (CL == 3) idesc0 = (idesc0 & ~(0x1Fu << 24)) | ((uint32_t)(256 >> 4) << 24);      // M = 256 across the pair
      int stage = 0;
      uint32_t phase = 0;
      WorkItem wi;
      for (int it = 0; work_item(cs, unit, n_units, it, wi); ++it) {
        const uint32_t idesc = idesc0 | ((uint32_t)(wi.nn >> 3) << 17);                      // N = this item's channel slice
        const int acc = 0;
        const uint32_t acc_phase = (uint32_t)it & 1u;
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);          // epilogue has drained the accumulators
        tc_fence_after();
        const uint32_t d_main = tmem_base, d_corr = tmem_base + CV_N;
        for (int kb = 0; kb < n_kb; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          const uint32_t sA_hi = smem_base + stage * STB;
          const uint32_t sA_lo = sA_hi + CV_A_BYTES;
          const uint32_t sB_hi = sA_lo + CV_A_BYTES;
          const uint32_t sB_lo = sB_hi + BLO;
#pragma unroll
          for (int k = 0; k < 2; ++k) {                       // UMMA_K = 32 B (8 tf32 / 16 fp16) inside the 64 B swizzle row
            const uint64_t a_hi = umma_desc_sw(sA_hi + 32u * k), a_lo = umma_desc_sw(sA_lo + 32u * k);
            const uint64_t b_hi = umma_desc_sw(sB_hi + 32u * k), b_lo = umma_desc_sw(sB_lo + 32u * k);
            if (CL == 3) {
              umma_ss_pair<F16>(d_main, a_hi, b_hi, idesc, (kb | k) != 0);
              umma_ss_pair<F16>(d_corr, a_lo, b_hi, idesc, (kb | k) != 0);
              umma_ss_pair<F16>(d_corr, a_hi, b_lo, idesc, 1u);
            } else {
              umma_ss<F16>(d_main, a_hi, b_hi, idesc, (kb | k) != 0);
              umma_ss<F16>(d_corr, a_lo, b_hi, idesc, (kb | k) != 0);
              umma_ss<F16>(d_corr, a_hi, b_lo, idesc, 1u);
            }
          }
          if (CL == 3) umma_commit_pair(empty_bar(stage), (uint16_t)0x3);      // stage free in both CTAs
          else if (CL == 2) umma_commit_mc(empty_bar(stage), (uint16_t)0x3);   // stage free in BOTH CTAs' books
          else umma_commit(empty_bar(stage));                  // smem stage free once these MMAs have read it
          if (++stage == NST) { stage = 0; phase ^= 1u; }
        }
        if (CL == 3) umma_commit_pair(tfull_bar(acc), (uint16_t)0x3);          // both CTAs' halves of the accumulators are complete
        else umma_commit(tfull_bar(acc));                      // accumulator complete
      }
    }
  } else {
    // =============================== epilogue (warps 2..5) ===============================
    const int q = warp & 3;                                    // TMEM lane quarter this warp may access
    const int eg = NEG == 2 ? (warp - 2) >> 2 : 0;             // epilogue group: columns [eg * 256 / NEG, (eg + 1) * 256 / NEG)
    constexpr int CPG = (CV_N / 32) / NEG;                     // 32-column chunks per group
    WorkItem wi;
    for (int it = 0; work_item(cs, unit, n_units, it, wi); ++it) {
      const int grp = wi.grp;
      const int acc = 0;
      const uint32_t acc_phase = (uint32_t)it & 1u;
      const int tile_raw = CSZ * grp + (int)rank;
      const bool dummy = tile_raw >= cs.n_tiles;
      const int tile = dummy ? cs.n_tiles - 1 : tile_raw;
      const TileAt ta = tile_at(cs, tile);
      const int b = ta.b, h0 = ta.h0, w0 = ta.w0;
      const CUtensorMap* tm_y_p = &mp.y[ta.shape];
      const int row = q * 32 + lane;                           // GEMM row = pixel inside the tile (h-major, tile-width pixels per row)
      const int h = h0 + (row >> ta.twl), w = w0 + (row & ((1 << ta.twl) - 1));
      const bool valid = !dummy && (h < (ta.shape == 2 ? cs.right_h : cs.H)) && (w < cs.W);
      mbar_wait(tfull_bar(acc), acc_phase);
      tc_fence_after();
      // TMEM chunk c of this item holds output columns 32 * (oc0 + c) ..; a tail slice has nn / 32 chunks, split between the groups
      const int oc0 = wi.n0 >> 5;
      const int n_chunks = min((cs.n_out + 31) / 32 - oc0, (wi.nn + 31) >> 5);
      const int cpg_item = NEG == 2 ? max(1, (wi.nn >> 5) / NEG) : CPG;
      const int c_lo = eg * cpg_item;
      const float sc = F16 ? (dev_out_scale ? __fmul_rn(out_scale, *dev_out_scale) : out_scale) : 1.f;   // powers of two: exact
      const bool issuer = (warp == 2 + 4 * eg) && (lane == 0);  // owns the bulk-store groups of its epilogue group
      const int c_end = min(n_chunks, c_lo + cpg_item);        // this group's chunks: [c_lo, c_end)
      auto grp_bar = [&]() { asm volatile("bar.sync %0, 128;" ::"r"(1 + eg) : "memory"); };
      // Chunk pipeline (8 x 32 columns, fully unrolled so every array index is static): the TMEM loads of chunk c+1 are in
      // flight while chunk c is scaled, staged and stored; the GroupNorm partial sums stay in registers until the accumulators
      // have been handed back to the MMA warp, so neither the TMEM latency nor the statistics sit in the exposed path.
      uint32_t bx[32], by[32], bz[32];       // main accumulator chunks alternate between bx / bz, by takes the correction
      float part[8 * CPG];                   // per-row (sum, sum of squares) of the 4 groups of each chunk
      const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
      if (c_lo < c_end) {
        tmem_ld32_nowait(t_lane + (uint32_t)(c_lo * 32), bx);
        tmem_ld32_nowait(t_lane + (uint32_t)(CV_N + c_lo * 32), by);
      }
      auto chunk = [&](const int j_, const int c, uint32_t (&cur)[32], uint32_t (&nxt)[32]) {
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          float f = __fadd_rn(__uint_as_float(cur[j]), __uint_as_float(by[j]));
          if (F16) f = __fmul_rn(f, sc);
          cur[j] = __float_as_uint(f);
        }
        if (c + 1 < c_end) {
          tmem_ld32_nowait(t_lane + (uint32_t)((c + 1) * 32), nxt);
          tmem_ld32_nowait(t_lane + (uint32_t)(CV_N + (c + 1) * 32), by);
        } else {                       // accumulators fully read: the MMA warp may start the next tile under the stores
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (CL == 3) mbar_arrive_cluster(mapa_rank(tempty_bar(acc), 0u));      // the leader's MMA thread waits for all 8 warps
            else mbar_arrive(tempty_bar(acc));
          }
        }
        if (bias) {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int col = (oc0 + c) * 32 + j;
            if (col < cs.n_out) cur[j] = __float_as_uint(__uint_as_float(cur[j]) + __ldg(bias + col));
          }
        }
        // ---- stage the 128 x 32 chunk in shared memory (SWIZZLE_128B: 16-byte slot j of row r lives at slot j ^ (r & 7),
        //      so the 32 lanes of a warp, one row each, write conflict-free) and hand it to the TMA unit: one bulk tensor
        //      store per chunk, fully coalesced, and the tile's out-of-range rows / columns are clipped by the hardware.
        const uint32_t buf = out_base + (uint32_t)(2 * eg + (j_ & 1)) * CV_OUT_BYTES;
        if (issuer) tma_store_wait_read<1>();                    // the store issued two chunks ago has drained this buffer
        grp_bar();
        {
          const uint32_t row_addr = buf + (uint32_t)row * 128u;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const uint32_t slot = (uint32_t)(j ^ (row & 7));
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(row_addr + slot * 16u), "r"(cur[4 * j]), "r"(cur[4 * j + 1]),
                         "r"(cur[4 * j + 2]), "r"(cur[4 * j + 3])
                         : "memory");
          }
        }
        fence_async_smem();
        grp_bar();
        if (issuer && !dummy) {
          tma_store_4d(tm_y_p, buf, (oc0 + c) * 32, w0, h0, b);
          tma_store_commit();
        }
        if (stats) {
          // GroupNorm(32 groups of 8 channels): this chunk covers groups 4c .. 4c+3; per-row partials only, reduced below
#pragma unroll
          for (int gq = 0; gq < 4; ++gq) {
            float s = 0.f, ss = 0.f;
            if (valid) {
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const float f = __uint_as_float(cur[8 * gq + j]);
                s += f;
                ss = fmaf(f, f, ss);
              }
            }
            part[8 * j_ + 2 * gq] = s;
            part[8 * j_ + 2 * gq + 1] = ss;
          }
        }
      };
#pragma unroll
      for (int j_ = 0; j_ < CPG; ++j_) {
        const int c = c_lo + j_;
        if (c < c_end) {
          if (j_ & 1) chunk(j_, c, bz, bx);
          else chunk(j_, c, bx, bz);
        }
      }
      if (stats) {
        // halving butterfly over the 32 rows of the warp per chunk: 9 shuffles instead of 40, the 8 totals end up on lanes
        // 0,4,..,28 which issue one fp64 atomic each.  Runs while the MMA warp is already working on the next tile.
#pragma unroll
        for (int j_ = 0; j_ < CPG; ++j_) {
          const int c = c_lo + j_;
          if (c < c_end) {
            float t[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) t[i] = part[8 * j_ + i];
            {
              const bool up = (lane & 16) != 0;
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const float send = up ? t[i] : t[i + 4];
                const float recv = __shfl_xor_sync(0xffffffffu, send, 16);
                t[i] = (up ? t[i + 4] : t[i]) + recv;
              }
            }
            {
              const bool up = (lane & 8) != 0;
#pragma unroll
              for (int i = 0; i < 2; ++i) {
                const float send = up ? t[i] : t[i + 2];
                const float recv = __shfl_xor_sync(0xffffffffu, send, 8);
                t[i] = (up ? t[i + 2] : t[i]) + recv;
              }
            }
            {
              const bool up = (lane & 4) != 0;
              const float send = up ? t[0] : t[1];
              const float recv = __shfl_xor_sync(0xffffffffu, send, 4);
              t[0] = (up ? t[1] : t[0]) + recv;
            }
            t[0] += __shfl_xor_sync(0xffffffffu, t[0], 2);
            t[0] += __shfl_xor_sync(0xffffffffu, t[0], 1);
            if ((lane & 3) == 0) {
              const int idx = ((lane & 16) ? 4 : 0) + ((lane & 8) ? 2 : 0) + ((lane & 4) ? 1 : 0);   // = 2*gq + {0: sum, 1: sumsq}
              atomicAdd(stats + ((size_t)b * 32 + (4 * (oc0 + c) + (idx >> 1))) * 2 + (idx & 1), (double)t[0]);
            }
          }
        }
      }
      if (c_lo >= c_end) {                   // nothing to read for this group (narrow outputs): release the accumulators right away
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (CL == 3) mbar_arrive_cluster(mapa_rank(tempty_bar(acc), 0u));
          else mbar_arrive(tempty_bar(acc));
        }
      }

    }
  }
  if (warp >= 2 && ((warp - 2) & 3) == 0 && lane == 0) tma_store_wait_all();     // every bulk tensor store of this CTA has landed
  __syncthreads();
  if (CL >= 2) cluster_sync_all();       // no CTA exits while the peer can still multicast into it / arrive on its barriers
  if (warp == 1) {
    if (CL == 3) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------------------------
// elementwise helpers (HBM-bound, 128-bit vectors)
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float tf32_hi(float x) { return __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); }

__global__ void __launch_bounds__(256)
split_tf32_kernel(const float4* __restrict__ x, long long n4, float4* __restrict__ hi, float4* __restrict__ lo) {
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n4; i += (long long)gridDim.x * 256) {
    const float4 v = __ldcs(x + i);
    float4 h = make_float4(tf32_hi(v.x), tf32_hi(v.y), tf32_hi(v.z), tf32_hi(v.w));
    hi[i] = h;
    lo[i] = make_float4(v.x - h.x, v.y - h.y, v.z - h.z, v.w - h.w);
  }
}

// y: raw conv output [B][HW][C]; stats: [B][G][2] (sum, sumsq) fp64.  out = relu((y-mean)*rstd*gamma + beta)
// written either as fp32 (out_lo == NULL) or as the TF32 hi/lo pair the next conv consumes.
__global__ void __launch_bounds__(256)
gn_relu_apply_kernel(const float4* __restrict__ y, const double* __restrict__ stats, const float* __restrict__ gamma,
                     const float* __restrict__ beta, int HW, int C, int groups, float eps, int relu, long long n4,
                     float4* __restrict__ out_hi, float4* __restrict__ out_lo) {
  const int c4n = C >> 2;
  const int cpg = C / groups;
  const double inv_n = 1.0 / ((double)HW * cpg);
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n4; i += (long long)gridDim.x * 256) {
    const int c = (int)(i % c4n) * 4;
    const long long pix = i / c4n;
    const int b = (int)(pix / HW);
    const int g = c / cpg;            // cpg is a multiple of 4 or the 4 channels share... (host guarantees cpg % 4 == 0)
    const double s = stats[((size_t)b * groups + g) * 2], ss = stats[((size_t)b * groups + g) * 2 + 1];
    const double mean = s * inv_n;
    double var = ss * inv_n - mean * mean;
    var = var < 0.0 ? 0.0 : var;
    const float rstd = (float)(1.0 / sqrt(var + (double)eps));
    const float mu = (float)mean;
    const float4 v = __ldcs(y + i);
    const float4 ga = *reinterpret_cast<const float4*>(gamma + c), be = *reinterpret_cast<const float4*>(beta + c);
    float4 o;
    o.x = fmaf((v.x - mu) * rstd, ga.x, be.x);
    o.y = fmaf((v.y - mu) * rstd, ga.y, be.y);
    o.z = fmaf((v.z - mu) * rstd, ga.z, be.z);
    o.w = fmaf((v.w - mu) * rstd, ga.w, be.w);
    if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
    if (out_lo) {
      const float4 h = make_float4(tf32_hi(o.x), tf32_hi(o.y), tf32_hi(o.z), tf32_hi(o.w));
      out_hi[i] = h;
      out_lo[i] = make_float4(o.x - h.x, o.y - h.y, o.z - h.z, o.w - h.w);
    } else {
      out_hi[i] = o;
    }
  }
}

// ---- fp16 two-term split (split_h2, tc_ptx.cuh) ----
__device__ __forceinline__ float amax4(float m, const float4 v) {
  return fmaxf(m, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
}

// pure HBM read: four independent 16-byte loads in flight per thread (B200 needs ~40 KB in flight per SM to saturate HBM)
__global__ void __launch_bounds__(256) amax_abs_kernel(const float4* __restrict__ x, long long n4, unsigned int* __restrict__ out_bits) {
  float m = 0.f;
  const long long step = (long long)gridDim.x * 256;
  long long i = (long long)blockIdx.x * 256 + threadIdx.x;
  for (; i + 3 * step < n4; i += 4 * step) {
    const float4 v0 = x[i], v1 = x[i + step], v2 = x[i + 2 * step], v3 = x[i + 3 * step];
    m = amax4(amax4(amax4(amax4(m, v0), v1), v2), v3);
  }
  for (; i < n4; i += step) m = amax4(m, x[i]);
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0) atomicMax(out_bits, __float_as_uint(m));     // non-negative floats order like their bits
}

__device__ __forceinline__ void split8(const float4 a, const float4 b, float scale, uint4& ph, uint4& pl) {
  __align__(16) __half h[8], l[8];
  split_h2(a.x * scale, h[0], l[0]); split_h2(a.y * scale, h[1], l[1]);
  split_h2(a.z * scale, h[2], l[2]); split_h2(a.w * scale, h[3], l[3]);
  split_h2(b.x * scale, h[4], l[4]); split_h2(b.y * scale, h[5], l[5]);
  split_h2(b.z * scale, h[6], l[6]); split_h2(b.w * scale, h[7], l[7]);
  ph = *reinterpret_cast<uint4*>(h);
  pl = *reinterpret_cast<uint4*>(l);
}

// hi/lo are [n] fp16; dev_amax (optional) selects a power-of-two scale on the device, its inverse is written to inv_scale_out.
// 8 elements per thread and step: 2 x 16-byte loads, 2 x 16-byte stores; two steps in flight.
__global__ void __launch_bounds__(256)
split_f16_kernel(const float4* __restrict__ x, long long n4, const unsigned int* __restrict__ dev_amax_bits,
                 uint2* __restrict__ hi, uint2* __restrict__ lo, float* __restrict__ inv_scale_out) {
  const float scale = dev_amax_bits ? pow2_scale_for(__uint_as_float(*dev_amax_bits)) : 1.f;
  if (inv_scale_out && blockIdx.x == 0 && threadIdx.x == 0) *inv_scale_out = 1.f / scale;
  const long long n8 = n4 >> 1;
  const long long step = (long long)gridDim.x * 256;
  uint4* hi8 = reinterpret_cast<uint4*>(hi);
  uint4* lo8 = reinterpret_cast<uint4*>(lo);
  const bool al16 = ((reinterpret_cast<uintptr_t>(hi) | reinterpret_cast<uintptr_t>(lo)) & 15) == 0;
  long long i = (long long)blockIdx.x * 256 + threadIdx.x;
  if (al16) {
    for (; i + step < n8; i += 2 * step) {
      const float4 a0 = __ldcs(x + 2 * i), a1 = __ldcs(x + 2 * i + 1);
      const float4 b0 = __ldcs(x + 2 * (i + step)), b1 = __ldcs(x + 2 * (i + step) + 1);
      uint4 ph, pl;
      split8(a0, a1, scale, ph, pl);
      hi8[i] = ph; lo8[i] = pl;
      split8(b0, b1, scale, ph, pl);
      hi8[i + step] = ph; lo8[i + step] = pl;
    }
    for (; i < n8; i += step) {
      uint4 ph, pl;
      split8(__ldcs(x + 2 * i), __ldcs(x + 2 * i + 1), scale, ph, pl);
      hi8[i] = ph; lo8[i] = pl;
    }
    i = 2 * n8 + (long long)blockIdx.x * 256 + threadIdx.x;       // odd float4 tail
  }
  for (; i < n4; i += step) {
    const float4 v = __ldcs(x + i);
    __half h[4], l[4];
    split_h2(v.x * scale, h[0], l[0]); split_h2(v.y * scale, h[1], l[1]);
    split_h2(v.z * scale, h[2], l[2]); split_h2(v.w * scale, h[3], l[3]);
    hi[i] = *reinterpret_cast<uint2*>(h);
    lo[i] = *reinterpret_cast<uint2*>(l);
  }
}

// GroupNorm + ReLU written directly as the fp16 (h, l) pair of the next conv; |out| is clamped to 60000 (never reached by
// a GroupNorm output with sane affine parameters) and *overflow_flag is raised if the clamp ever fires.
__global__ void __launch_bounds__(256)
gn_relu_apply_f16_kernel(const float4* __restrict__ y, const double* __restrict__ stats, const float* __restrict__ gamma,
                         const float* __restrict__ beta, int HW, int C, int groups, float eps, int relu, long long n4,
                         uint2* __restrict__ out_h, uint2* __restrict__ out_l, int* __restrict__ overflow_flag) {
  const int c4n = C >> 2;
  const int cpg = C / groups;
  const double inv_n = 1.0 / ((double)HW * cpg);
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n4; i += (long long)gridDim.x * 256) {
    const int c = (int)(i % c4n) * 4;
    const long long pix = i / c4n;
    const int b = (int)(pix / HW);
    const int g = c / cpg;
    const double s = stats[((size_t)b * groups + g) * 2], ss = stats[((size_t)b * groups + g) * 2 + 1];
    const double mean = s * inv_n;
    double var = ss * inv_n - mean * mean;
    var = var < 0.0 ? 0.0 : var;
    const float rstd = (float)(1.0 / sqrt(var + (double)eps));
    const float mu = (float)mean;
    const float4 v = __ldcs(y + i);
    const float4 ga = *reinterpret_cast<const float4*>(gamma + c), be = *reinterpret_cast<const float4*>(beta + c);
    float o[4];
    o[0] = fmaf((v.x - mu) * rstd, ga.x, be.x); o[1] = fmaf((v.y - mu) * rstd, ga.y, be.y);
    o[2] = fmaf((v.z - mu) * rstd, ga.z, be.z); o[3] = fmaf((v.w - mu) * rstd, ga.w, be.w);
    __half h[4], l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (relu) o[j] = fmaxf(o[j], 0.f);
      if (fabsf(o[j]) > 60000.f) { o[j] = copysignf(60000.f, o[j]); if (overflow_flag) *overflow_flag = 1; }
      split_h2(o[j], h[j], l[j]);
    }
    out_h[i] = *reinterpret_cast<uint2*>(h);
    out_l[i] = *reinterpret_cast<uint2*>(l);
  }
}

// Fast path of the above for C/8 | 256 and 8 | C/groups: a thread owns 8 channels of one group (mean, rstd, gamma, beta live in
// registers for the whole kernel: no per-element double math or integer division), C/8 threads cover a pixel, blockIdx.y is the
// image and blockIdx.x a contiguous range of pixels; 32-byte loads, 2 x 16-byte stores, two pixels in flight per thread.
__global__ void __launch_bounds__(256)
gn_relu_apply_f16_v8_kernel(const float4* __restrict__ y, const double* __restrict__ stats, const float* __restrict__ gamma,
                            const float* __restrict__ beta, int HW, int C, int groups, float eps, int relu, int pix_per_cta,
                            uint4* __restrict__ out_h, uint4* __restrict__ out_l, int* __restrict__ overflow_flag) {
  const int tpp = C >> 3;                 // threads per pixel
  const int ppp = 256 / tpp;              // pixels per pass
  const int c = (threadIdx.x % tpp) * 8;
  const int b = blockIdx.y;
  const int cpg = C / groups;
  const int g = c / cpg;
  const double inv_n = 1.0 / ((double)HW * cpg);
  const double s = stats[((size_t)b * groups + g) * 2], ss = stats[((size_t)b * groups + g) * 2 + 1];
  const double mean = s * inv_n;
  double var = ss * inv_n - mean * mean;
  var = var < 0.0 ? 0.0 : var;
  const float rstd = (float)(1.0 / sqrt(var + (double)eps));
  const float mu = (float)mean;
  float ga[8], be[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { ga[j] = gamma[c + j]; be[j] = beta[c + j]; }
  const int p0 = blockIdx.x * pix_per_cta;
  const int p1 = min(HW, p0 + pix_per_cta);
  const size_t img = (size_t)b * HW;
  bool clamped = false;
  auto apply = [&](const float4 a, const float4 q, size_t idx8) {
    float o[8] = {a.x, a.y, a.z, a.w, q.x, q.y, q.z, q.w};
    __align__(16) __half h[8], l[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      o[j] = fmaf((o[j] - mu) * rstd, ga[j], be[j]);
      if (relu) o[j] = fmaxf(o[j], 0.f);
      if (fabsf(o[j]) > 60000.f) { o[j] = copysignf(60000.f, o[j]); clamped = true; }
      split_h2(o[j], h[j], l[j]);
    }
    out_h[idx8] = *reinterpret_cast<uint4*>(h);
    out_l[idx8] = *reinterpret_cast<uint4*>(l);
  };
  int p = p0 + threadIdx.x / tpp;
  for (; p + ppp < p1; p += 2 * ppp) {
    const size_t i0 = ((img + p) * C + c) >> 3, i1 = ((img + p + ppp) * C + c) >> 3;
    const float4 a0 = __ldcs(y + 2 * i0), a1 = __ldcs(y + 2 * i0 + 1);
    const float4 b0 = __ldcs(y + 2 * i1), b1 = __ldcs(y + 2 * i1 + 1);
    apply(a0, a1, i0);
    apply(b0, b1, i1);
  }
  for (; p < p1; p += ppp) {
    const size_t i0 = ((img + p) * C + c) >> 3;
    apply(__ldcs(y + 2 * i0), __ldcs(y + 2 * i0 + 1), i0);
  }
  if (clamped && overflow_flag) *overflow_flag = 1;
}

// w [n_out][Cin][taps] (nn.Conv2d / nn.Linear) -> packed [n_mma][tap*Cin + ci] (rows >= n_out are zero) as fp16 h / l
__global__ void pack_conv_weight_f16_kernel(const float* __restrict__ w, int n_out, int n_mma, int Cin, int taps, float scale,
                                            __half* __restrict__ hi, __half* __restrict__ lo) {
  const long long n = (long long)n_mma * Cin * taps;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const int ci = (int)(i % Cin);
    const int tap = (int)((i / Cin) % taps);
    const int co = (int)(i / ((long long)Cin * taps));
    const float v = co < n_out ? w[((size_t)co * Cin + ci) * taps + tap] * scale : 0.f;
    split_h2(v, hi[i], lo[i]);
  }
}

// w [Cout][Cin][3][3] (nn.Conv2d) -> packed [Cout][tap][Cin] split into TF32 hi / lo
__global__ void pack_conv_weight_kernel(const float* __restrict__ w, int Cout, int Cin, float* __restrict__ hi,
                                        float* __restrict__ lo) {
  const long long n = (long long)Cout * Cin * 9;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const int ci = (int)(i % Cin);
    const int tap = (int)((i / Cin) % 9);
    const int co = (int)(i / ((long long)Cin * 9));
    const float v = w[((size_t)co * Cin + ci) * 9 + tap];
    const float h = tf32_hi(v);
    hi[i] = h;
    lo[i] = v - h;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
EncodeTiledFn tc_get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

constexpr int CV_SHAPE_TW[3] = {16, 32, 8}, CV_SHAPE_TH[3] = {8, 4, 16};

static int make_act_map(CUtensorMap* tm, const void* ptr, int B, int H, int W, int C, bool f16, int shape) {
  EncodeTiledFn enc = tc_get_encode();
  if (!enc) return fail("%s", "cuTensorMapEncodeTiled is unavailable (driver too old?)");
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  const cuuint64_t es = f16 ? 2 : 4;
  cuuint64_t strides[3] = {(cuuint64_t)C * es, (cuuint64_t)W * C * es, (cuuint64_t)H * W * C * es};
  cuuint32_t box[4] = {(cuuint32_t)(f16 ? CV_KB_F16 : CV_KB), (cuuint32_t)CV_SHAPE_TW[shape], (cuuint32_t)CV_SHAPE_TH[shape], 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(tm, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled(activation) failed: %s%lld", "", (long long)r);
  return 0;
}
static int make_out_map(CUtensorMap* tm, float* y, int B, int H, int W, int n_out, int ldy, int shape, int h_clip) {
  EncodeTiledFn enc = tc_get_encode();
  if (!enc) return fail("%s", "cuTensorMapEncodeTiled is unavailable (driver too old?)");
  // columns >= n_out and rows >= h_clip (<= H: the right strip stops where the bottom strip begins) are clipped by the TMA unit
  cuuint64_t dims[4] = {(cuuint64_t)n_out, (cuuint64_t)W, (cuuint64_t)h_clip, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)ldy * 4, (cuuint64_t)W * ldy * 4, (cuuint64_t)H * W * ldy * 4};
  cuuint32_t box[4] = {32, (cuuint32_t)CV_SHAPE_TW[shape], (cuuint32_t)CV_SHAPE_TH[shape], 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, y, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled(output) failed: %s%lld", "", (long long)r);
  return 0;
}
static int make_w_map(CUtensorMap* tm, const void* ptr, int n_mma, int Ktot, bool f16, int box_rows) {
  EncodeTiledFn enc = tc_get_encode();
  if (!enc) return fail("%s", "cuTensorMapEncodeTiled is unavailable (driver too old?)");
  cuuint64_t dims[2] = {(cuuint64_t)Ktot, (cuuint64_t)n_mma};
  cuuint64_t strides[1] = {(cuuint64_t)Ktot * (f16 ? 2 : 4)};
  cuuint32_t box[2] = {(cuuint32_t)(f16 ? CV_KB_F16 : CV_KB), (cuuint32_t)box_rows};   // half a weight tile (or tail slice) per TMA request
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(tm, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled(weights) failed: %s%lld", "", (long long)r);
  return 0;
}

}  // namespace ptb

using namespace ptb;

extern "C" int ptb_split_tf32(const float* x, int64_t n, float* hi, float* lo, void* stream) {
  PTB_REQUIRE(n >= 0 && n % 4 == 0, "n must be a multiple of 4");
  PTB_REQUIRE(((uintptr_t)x % 16 == 0) && ((uintptr_t)hi % 16 == 0) && ((uintptr_t)lo % 16 == 0), "16-byte alignment");
  if (n == 0) return 0;
  long long blocks = (n / 4 + 255) / 256;
  const long long cap = (long long)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  split_tf32_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(x), n / 4,
                                                                       reinterpret_cast<float4*>(hi), reinterpret_cast<float4*>(lo));
  return check_launch("ptb_split_tf32");
}

extern "C" int ptb_conv3x3_pack_weight(const float* w_oihw, int Cout, int Cin, float* w_hi, float* w_lo, void* stream) {
  PTB_REQUIRE(Cout > 0 && Cin > 0 && w_oihw && w_hi && w_lo, "shape / NULL");
  const long long n = (long long)Cout * Cin * 9;
  pack_conv_weight_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(w_oihw, Cout, Cin, w_hi, w_lo);
  return check_launch("ptb_conv3x3_pack_weight");
}

template <bool F16>
static int conv_launch(const void* x_hi, const void* x_lo, const void* w_hi, const void* w_lo, int B, int H, int W, int Cin, int taps,
                       int n_out, int n_mma, float* y, int ldy, const float* bias, double* gn_stats, float out_scale,
                       const float* dev_out_scale, void* stream, const char* what) {
  ConvShape cs;
  cs.B = B; cs.H = H; cs.W = W; cs.Cin = Cin;
  {   // tile plan (see ConvShape)
    const int rh = H % 8, rw = W % 16;
    const bool bottom = rh >= 1 && rh <= 4;
    cs.tiles_h = bottom ? H / 8 : (H + 7) / 8;
    cs.bottom_h0 = cs.tiles_h * 8;
    cs.n_bottom = bottom ? (W + 31) / 32 : 0;
    const bool right = rw >= 1 && rw <= 8 && cs.tiles_h > 0;
    cs.tiles_w = right ? W / 16 : (W + 15) / 16;
    cs.right_w0 = cs.tiles_w * 16;
    cs.right_h = cs.tiles_h * 8 < H ? cs.tiles_h * 8 : H;
    cs.n_right = right ? (cs.right_h + 15) / 16 : 0;
    cs.n_main = cs.tiles_h * cs.tiles_w;
    cs.per_img = cs.n_main + cs.n_right + cs.n_bottom;
    cs.n_tiles = B * cs.per_img;
  }
  ConvMaps mp;
  int rc;
  for (int sh = 0; sh < 3; ++sh) {
    if ((rc = make_out_map(&mp.y[sh], y, B, H, W, n_out, ldy, sh, sh == 2 && cs.n_right > 0 ? cs.right_h : H))) return rc;
    if ((rc = make_act_map(&mp.x[sh][0], x_hi, B, H, W, Cin, F16, sh))) return rc;
    if ((rc = make_act_map(&mp.x[sh][1], x_lo, B, H, W, Cin, F16, sh))) return rc;
  }
  for (int kd = 0; kd < 3; ++kd) {     // box rows n_mma/2 (full tile), /4 and /8 (tail slices; only used when n_mma == 256)
    const int rows = (n_mma == CV_N) ? (n_mma / 2) >> kd : n_mma / 2;
    if ((rc = make_w_map(&mp.w[kd][0], w_hi, n_mma, taps * Cin, F16, rows))) return rc;
    if ((rc = make_w_map(&mp.w[kd][1], w_lo, n_mma, taps * Cin, F16, rows))) return rc;
  }
  cs.taps = taps; cs.n_mma = n_mma; cs.n_out = n_out; cs.ldy = ldy;
  // a function attribute is per DEVICE and a process may drive several: set it on every call (a few hundred ns)
  if (cudaFuncSetAttribute(conv_tc_kernel<1, F16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CV_SMEM_BYTES) != cudaSuccess ||
      cudaFuncSetAttribute(conv_tc_kernel<2, F16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CV_SMEM_BYTES) != cudaSuccess ||
      cudaFuncSetAttribute(conv_tc_kernel<3, F16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CV_SMEM_BYTES_PAIR) != cudaSuccess)
    return fail("%s", "cudaFuncSetAttribute(MaxDynamicSharedMemorySize) failed for the conv kernel");
  const int sms = sm_count();
  // PTB_CONV_CLUSTER=2 selects the 2-CTA weight-multicast variant.  Measured on B200 it is exactly as fast as independent
  // CTAs (0.648 vs 0.656 ms per 3xTF32 layer): that kernel is tensor-pipe bound (730 TFLOP/s of TF32 MMA work = what
  // cuDNN's TF32 conv reaches on the same part), not operand-stream bound, so the simpler mode is the default.
  // PTB_CONV_CLUSTER: 1 = independent CTAs, 2 = weight multicast between two cta_group::1 CTAs, 3 = CTA-pair MMA (cta_group::2).
  // Default: 3 for the 256-channel 3x3 convolutions of the towers (the shapes it was validated on), 1 otherwise.
  const char* e_cl = getenv("PTB_CONV_CLUSTER");
  int cluster_mode = (n_mma == CV_N && taps == 9 && F16) ? 3 : 1;
  if (e_cl && e_cl[0] >= '1' && e_cl[0] <= '3') cluster_mode = e_cl[0] - '0';
  if (cluster_mode == 3 && (n_mma % 32 != 0 || !F16)) cluster_mode = 1;
  if (cluster_mode >= 2 && cs.n_tiles >= 2 && sms >= 2) {
    int grid = (sms / 2) * 2;
    const int groups = (cs.n_tiles + 1) / 2;
    if (grid > 2 * groups) grid = 2 * groups;
    const int n_units = grid / 2;
    cs.q_full = groups / n_units; cs.rem = groups % n_units; cs.tail_s = 1;
    const char* e_ts = getenv("PTB_CONV_TAIL_SPLIT");          // "0": no tail split (A-B timing)
    if (cluster_mode == 3 && n_mma == CV_N && cs.rem > 0 && !(e_ts && e_ts[0] == '0')) {
      if (cs.rem * 4 <= n_units) cs.tail_s = 4;
      else if (cs.rem * 2 <= n_units) cs.tail_s = 2;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(cluster_mode == 3 ? CV_THREADS_PAIR : CV_THREADS);
    cfg.dynamicSmemBytes = cluster_mode == 3 ? CV_SMEM_BYTES_PAIR : CV_SMEM_BYTES;
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e = cluster_mode == 3
                        ? cudaLaunchKernelEx(&cfg, conv_tc_kernel<3, F16>, mp, cs, y, gn_stats, out_scale,
                                             dev_out_scale, bias)
                        : cudaLaunchKernelEx(&cfg, conv_tc_kernel<2, F16>, mp, cs, y, gn_stats, out_scale,
                                             dev_out_scale, bias);
    if (e != cudaSuccess) return fail("conv: cluster launch failed: %s", cudaGetErrorString(e));
  } else {
    int grid = sms;
    if (grid > cs.n_tiles) grid = cs.n_tiles;
    cs.q_full = cs.n_tiles / grid; cs.rem = cs.n_tiles % grid; cs.tail_s = 1;
    conv_tc_kernel<1, F16><<<grid, CV_THREADS, CV_SMEM_BYTES, (cudaStream_t)stream>>>(mp, cs, y,
                                                                                             gn_stats, out_scale, dev_out_scale, bias);
  }
  return check_launch(what);
}

extern "C" int ptb_conv3x3_c256_tf32x3(const float* x_hi, const float* x_lo, const float* w_hi, const float* w_lo, int B, int H,
                                       int W, int Cin, float* y, double* gn_stats, void* stream) {
  PTB_REQUIRE(B > 0 && H > 0 && W > 0 && Cin > 0, "shape");
  PTB_REQUIRE(Cin % CV_KB == 0, "Cin must be a multiple of 16");
  PTB_REQUIRE(x_hi && x_lo && w_hi && w_lo && y, "NULL input");
  PTB_REQUIRE(((uintptr_t)x_hi % 16 == 0) && ((uintptr_t)x_lo % 16 == 0) && ((uintptr_t)w_hi % 16 == 0) &&
                  ((uintptr_t)w_lo % 16 == 0) && ((uintptr_t)y % 16 == 0), "16-byte alignment");
  return conv_launch<false>(x_hi, x_lo, w_hi, w_lo, B, H, W, Cin, 9, CV_N, CV_N, y, CV_N, nullptr, gn_stats, 1.f, nullptr, stream,
                            "ptb_conv3x3_c256_tf32x3");
}

extern "C" int ptb_conv3x3_c256_f16x2(const void* x_h, const void* x_l, const void* w_h, const void* w_l, int B, int H, int W, int Cin,
                                      float out_scale, const float* dev_out_scale, float* y, double* gn_stats, void* stream) {
  PTB_REQUIRE(B > 0 && H > 0 && W > 0 && Cin > 0, "shape");
  PTB_REQUIRE(Cin % CV_KB_F16 == 0, "Cin must be a multiple of 32");
  PTB_REQUIRE(x_h && x_l && w_h && w_l && y, "NULL input");
  PTB_REQUIRE(((uintptr_t)x_h % 16 == 0) && ((uintptr_t)x_l % 16 == 0) && ((uintptr_t)w_h % 16 == 0) && ((uintptr_t)w_l % 16 == 0) &&
                  ((uintptr_t)y % 16 == 0), "16-byte alignment");
  return conv_launch<true>(x_h, x_l, w_h, w_l, B, H, W, Cin, 9, CV_N, CV_N, y, CV_N, nullptr, gn_stats, out_scale, dev_out_scale, stream,
                           "ptb_conv3x3_c256_f16x2");
}

extern "C" int ptb_split_f16(const float* x, int64_t n, int auto_scale, void* hi, void* lo, float* dev_inv_scale, void* workspace,
                             void* stream) {
  PTB_REQUIRE(n >= 0 && n % 4 == 0, "n must be a multiple of 4");
  PTB_REQUIRE(((uintptr_t)x % 16 == 0) && ((uintptr_t)hi % 8 == 0) && ((uintptr_t)lo % 8 == 0), "alignment");
  PTB_REQUIRE(!auto_scale || (workspace && dev_inv_scale), "auto_scale needs a 4-byte workspace and dev_inv_scale");
  if (n == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  long long blocks = (n / 4 + 255) / 256;
  const long long cap = (long long)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  unsigned int* amax = nullptr;
  if (auto_scale) {
    amax = reinterpret_cast<unsigned int*>(workspace);
    if (cudaMemsetAsync(amax, 0, 4, st) != cudaSuccess) return fail("%s", "ptb_split_f16: cudaMemsetAsync failed");
    amax_abs_kernel<<<(unsigned)blocks, 256, 0, st>>>(reinterpret_cast<const float4*>(x), n / 4, amax);
    int rc = check_launch("ptb_split_f16/amax");
    if (rc) return rc;
  }
  split_f16_kernel<<<(unsigned)blocks, 256, 0, st>>>(reinterpret_cast<const float4*>(x), n / 4, amax, reinterpret_cast<uint2*>(hi),
                                                    reinterpret_cast<uint2*>(lo), dev_inv_scale);
  return check_launch("ptb_split_f16");
}

extern "C" int ptb_amax_abs(const float* x, int64_t n, unsigned int* dev_amax_bits, int accumulate, void* stream) {
  PTB_REQUIRE(n >= 0 && n % 4 == 0, "n must be a multiple of 4");
  PTB_REQUIRE(((uintptr_t)x % 16 == 0) && dev_amax_bits, "alignment / NULL");
  cudaStream_t st = (cudaStream_t)stream;
  if (!accumulate && cudaMemsetAsync(dev_amax_bits, 0, 4, st) != cudaSuccess) return fail("%s", "ptb_amax_abs: cudaMemsetAsync failed");
  if (n == 0) return 0;
  long long blocks = (n / 4 + 255) / 256;
  const long long cap = (long long)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  amax_abs_kernel<<<(unsigned)blocks, 256, 0, st>>>(reinterpret_cast<const float4*>(x), n / 4, dev_amax_bits);
  return check_launch("ptb_amax_abs");
}

extern "C" int ptb_split_f16_amax(const float* x, int64_t n, const unsigned int* dev_amax_bits, void* hi, void* lo,
                                  float* dev_inv_scale, void* stream) {
  PTB_REQUIRE(n >= 0 && n % 4 == 0, "n must be a multiple of 4");
  PTB_REQUIRE(((uintptr_t)x % 16 == 0) && ((uintptr_t)hi % 8 == 0) && ((uintptr_t)lo % 8 == 0), "alignment");
  PTB_REQUIRE(dev_amax_bits && dev_inv_scale, "dev_amax_bits and dev_inv_scale are required");
  if (n == 0) return 0;
  long long blocks = (n / 4 + 255) / 256;
  const long long cap = (long long)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  split_f16_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(x), n / 4, dev_amax_bits,
                                                                      reinterpret_cast<uint2*>(hi), reinterpret_cast<uint2*>(lo),
                                                                      dev_inv_scale);
  return check_launch("ptb_split_f16_amax");
}

extern "C" int ptb_conv3x3_pack_weight_f16(const float* w_oihw, int Cout, int Cin, float scale, void* w_h, void* w_l, void* stream) {
  PTB_REQUIRE(Cout > 0 && Cin > 0 && w_oihw && w_h && w_l && scale > 0.f, "shape / NULL");
  const long long n = (long long)Cout * Cin * 9;
  pack_conv_weight_f16_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(w_oihw, Cout, Cout, Cin, 9, scale,
                                                                                           reinterpret_cast<__half*>(w_h),
                                                                                           reinterpret_cast<__half*>(w_l));
  return check_launch("ptb_conv3x3_pack_weight_f16");
}

extern "C" int ptb_conv_tc_pack_weight_f16(const float* w, int n_out, int n_mma, int Cin, int taps, float scale, void* w_h, void* w_l,
                                           void* stream) {
  PTB_REQUIRE(n_out > 0 && Cin > 0 && (taps == 1 || taps == 9) && w && w_h && w_l && scale > 0.f, "shape / NULL");
  PTB_REQUIRE(n_mma >= n_out && n_mma % 16 == 0 && n_mma <= CV_N, "n_mma must be a multiple of 16 in [n_out, 256]");
  const long long n = (long long)n_mma * Cin * taps;
  pack_conv_weight_f16_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(w, n_out, n_mma, Cin, taps, scale,
                                                                                           reinterpret_cast<__half*>(w_h),
                                                                                           reinterpret_cast<__half*>(w_l));
  return check_launch("ptb_conv_tc_pack_weight_f16");
}

extern "C" int ptb_conv_tc_f16x2(const void* x_h, const void* x_l, const void* w_h, const void* w_l, int B, int H, int W, int Cin,
                                 int taps, int n_out, int n_mma, float out_scale, const float* dev_out_scale, const float* bias,
                                 float* y, int ldy, void* stream) {
  PTB_REQUIRE(B > 0 && H > 0 && W > 0 && Cin > 0 && (taps == 1 || taps == 9), "shape");
  PTB_REQUIRE(Cin % CV_KB_F16 == 0, "Cin must be a multiple of 32");
  PTB_REQUIRE(n_out > 0 && n_mma >= n_out && n_mma % 16 == 0 && n_mma <= CV_N, "n_mma must be a multiple of 16 in [n_out, 256]");
  PTB_REQUIRE(ldy >= n_out && ldy % 4 == 0, "ldy must be a multiple of 4 and >= n_out");
  PTB_REQUIRE(x_h && x_l && w_h && w_l && y, "NULL input");
  PTB_REQUIRE(((uintptr_t)x_h % 16 == 0) && ((uintptr_t)x_l % 16 == 0) && ((uintptr_t)w_h % 16 == 0) && ((uintptr_t)w_l % 16 == 0) &&
                  ((uintptr_t)y % 16 == 0), "16-byte alignment");
  return conv_launch<true>(x_h, x_l, w_h, w_l, B, H, W, Cin, taps, n_out, n_mma, y, ldy, bias, nullptr, out_scale, dev_out_scale, stream,
                           "ptb_conv_tc_f16x2");
}

extern "C" int ptb_gn_relu_apply_f16(const float* y, const double* gn_stats, const float* gamma, const float* beta, int B, int HW,
                                     int C, int groups, float eps, int relu, void* out_h, void* out_l, int* overflow_flag,
                                     void* stream) {
  PTB_REQUIRE(B > 0 && HW > 0 && C > 0 && groups > 0 && C % groups == 0, "shape");
  PTB_REQUIRE((C / groups) % 4 == 0 && C % 4 == 0, "channels per group must be a multiple of 4");
  PTB_REQUIRE(y && gn_stats && gamma && beta && out_h && out_l, "NULL input");
  const int cpg = C / groups;
  if (C % 8 == 0 && cpg % 8 == 0 && C <= 2048 && 256 % (C / 8) == 0 && ((uintptr_t)y % 32 == 0) && ((uintptr_t)out_h % 16 == 0) &&
      ((uintptr_t)out_l % 16 == 0)) {
    const int ppp2 = 2 * (256 / (C / 8));                         // pixels per CTA and double-pass
    int chunks = (sm_count() * 4 + B - 1) / B;                   // one wave of 4 CTAs (64 regs x 256 thr) per SM over all images
    int pix_per_cta = (HW + chunks - 1) / chunks;
    pix_per_cta = ((pix_per_cta + ppp2 - 1) / ppp2) * ppp2;
    chunks = (HW + pix_per_cta - 1) / pix_per_cta;
    gn_relu_apply_f16_v8_kernel<<<dim3((unsigned)chunks, (unsigned)B), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float4*>(y), gn_stats, gamma, beta, HW, C, groups, eps, relu, pix_per_cta,
        reinterpret_cast<uint4*>(out_h), reinterpret_cast<uint4*>(out_l), overflow_flag);
    return check_launch("ptb_gn_relu_apply_f16");
  }
  const long long n4 = (long long)B * HW * C / 4;
  long long blocks = (n4 + 255) / 256;
  const long long cap = (long long)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  gn_relu_apply_f16_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(y), gn_stats, gamma, beta,
                                                                              HW, C, groups, eps, relu, n4,
                                                                              reinterpret_cast<uint2*>(out_h),
                                                                              reinterpret_cast<uint2*>(out_l), overflow_flag);
  return check_launch("ptb_gn_relu_apply_f16");
}

extern "C" int ptb_gn_relu_apply(const float* y, const double* gn_stats, const float* gamma, const float* beta, int B, int HW,
                                 int C, int groups, float eps, int relu, float* out_hi, float* out_lo, void* stream) {
  PTB_REQUIRE(B > 0 && HW > 0 && C > 0 && groups > 0 && C % groups == 0, "shape");
  PTB_REQUIRE((C / groups) % 4 == 0 && C % 4 == 0, "channels per group must be a multiple of 4");
  PTB_REQUIRE(y && gn_stats && gamma && beta && out_hi, "NULL input");
  const long long n4 = (long long)B * HW * C / 4;
  long long blocks = (n4 + 255) / 256;
  const long long cap = (long long)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  gn_relu_apply_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(y), gn_stats, gamma, beta,
                                                                          HW, C, groups, eps, relu, n4,
                                                                          reinterpret_cast<float4*>(out_hi),
                                                                          reinterpret_cast<float4*>(out_lo));
  return check_launch("ptb_gn_relu_apply");
}
