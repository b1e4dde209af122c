// Tensor-core (tcgen05) ConvTranspose3d k=3, stride 2, padding 1, output_padding 1: the up-sampling convs of the hourglasses
//   conv5 128->64 / 64->64 (1/16 -> 1/8 res) and conv6 64->32 (1/8 -> 1/4 res): gwcnet/hourglass.py:35-41,
//   psmnet/psmnet_cost_processor.py:99-106 (deconv3d_bn).
// Per dimension an output index o gathers  o even (=2m): tap k=1 from input m;  o odd (=2m+1): k=0 from m+1 and k=2 from m.
// Same machinery as conv3d_tcg.cu / conv3d_tcs2.cu (3xFP16 split, LDG-staged swizzled operands, warp-specialised
// persistent CTA).  An accumulator tile holds the output rows of ONE parity class: plane od, rows oh = 2j + ph for
// R = 128/Win consecutive j, all 2*Win output columns.  For each valid tap pair (kd, kh) the operand tile is the R input
// rows j (+1 for k=0) of input plane id, un-shifted in w, and one MMA with the kw slices stacked along N gives
//   E[m] = A[m].W1 -> output column 2m,      P2[m] = A[m].W2 and P0[m] = A[m].W0 -> output column 2m+1 = P2[m] + P0[m+1];
// the epilogue does that single right shift (zero at m = Win-1: the column beyond the input) and writes both columns.
// Tap pairs per tile: 1, 2, 2 or 4 depending on (od&1, ph); work items interleave the classes so every CTA gets a mix.
// GENERAL WIDTHS (GW = true, W = 128 instantiations; see conv3d_tcg.cu): an M tile is a 128-column segment of one INPUT row of
// runtime width Wr starting at input column ct * 127; tile column 127 is the halo that provides P0[m+1] (zero beyond the image) and
// its two output columns are not stored.
// KS = 4: ConvTranspose3d(k=4, s=2, p=1) of StereoBase's hourglass (stereobase/hourglass.py:35-60 conv*_up): per dimension
//   o = 2m: taps k=1 (input m) and k=3 (input m-1);   o = 2m+1: taps k=2 (input m) and k=0 (input m+1)
// -- every parity class has 2 x 2 (kd, kh) tap pairs, the four kw slices are stacked along N as [W1 | W3 | W2 | W0] and the
// epilogue forms  even[m] = P1[m] + P3[m-1],  odd[m] = P2[m] + P0[m+1]  (one left and one right shift).
#include <cstdlib>

#include "tc_common.cuh"

namespace osb {

struct TcdcParams {
  const float* x;          // (B, D, H, W, Cin) channels-last (fp16 in the H16 instantiations)
  const void* w;           // fp16 [3 kd][Cin/KC][3 kh][3*Cout][KC hi | KC lo]  (ops.pack_tc_weight)
  const float* scale;
  const float* shift;
  const float* residual;
  float* y;                // fp16 in the H16 instantiations
  int B, D, H, Cin;        // INPUT extent D x H x W; output is 2D x 2H x 2W
  int act;
  float kappa;       // expected round-towards-zero loss per accumulating MMA (tc_common.cuh)
  unsigned int* overflow;  // sticky fp16-range flag (tc_common.cuh)
  int out_ndhwc, res_ndhwc;
  int items, hblocks;
  int Wr, ctiles;          // general-width instantiations: INPUT width and column tiles per row (whole-row kernels: W, 1)
  int ystride;             // channels per voxel of the channels-last y / residual (0 = COUT); > COUT: this launch writes a channel slice
  int cout_real;           // channels of an NCDHW output / residual (<= COUT: zero-padded channel plans write only the real ones)
};

template <int COUT, int KC, int W, int TILES, bool GW = false, int KS_ = 3>     // W = INPUT width, KS_ = kernel size (3 or 4)
struct TcdcCfg {
  static_assert(!GW || W == 128, "general-width tiles are 128-column segments of one input row");
  static_assert(KS_ == 3 || (KS_ == 4 && !GW), "kernel size 3 (any width) or 4 (whole-row tiles)");
  static constexpr int KS = KS_;
  static constexpr int HALO = GW ? 1 : 0;                   // halo columns on the RIGHT of a column tile
  static constexpr int CSTEP = 128 - HALO;                  // input columns a column tile produces outputs for
  static constexpr int R = 128 / W;                         // input rows (= output rows of one parity) per M tile
  static constexpr int ROWB = KC * 4;                       // bytes per K-major operand row: [KC fp16 hi | KC fp16 lo]
  static constexpr int UNIT_BYTES = 128 * ROWB;
  static constexpr int N3 = KS_ * COUT;                     // kw slices stacked along N
  static constexpr int B_SLICE = N3 * ROWB;                 // one kh weight slice (hi and lo halves of every row)
  // A-unit ring.  NLW loader warps (1-4 and 10) fill the units round-robin (unit u belongs to warp u mod NLW) into a ring as deep as
  // shared memory allows (at most 10 units).  Each loader warp enumerates ONLY ITS OWN units: when every warp walked the whole
  // (tile, tap) sequence and picked every NLW-th unit, that scalar control flow was the bound of these kernels -- a conv6 run with
  // loads, conversions, MMAs and stores all disabled still took 0.37 of 0.69 ms, two thirds of the loader warps' stall samples on
  // the loop lines (profiles/r2_conv6_barrier_skeleton_stalls.txt).
  static constexpr int NLW = 5;
  static constexpr int FIXED_SMEM = 1024 + TC_BSLOTS * KS_ * B_SLICE + 1024 + 2 * 4 * 2 * 32 * 4 + 3 * COUT * 4 + TP_BYTES;
  static constexpr int STAGES = (232448 - FIXED_SMEM) / UNIT_BYTES < 10 ? (232448 - FIXED_SMEM) / UNIT_BYTES : 10;
  static_assert(STAGES >= NLW, "the ring must hold at least one unit per loader warp");
  static constexpr int HBLK = TILES * R;                    // output rows per work item
  static constexpr int KSTEPS = KC / 16;                    // K = 16 fp16 channels per MMA
  static constexpr int LO = KC / 8;                         // descriptor offset (16-byte units) of the lo half of a row
  static constexpr int A_OFF = 0;
  static constexpr int B_OFF = A_OFF + STAGES * UNIT_BYTES;
  static constexpr int BAR_OFF = B_OFF + TC_BSLOTS * KS_ * B_SLICE;
  static constexpr int THREADS = 32 + 128 + 128 + 64;       // MMA | A loaders | epilogue | weight loaders (11 warps)
  static constexpr size_t SMEM = 1024 + (size_t)BAR_OFF + 1024 + 2 * 4 * 2 * 32 * 4 + 3 * COUT * 4 + TP_BYTES;
  static_assert(SMEM <= 232448, "shared memory budget of one CTA exceeded");
  static_assert(TILES * N3 <= 512, "accumulators exceed TMEM");
  static_assert(B_SLICE % 1024 == 0 && UNIT_BYTES % 1024 == 0, "operand tiles must stay 1024-byte aligned");
  static_assert(N3 % 16 == 0 && N3 <= 256, "invalid UMMA N");
};

// work item = (image b, output plane od, row parity ph, block of TILES*R input rows); parity bits vary fastest so that the
// 1/2/2/4-tap classes are interleaved over the persistent CTAs
struct ItemDc {
  int b, od, ph, j0, last_kd, last_kh, ct, nkd;
};
// output index o gathers tap k from input (o + 1 - k) / 2 when that is an integer inside [0, n)
__device__ __forceinline__ bool kd_valid(int od, int kd, int D) {
  const int num = od + 1 - kd;
  return !(num & 1) && num >= 0 && (num >> 1) < D;
}
// rows outside the image are staged as zeros rather than skipped, so only the parity decides
__device__ __forceinline__ bool kh_valid(int ph, int kh) { return ((ph + 1 - kh) & 1) == 0; }
template <class C>
__device__ __forceinline__ ItemDc decode_dc(const TcdcParams& p, int it) {
  ItemDc w;
  w.ct = 0;
  if (C::HALO) {                                    // general widths: the column tile varies fastest
    w.ct = it % p.ctiles;
    it /= p.ctiles;
  }
  w.ph = it & 1;
  it >>= 1;
  const int Do = 2 * p.D;
  w.od = it % Do;
  it /= Do;
  w.j0 = (it % p.hblocks) * C::HBLK;
  w.b = it / p.hblocks;
  w.last_kd = w.last_kh = -1, w.nkd = 0;
#pragma unroll
  for (int k = 0; k < C::KS; ++k) {                 // last valid taps in issue order; number of input planes feeding this class
    if (kd_valid(w.od, k, p.D)) w.last_kd = k, ++w.nkd;
    if (kh_valid(w.ph, k)) w.last_kh = k;
  }
  return w;
}

// H16: fp16 activations in and out, one hi x hi MMA per k-step (see conv3d_tcg.cu)
template <int COUT, int KC, int W, int TILES, bool GW = false, int KS = 3, bool H16 = false>
__global__ void __launch_bounds__(TcdcCfg<COUT, KC, W, TILES, GW, KS>::THREADS, 1) conv3d_tcdc_kernel(const TcdcParams p) {
  using C = TcdcCfg<COUT, KC, W, TILES, GW, KS>;
  using A = TcAct<H16>;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* a_buf = smem + C::A_OFF;
  uint8_t* b_buf = smem + C::B_OFF;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::BAR_OFF);
  uint64_t* a_ready = bars;                         // [STAGES] loaders -> MMA        (32 arrivals: one warp)
  uint64_t* a_empty = a_ready + C::STAGES;          // [STAGES] MMA -> loaders        (tcgen05.commit)
  uint64_t* b_full = a_empty + C::STAGES;           // [2][KS]  weight producer -> MMA (expect_tx + TMA bytes)
  uint64_t* b_empty = b_full + TC_BSLOTS * KS;      // [2][KS]  MMA -> weight producer (tcgen05.commit)
  uint64_t* acc_full = b_empty + TC_BSLOTS * KS;                // [TILES]
  uint64_t* acc_empty = acc_full + TILES;           // [TILES]  (128 arrivals)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + TILES);
  float* xchg = reinterpret_cast<float*>(smem + C::BAR_OFF + 1024);   // [2][4 quadrants][2 sides][32]
  float* s_scale = xchg + 2 * 4 * 2 * 32;
  float* s_shift = s_scale + COUT;
  float* zeros = s_shift + COUT;
  float* tpose = zeros + COUT;                      // [4 warps][32][TP_STRIDE] transpose tiles of the epilogue

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nchunk = p.Cin / KC;
  const int Wp = GW ? p.Wr : W;                     // INPUT width (the output is 2 * Wp wide)
  const int YS = (W < 32 && p.ystride) ? p.ystride : COUT;   // (compile-time COUT in the wide instantiations: slices exist at W' = 16 only)      // channel stride of the channels-last output / residual

  if (threadIdx.x == 0) {
    for (int s = 0; s < C::STAGES; ++s) {
      mbar_init(&a_ready[s], 32);                     // one loader warp fills a unit
      mbar_init(&a_empty[s], 1);
    }
    for (int k = 0; k < TC_BSLOTS * KS; ++k) {
      mbar_init(&b_full[k], 1);
      mbar_init(&b_empty[k], 1);
    }
    for (int t = 0; t < TILES; ++t) {
      mbar_init(&acc_full[t], 1);
      mbar_init(&acc_empty[t], 128);
    }
    fence_mbar_init();
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  for (int c = threadIdx.x; c < COUT; c += blockDim.x) {
    s_scale[c] = p.scale ? p.scale[c] : 1.f;
    s_shift[c] = p.shift ? p.shift[c] : 0.f;
    zeros[c] = 0.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  // ---------------------------------------------------------------------------------------------- MMA issuer
  if (warp == 0) {
    const uint32_t idesc = idesc_f16(128, C::N3);
    const uint64_t dbase = (KC == 32) ? desc_sw128_base() : desc_sw64_base();
    const uint32_t b16 = (smem_u32(b_buf) & 0x3FFFF) >> 4;
    uint32_t unitc = 0, itc = 0;
    uint32_t bph[KS] = {};                            // per-slice use counters (slices are loaded only for valid kh)
    for (int it = blockIdx.x; it < p.items; it += gridDim.x, ++itc) {
      const ItemDc w = decode_dc<C>(p, it);
      const int ntiles = min(TILES, (p.H - w.j0 + C::R - 1) / C::R);
      uint32_t started = 0;
      for (int kd = 0; kd < KS; ++kd) {
        if (!kd_valid(w.od, kd, p.D)) continue;
        for (int ch = 0; ch < nchunk; ++ch) {
          const bool last_phase = (kd == w.last_kd) && (ch == nchunk - 1);
#pragma unroll
          for (int t = 0; t < TILES; ++t) {
#pragma unroll
            for (int kh = 0; kh < KS; ++kh) {
              if (!kh_valid(w.ph, kh)) continue;        // warp-uniform
              const uint32_t slot = unitc % C::STAGES, ph = (unitc / C::STAGES) & 1;
              mbar_wait(&a_ready[slot], ph);
              const uint32_t bslot = (bph[kh] & 1) * KS + kh;  // the buffers of tap kh alternate between its uses
              if (t == 0) mbar_wait(&b_full[bslot], (bph[kh] >> 1) & 1);   // first use of slice kh in this phase
              tc_fence_after();
              const uint32_t accum = (started >> t) & 1;
              if (!accum) {                             // hand-shake taken for unused tiles too (parity must not alias)
                mbar_wait(&acc_empty[t], (itc & 1) ^ 1);
                tc_fence_after();
                started |= 1u << t;
              }
              if (t < ntiles) {
                if (elect_one()) {
                  const uint64_t da0 = dbase | (uint64_t)((smem_u32(a_buf + slot * C::UNIT_BYTES) & 0x3FFFF) >> 4);
                  const uint32_t acc = tmem + t * C::N3;
                  const uint64_t db0 = dbase | (uint64_t)(b16 + (bslot * C::B_SLICE) / 16);
#pragma unroll
                  for (int ks = 0; ks < C::KSTEPS; ++ks) {
                    if constexpr (H16) {
                      mma_f16(acc, da0 + 2 * ks, db0 + 2 * ks, idesc, ks > 0 ? 1u : accum);
                    } else {
                      mma_f16(acc, da0 + C::LO + 2 * ks, db0 + 2 * ks, idesc, ks > 0 ? 1u : accum);   // small terms first
                      mma_f16(acc, da0 + 2 * ks, db0 + C::LO + 2 * ks, idesc, 1);
                      mma_f16(acc, da0 + 2 * ks, db0 + 2 * ks, idesc, 1);
                    }
                  }
                }
                __syncwarp();
              }
              if (elect_one()) {
                mma_commit(&a_empty[slot]);
                if (t == TILES - 1) mma_commit(&b_empty[bslot]);                 // last user of slice kh in this phase
                if (last_phase && kh == w.last_kh) mma_commit(&acc_full[t]);     // tile t has received its last tap
              }
              __syncwarp();
              if (t == TILES - 1) ++bph[kh];
              ++unitc;
            }
          }
        }
      }
    }
  }
  // ---------------------------------------------------------------------------------------------- A-unit loaders
  // One loader WARP per unit, units round-robin over the NLW loader warps (unit u -> warp u % NLW, ring slot u % STAGES), so NLW
  // units' global loads are in flight per SM; a slot is refilled in unit order (the a_empty wait of use n cannot be overtaken: use
  // n + 1 of that slot belongs to a warp that has not filled it yet, so no mbarrier phase is skipped).  ncu
  // (profiles/r1_ncu_summary.md, r1_tcdc_conv6): with all four warps on one unit at a time the loaders sat on the load latency and
  // the tensor pipe was 17 % busy.  Each warp enumerates ONLY its own units (see the Cfg note): one runtime loop, one copy of the
  // body (unrolled bodies took the kernel to 254 KB of code).
  else if (warp < 5 || warp == 10) {
    const int lw = warp < 5 ? warp - 1 : 4;
    static_assert(KC == 16, "lane_voxel / unit-row mapping below is written for 64-byte operand rows");
    constexpr int CPR = KC / 4;                      // fp32 16-byte chunks per voxel of the K chunk
    constexpr int VPL = 32 / CPR;                    // voxels covered by one warp-wide LDG.128
    constexpr int NLD = 128 / VPL;                   // loads per lane per unit
    static_assert(W % VPL == 0, "a load instruction must not straddle image rows");
    const int v0 = lane_voxel<KC>(lane), c = lane % CPR;   // permuted voxel order: conflict-free STS.64 (tc_common.cuh)
    float amax = 0.f;
    uint32_t ubase = 0;                              // global index of the current phase's first unit
    int first = lw;                                  // this warp's first local unit index in the current phase: (ubase + first) % NLW == lw
    auto fill = [&](const typename A::T* base, size_t rstride, size_t cstride, int h_first, int h_step, uint32_t u, int col0) {
      // base: this lane's address for load 0; load j covers operand rows VPL*j .. VPL*j + VPL - 1 = columns (VPL*j) % W ..
      // of tile row (VPL*j) / W, read from image row h_first + h_step * tile row (rstride / cstride floats per tile row / column).
      // General widths: col0 = INPUT column of load 0 (columns >= Wp are zero: beyond the image).
      typename A::V v[NLD];
#pragma unroll
      for (int j = 0; j < NLD; ++j) {
        const int hin = h_first + h_step * ((VPL * j) / W);
        const size_t off = (size_t)((VPL * j) / W) * rstride + (size_t)((VPL * j) % W) * cstride;
        bool ok = hin >= 0 && hin < p.H;
        if (GW) ok = ok && (unsigned)(col0 + VPL * j) < (unsigned)Wp;
        if constexpr (H16) v[j] = ok ? __ldg(reinterpret_cast<const uint2*>(base + (ptrdiff_t)off)) : make_uint2(0u, 0u);
        else v[j] = ok ? __ldg(reinterpret_cast<const float4*>(base + (ptrdiff_t)off)) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      const uint32_t slot = u % C::STAGES, ph = (u / C::STAGES) & 1;   // u = global unit index
      mbar_wait_relaxed(&a_empty[slot], ph ^ 1);
      uint8_t* tile = a_buf + slot * C::UNIT_BYTES;
#pragma unroll
      for (int j = 0; j < NLD; ++j) {
        if constexpr (H16) stage_f16_hi<KC>(tile, v0 + VPL * j, c, v[j]);
        else stage_f16_split<KC>(tile, v0 + VPL * j, c, v[j], amax);
      }
      fence_proxy_async();
      mbar_arrive(&a_ready[slot]);
    };
    for (int it = blockIdx.x; it < p.items; it += gridDim.x) {
      const ItemDc w = decode_dc<C>(p, it);
      for (int kd = 0; kd < KS; ++kd) {
        if (!kd_valid(w.od, kd, p.D)) continue;
        const int id = (w.od + 1 - kd) >> 1;         // input plane feeding output plane od through tap kd
        const typename A::T* plane = reinterpret_cast<const typename A::T*>(p.x) + ((size_t)w.b * p.D + id) * p.H * (size_t)Wp * p.Cin;
        const int col0 = w.ct * C::CSTEP + v0;       // INPUT column of this lane's first load (whole-row kernels: v0)
        // valid kh taps of this row parity in issue order: k3: ph 0 -> {1}, ph 1 -> {0, 2};  k4: ph 0 -> {1, 3}, ph 1 -> {0, 2}
        const int nkh = (KS == 4 || w.ph) ? 2 : 1, kh0 = w.ph ? 0 : 1;
        const int upp = TILES * nkh;                 // units per (kd, chunk) phase, local index = t * nkh + tap index
        for (int ch = 0; ch < nchunk; ++ch) {
#pragma unroll 1
          for (int j = first; j < upp; j += C::NLW) {
            const int t = nkh == 2 ? (j >> 1) : j, kh = kh0 + 2 * (nkh == 2 ? (j & 1) : 0);
            // operand row v = input voxel (row j0 + t*R + v / W + (ph + 1 - kh) / 2, column v % W): output row 2j + ph gathers
            // tap kh from input row j + (ph + 1 - kh) / 2  (k3: +1 for kh = 0; k4: +1 for kh = 0, -1 for kh = 3)
            const int h_first = w.j0 + t * C::R + ((w.ph + 1 - kh) >> 1);
            const typename A::T* base = plane + ((ptrdiff_t)h_first * Wp + col0) * p.Cin + ch * KC + c * 4;
            fill(base, (size_t)Wp * p.Cin, (size_t)p.Cin, h_first, 1, ubase + j, col0);
          }
          ubase += upp;
          first = (first + C::NLW - upp % C::NLW) % C::NLW;
        }
      }
    }
    tc_report_overflow(p.overflow, amax);
  }
  // ---------------------------------------------------------------------------------------------- epilogue
  else if (warp < 9) {
    const int q = warp & 3;                          // TMEM lane quadrant this warp may read
    const int m = q * 32 + lane;                     // operand row owned by this thread
    const int rr = m / W, wcol = m % W;              // input row inside the tile, input column
    const bool has_right_q = (((q + 1) * 32) % W) != 0;   // the next quadrant continues the same image row
    const bool has_left_q = ((q * 32) % W) != 0;          // (k4 only) the previous quadrant does
    const int Do = 2 * p.D, Ho = 2 * p.H;
    const int Wo = 2 * Wp;
    uint32_t itc = 0, exc = 0;
    float yamax = 0.f;                               // H16: largest stored magnitude (fp16 saturation at 65504)
    for (int it = blockIdx.x; it < p.items; it += gridDim.x, ++itc) {
      const ItemDc w = decode_dc<C>(p, it);
      const int ntiles = min(TILES, (p.H - w.j0 + C::R - 1) / C::R);
      // tap pairs of this parity class: (1 or 2 kd) x (1 or 2 kh); each adds chunks x k-steps x 3 MMAs (tc_common.cuh: rz_kappa)
      const float corr = 1.f + p.kappa * (float)(w.nkd * (KS == 4 ? 2 : w.ph + 1) * nchunk * C::KSTEPS * A::TERMS);
      // general widths: input column of this thread's tile column; the halo column and columns beyond the image are not stored
      const int col = GW ? w.ct * C::CSTEP + m : wcol;
      const bool cvalid = !GW || (m < C::CSTEP && col < Wp);
      const uint32_t vmask = GW ? __ballot_sync(0xffffffffu, cvalid) : 0xffffffffu;
      for (int t = 0; t < ntiles; ++t) {
        const int j = w.j0 + t * C::R + rr;
        const bool live = j < p.H;
        const int oh = 2 * j + w.ph;
        const size_t vox = (((size_t)w.b * Do + w.od) * Ho + oh) * Wo + 2 * col;       // NDHWC index of the EVEN output voxel
        if (live && cvalid && p.residual && p.res_ndhwc) {
          // the residual streams from HBM: start pulling this thread's two voxels (2*COUT floats, contiguous) into L2 while
          // the tile is still being accumulated, so the loads after the transpose do not expose the DRAM latency per tile
          const float* rp = p.residual + vox * YS;
#pragma unroll
          for (int k = 0; k < 2 * COUT; k += 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(rp + k));
        }
        mbar_wait_relaxed(&acc_full[t], itc & 1);
        tc_fence_after();
        const size_t plane = (size_t)Do * Ho * Wo;                                   // NCDHW channel stride
        const size_t ncdhw0 = (size_t)w.b * p.cout_real * plane + ((size_t)w.od * Ho + oh) * Wo + 2 * col;
        const uint32_t trow = tmem + ((uint32_t)(q * 32) << 16) + t * C::N3;
#pragma unroll 1
        for (int cg = 0; cg < COUT; cg += 32) {
          float ev[32], od_[32];
          float* xb = xchg + (exc & 1) * (4 * 2 * 32);
          ++exc;
          if constexpr (KS == 3) {
          // accumulator column groups: raw[0] = E (kw=1), raw[1] = P2 (kw=2), raw[2] = P0 (kw=0)
          uint32_t raw[3][32];
#pragma unroll
          for (int kw = 0; kw < 3; ++kw)
#pragma unroll
            for (int c0 = 0; c0 < 32; c0 += 16) tmem_ld16_nowait(trow + kw * COUT + cg + c0, &raw[kw][c0]);
          tmem_ld_wait();
          if (cg + 32 >= COUT) {                      // whole tile in registers: hand it back to the MMA warp
            tc_fence_before();
            mbar_arrive(&acc_empty[t]);
          }
          if (lane == 0) {
#pragma unroll
            for (int i = 0; i < 32; ++i) xb[(q * 2) * 32 + i] = __uint_as_float(raw[2][i]);
          }
          named_bar_sync(1, 128);
          const float* xr = has_right_q ? xb + ((q + 1) * 2) * 32 : zeros;
#pragma unroll
          for (int i0 = 0; i0 < 32; i0 += 4) {        // neighbour values loaded unconditionally, merged with selects (no branches)
            const float4 r4 = *reinterpret_cast<const float4*>(xr + i0);
            const float re[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int i = i0 + k;
              float right = __shfl_down_sync(0xffffffffu, __uint_as_float(raw[2][i]), 1);   // P0 of input column m+1
              right = (lane == 31) ? re[k] : right;                                        // zero beyond the last input column
              if (W < 32) right = (wcol == W - 1) ? 0.f : right;                           // row seams inside the warp
              ev[i] = __uint_as_float(raw[0][i]) * corr;
              od_[i] = (__uint_as_float(raw[1][i]) + right) * corr;
            }
          }
          } else {
          // k4: accumulator column groups [P1 | P3 | P2 | P0].  The two shifted groups first (their raw values die in the shuffles),
          // then the two aligned ones: at most 128 accumulator values are live at a time.
          uint32_t ra[32], rb[32];
#pragma unroll
          for (int c0 = 0; c0 < 32; c0 += 16) {
            tmem_ld16_nowait(trow + 1 * COUT + cg + c0, &ra[c0]);       // P3
            tmem_ld16_nowait(trow + 3 * COUT + cg + c0, &rb[c0]);       // P0
          }
          tmem_ld_wait();
          if (lane == 31) {
#pragma unroll
            for (int i = 0; i < 32; ++i) xb[(q * 2 + 1) * 32 + i] = __uint_as_float(ra[i]);   // P3 of this quadrant's last column
          }
          if (lane == 0) {
#pragma unroll
            for (int i = 0; i < 32; ++i) xb[(q * 2) * 32 + i] = __uint_as_float(rb[i]);       // P0 of this quadrant's first column
          }
          named_bar_sync(1, 128);
          const float* xl = has_left_q ? xb + ((q - 1) * 2 + 1) * 32 : zeros;
          const float* xr = has_right_q ? xb + ((q + 1) * 2) * 32 : zeros;
#pragma unroll
          for (int i0 = 0; i0 < 32; i0 += 4) {
            const float4 l4 = *reinterpret_cast<const float4*>(xl + i0);
            const float4 r4 = *reinterpret_cast<const float4*>(xr + i0);
            const float le[4] = {l4.x, l4.y, l4.z, l4.w}, re[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int i = i0 + k;
              const float left = __shfl_up_sync(0xffffffffu, __uint_as_float(ra[i]), 1);      // P3 of input column m-1
              const float right = __shfl_down_sync(0xffffffffu, __uint_as_float(rb[i]), 1);   // P0 of input column m+1
              ev[i] = (lane == 0) ? le[k] : left;          // zero before the first input column
              od_[i] = (lane == 31) ? re[k] : right;       // zero beyond the last one
              if (W < 32) {                                // row seams inside the warp are image edges
                ev[i] = (wcol == 0) ? 0.f : ev[i];
                od_[i] = (wcol == W - 1) ? 0.f : od_[i];
              }
            }
          }
#pragma unroll
          for (int c0 = 0; c0 < 32; c0 += 16) {
            tmem_ld16_nowait(trow + 0 * COUT + cg + c0, &ra[c0]);       // P1
            tmem_ld16_nowait(trow + 2 * COUT + cg + c0, &rb[c0]);       // P2
          }
          tmem_ld_wait();
          if (cg + 32 >= COUT) {                      // whole tile in registers: hand it back to the MMA warp
            tc_fence_before();
            mbar_arrive(&acc_empty[t]);
          }
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            ev[i] = (ev[i] + __uint_as_float(ra[i])) * corr;
            od_[i] = (od_[i] + __uint_as_float(rb[i])) * corr;
          }
          }
          // coalesced channels-last path (BN/residual/act inside); W < 32: the warp's two input rows map to output rows that are
          // not adjacent in memory -> per-thread stores below
          if (H16 && W >= 32 && live && p.out_ndhwc) {    // fp16 output, no residual (checked at the entry point)
            __half* y0 = reinterpret_cast<__half*>(p.y) + (vox - 2 * lane) * YS + cg;
            store_ndhwc_chunk32(tpose + q * TP_WARP_FLOATS, lane, ev, y0, nullptr, 2 * YS, s_scale + cg, s_shift + cg, p.act, vmask,
                                nullptr, &yamax);
            store_ndhwc_chunk32(tpose + q * TP_WARP_FLOATS, lane, od_, y0 + YS, nullptr, 2 * YS, s_scale + cg, s_shift + cg, p.act, vmask,
                                nullptr, &yamax);
          } else if (!H16 && W >= 32 && live && p.out_ndhwc && (!p.residual || p.res_ndhwc)) {
            // lane k owns output voxels (vox0 + 2k) and (vox0 + 2k + 1): two transposes with a 2-voxel lane stride
            float* y0 = p.y + (vox - 2 * lane) * YS + cg;
            const float* r0 = p.residual ? p.residual + (vox - 2 * lane) * YS + cg : nullptr;
            store_ndhwc_chunk32(tpose + q * TP_WARP_FLOATS, lane, ev, y0, r0, 2 * YS, s_scale + cg, s_shift + cg, p.act, vmask);
            store_ndhwc_chunk32(tpose + q * TP_WARP_FLOATS, lane, od_, y0 + YS, r0 ? r0 + YS : nullptr, 2 * YS, s_scale + cg,
                                s_shift + cg, p.act, vmask);
          } else if (live && cvalid) {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              ev[i] = fmaf(ev[i], s_scale[cg + i], s_shift[cg + i]);
              od_[i] = fmaf(od_[i], s_scale[cg + i], s_shift[cg + i]);
            }
            if (p.residual) {
              if (p.res_ndhwc) {
                const float4* rp = reinterpret_cast<const float4*>(p.residual + vox * YS + cg);
                const float4* rq = reinterpret_cast<const float4*>(p.residual + (vox + 1) * YS + cg);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                  const float4 a = __ldg(rp + i), bq = __ldg(rq + i);
                  ev[4 * i] += a.x, ev[4 * i + 1] += a.y, ev[4 * i + 2] += a.z, ev[4 * i + 3] += a.w;
                  od_[4 * i] += bq.x, od_[4 * i + 1] += bq.y, od_[4 * i + 2] += bq.z, od_[4 * i + 3] += bq.w;
                }
              } else {
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                  if (cg + i >= p.cout_real) continue;
                  const float2 rv = __ldg(reinterpret_cast<const float2*>(p.residual + ncdhw0 + (size_t)(cg + i) * plane));
                  ev[i] += rv.x, od_[i] += rv.y;
                }
              }
            }
            if (p.act == OSB_ACT_RELU) {
#pragma unroll
              for (int i = 0; i < 32; ++i) ev[i] = fmaxf(ev[i], 0.f), od_[i] = fmaxf(od_[i], 0.f);
            } else if (p.act == OSB_ACT_LEAKY) {
#pragma unroll
              for (int i = 0; i < 32; ++i) {
                ev[i] = ev[i] > 0.f ? ev[i] : 0.01f * ev[i];
                od_[i] = od_[i] > 0.f ? od_[i] : 0.01f * od_[i];
              }
            }
            if constexpr (H16) {
              __half* yh = reinterpret_cast<__half*>(p.y);
              if (p.out_ndhwc) {
                uint2* yp = reinterpret_cast<uint2*>(yh + vox * YS + cg);
                uint2* yq = reinterpret_cast<uint2*>(yh + (vox + 1) * YS + cg);
#pragma unroll
                for (int i = 0; i < 32; ++i) yamax = fmaxf(yamax, fmaxf(fabsf(ev[i]), fabsf(od_[i])));
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                  yp[i] = make_uint2(cvt_f16x2_sat(ev[4 * i], ev[4 * i + 1]), cvt_f16x2_sat(ev[4 * i + 2], ev[4 * i + 3]));
                  yq[i] = make_uint2(cvt_f16x2_sat(od_[4 * i], od_[4 * i + 1]), cvt_f16x2_sat(od_[4 * i + 2], od_[4 * i + 3]));
                }
              } else {
#pragma unroll
                for (int i = 0; i < 32; ++i)           // columns 2w, 2w+1 as one fp16 pair
                  if (cg + i < p.cout_real) {
                    yamax = fmaxf(yamax, fmaxf(fabsf(ev[i]), fabsf(od_[i])));
                    *reinterpret_cast<uint32_t*>(yh + ncdhw0 + (size_t)(cg + i) * plane) = cvt_f16x2_sat(ev[i], od_[i]);
                  }
              }
            } else if (p.out_ndhwc) {
              float4* yp = reinterpret_cast<float4*>(p.y + vox * YS + cg);
              float4* yq = reinterpret_cast<float4*>(p.y + (vox + 1) * YS + cg);
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                yp[i] = make_float4(ev[4 * i], ev[4 * i + 1], ev[4 * i + 2], ev[4 * i + 3]);
                yq[i] = make_float4(od_[4 * i], od_[4 * i + 1], od_[4 * i + 2], od_[4 * i + 3]);
              }
            } else {
#pragma unroll
              for (int i = 0; i < 32; ++i)             // columns 2w, 2w+1 of consecutive lanes: 256 contiguous bytes per warp
                if (cg + i < p.cout_real) *reinterpret_cast<float2*>(p.y + ncdhw0 + (size_t)(cg + i) * plane) = make_float2(ev[i], od_[i]);
            }
          }
        }
      }
      for (int t = ntiles; t < TILES; ++t) {            // unused tiles keep the barrier phases in step
        mbar_wait_relaxed(&acc_full[t], itc & 1);
        mbar_arrive(&acc_empty[t]);
      }
    }
    if constexpr (H16) tc_report_overflow(p.overflow, yamax);
  }
  // ---------------------------------------------------------------------------------------------- weight-slice producer
  // One elected lane streams the pre-swizzled (kd, chunk, kh) slices with 1-D TMA bulk copies into the two buffers of tap kh, up
  // to a whole use ahead of the MMAs (tc_common.cuh: bulk_g2s).
  else if (warp == 9) {
    if (elect_one()) {
      const uint8_t* wsrc = reinterpret_cast<const uint8_t*>(p.w);
      uint32_t bph[KS] = {};
      for (int it = blockIdx.x; it < p.items; it += gridDim.x) {
        const ItemDc w = decode_dc<C>(p, it);
        for (int kd = 0; kd < KS; ++kd) {
          if (!kd_valid(w.od, kd, p.D)) continue;         // same phase enumeration as the MMA warp and the A loaders
          for (int ch = 0; ch < nchunk; ++ch) {
            for (int kh = 0; kh < KS; ++kh) {
              if (!kh_valid(w.ph, kh)) continue;
              const uint32_t slot = (bph[kh] & 1) * KS + kh;
              const size_t slice = ((size_t)kd * nchunk + ch) * KS + kh;
              mbar_wait_relaxed(&b_empty[slot], ((bph[kh] >> 1) & 1) ^ 1);
              mbar_arrive_expect_tx(&b_full[slot], C::B_SLICE);
              bulk_g2s(b_buf + slot * C::B_SLICE, wsrc + slice * C::B_SLICE, C::B_SLICE, &b_full[slot]);
              ++bph[kh];
            }
          }
        }
      }
    }
    __syncwarp();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
}

template <int COUT, int KC, int W, int TILES, bool GW = false, int KS = 3, bool H16 = false>
static int launch_tcdc(TcdcParams& p, cudaStream_t stream) {
  using C = TcdcCfg<COUT, KC, W, TILES, GW, KS>;
  auto kernel = conv3d_tcdc_kernel<COUT, KC, W, TILES, GW, KS, H16>;
  static PerDeviceFlag configured;
  if (!configured.here()) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM);
    if (e != cudaSuccess) {
      set_error("conv3d_tcg: cannot reserve %zu bytes of shared memory: %s", C::SMEM, cudaGetErrorString(e));
      return OSB_ECUDA;
    }
    configured.here() = true;
  }
  if (W >= 32 && p.ystride && p.ystride != COUT) {
    set_error("conv3d_tcdc: channel slices are instantiated for W = 16 only");
    return OSB_EUNSUPPORTED;
  }
  p.hblocks = (p.H + C::HBLK - 1) / C::HBLK;
  if (p.cout_real <= 0 || p.cout_real > COUT) p.cout_real = COUT;
  if (GW) p.ctiles = (p.Wr + C::CSTEP - 1) / C::CSTEP;
  else p.Wr = W, p.ctiles = 1;
  const long long items = (long long)p.B * (2 * p.D) * 2 * p.hblocks * p.ctiles;
  OSB_REQUIRE(items < (1ll << 31), "conv3d_tcdc: too many work items");
  p.items = (int)items;
  const int sms = sm_count();
  const int grid = p.items < sms ? p.items : sms;
  kernel<<<grid, C::THREADS, C::SMEM, stream>>>(p);
  count_launch();
  cudaError_t le = cudaGetLastError();
  if (le != cudaSuccess) {
    cudaFuncAttributes fa{};
    (void)cudaFuncGetAttributes(&fa, kernel);
    set_error("conv3d_tcdc_kernel<%d,%d,%d,%d>: launch failed: %s (threads %d, kernel maxThreadsPerBlock %d, regs %d, static smem %zu, "
              "dynamic smem %zu, max dynamic %d)", COUT, KC, W, TILES, cudaGetErrorString(le), C::THREADS, fa.maxThreadsPerBlock,
              fa.numRegs, fa.sharedSizeBytes, C::SMEM, fa.maxDynamicSharedSizeBytes);
    return OSB_ECUDA;
  }
  return OSB_OK;
}

// conv3d_tcdq.cu: one work item per output-parity quad (conv6 shape); -1 = shape not instantiated there
int launch_tcdq(const float* x, const void* w, const float* scale, const float* shift, const float* residual, float* y, int B,
                int Cin, int Cout, int D, int H, int W, int act, cudaStream_t stream);

}  // namespace osb

extern "C" {

int osb_deconv3d_tc_supported(int Cin, int Cout, int W) {
  if (Cin % 16 != 0 || Cin < 16) return 0;
  if ((W == 32 && Cout == 64) || (W == 64 && Cout == 32)) return 1;                          // whole-row variants
  return (osb_tc_general_width(W) && (Cout == 32 || Cout == 64)) ? 1 : 0;                   // 128-column tiles of the INPUT row
}

int osb_deconv3d_k4_tc_supported(int Cin, int Cout, int W) {
  if (Cin % 16 != 0 || Cin < 16) return 0;
  return ((W == 32 && Cout == 64) || (W == 64 && Cout == 32) || (W == 16 && (Cout == 64 || Cout == 32))) ? 1 : 0;
}

static int deconv3d_k4_tc_impl(const float* x_ndhwc, const void* w_split, const float* scale, const float* shift,
                               const float* residual, float* y, int B, int Cin, int Cout, int cout_real, int D, int H, int W, int act,
                               int out_ndhwc, int res_ndhwc, int ystride, osb_stream_t stream);

int osb_deconv3d_k4_tc_fwd(const float* x_ndhwc, const void* w_split, const float* scale, const float* shift,
                           const float* residual, float* y, int B, int Cin, int Cout, int cout_real, int D, int H, int W, int act,
                           int out_ndhwc, int res_ndhwc, osb_stream_t stream) {
  return deconv3d_k4_tc_impl(x_ndhwc, w_split, scale, shift, residual, y, B, Cin, Cout, cout_real, D, H, W, act, out_ndhwc, res_ndhwc, 0,
                             stream);
}

int osb_deconv3d_k4_tc_cs_fwd(const float* x_ndhwc, const void* w_split, const float* scale, const float* shift, float* y, int B,
                              int Cin, int Cout, int D, int H, int W, int act, int ystride, osb_stream_t stream) {
  return deconv3d_k4_tc_impl(x_ndhwc, w_split, scale, shift, nullptr, y, B, Cin, Cout, Cout, D, H, W, act, 1, 1, ystride, stream);
}

static int deconv3d_k4_tc_impl(const float* x_ndhwc, const void* w_split, const float* scale, const float* shift,
                               const float* residual, float* y, int B, int Cin, int Cout, int cout_real, int D, int H, int W, int act,
                               int out_ndhwc, int res_ndhwc, int ystride, osb_stream_t stream) {
  using namespace osb;
  OSB_REQUIRE(x_ndhwc && w_split && y, "deconv3d_k4_tc: null pointer");
  OSB_REQUIRE(ystride == 0 || (ystride >= Cout && ystride % 4 == 0 && out_ndhwc && (!residual || res_ndhwc)),
              "deconv3d_k4_tc: a channel slice (ystride %d) needs channels-last tensors", ystride);
  OSB_REQUIRE(B > 0 && D > 0 && H > 0, "deconv3d_k4_tc: empty shape");
  OSB_REQUIRE(osb_deconv3d_k4_tc_supported(Cin, Cout, W), "deconv3d_k4_tc: unsupported shape Cin=%d Cout=%d W=%d", Cin, Cout, W);
  OSB_REQUIRE(act >= 0 && act <= 2, "deconv3d_k4_tc: unknown activation %d", act);
  OSB_REQUIRE(cout_real >= 1 && cout_real <= Cout && (out_ndhwc == 0 || cout_real == Cout) && (!residual || res_ndhwc == 0 || cout_real == Cout),
              "deconv3d_k4_tc: only NCDHW tensors may hold fewer (%d) channels than the packed %d", cout_real, Cout);
  TcdcParams p{};
  p.cout_real = cout_real, p.ystride = ystride;
  p.x = x_ndhwc, p.w = w_split, p.scale = scale, p.shift = shift, p.residual = residual, p.y = y;
  p.B = B, p.D = D, p.H = H, p.Cin = Cin, p.act = act, p.out_ndhwc = out_ndhwc, p.res_ndhwc = res_ndhwc;
  p.kappa = rz_kappa(), p.overflow = tc_overflow_flag();
  OSB_REQUIRE(p.overflow, "tensor-core conv: cannot allocate the overflow flag");
  cudaStream_t s = (cudaStream_t)stream;
  if (W == 16 && Cout == 64) return launch_tcdc<64, 16, 16, 2, false, 4>(p, s);   // StereoBase conv3_up: 6c -> 4c = 96 as slices 64 + 32
  if (W == 16 && Cout == 32) return launch_tcdc<32, 16, 16, 4, false, 4>(p, s);
  if (W == 32) return launch_tcdc<64, 16, 32, 2, false, 4>(p, s);
  return launch_tcdc<32, 16, 64, 4, false, 4>(p, s);
}

// ---- fp16 activations (H16 instantiations of the k4 kernel): same shapes as osb_deconv3d_k4_tc_supported, no residual
static int deconv3d_k4_tc_h16_impl(const void* x_ndhwc, const void* w_split, const float* scale, const float* shift, float* y, int B,
                                   int Cin, int Cout, int cout_real, int D, int H, int W, int act, int out_ndhwc, int ystride,
                                   osb_stream_t stream) {
  using namespace osb;
  OSB_REQUIRE(x_ndhwc && w_split && y, "deconv3d_k4_tc_h16: null pointer");
  OSB_REQUIRE(B > 0 && D > 0 && H > 0, "deconv3d_k4_tc_h16: empty shape");
  OSB_REQUIRE(osb_deconv3d_k4_tc_supported(Cin, Cout, W), "deconv3d_k4_tc_h16: unsupported shape Cin=%d Cout=%d W=%d", Cin, Cout, W);
  OSB_REQUIRE(act >= 0 && act <= 2, "deconv3d_k4_tc_h16: unknown activation %d", act);
  OSB_REQUIRE(ystride == 0 || (W == 16 && ystride >= Cout && ystride % 4 == 0 && out_ndhwc), "deconv3d_k4_tc_h16: bad channel stride %d",
              ystride);
  OSB_REQUIRE(cout_real >= 1 && cout_real <= Cout && (out_ndhwc == 0 || cout_real == Cout),
              "deconv3d_k4_tc_h16: only NCDHW outputs may hold fewer (%d) channels than the packed %d", cout_real, Cout);
  OSB_REQUIRE((reinterpret_cast<uintptr_t>(x_ndhwc) & 15) == 0 && (reinterpret_cast<uintptr_t>(w_split) & 15) == 0 &&
                  (reinterpret_cast<uintptr_t>(y) & 7) == 0,
              "deconv3d_k4_tc_h16: x and w must be 16-byte, y 8-byte aligned");
  TcdcParams p{};
  p.cout_real = cout_real, p.ystride = ystride;
  p.x = static_cast<const float*>(x_ndhwc), p.w = w_split, p.scale = scale, p.shift = shift, p.y = y;
  p.B = B, p.D = D, p.H = H, p.Cin = Cin, p.act = act, p.out_ndhwc = out_ndhwc ? 1 : 0, p.res_ndhwc = 1;
  p.kappa = rz_kappa(), p.overflow = tc_overflow_flag();
  OSB_REQUIRE(p.overflow, "tensor-core conv: cannot allocate the overflow flag");
  cudaStream_t s = (cudaStream_t)stream;
  if (W == 16 && Cout == 64) return launch_tcdc<64, 16, 16, 2, false, 4, true>(p, s);
  if (W == 16 && Cout == 32) return launch_tcdc<32, 16, 16, 4, false, 4, true>(p, s);
  if (W == 32) return launch_tcdc<64, 16, 32, 2, false, 4, true>(p, s);
  return launch_tcdc<32, 16, 64, 4, false, 4, true>(p, s);
}

int osb_deconv3d_k4_tc_h16_fwd(const void* x_ndhwc, const void* w_split, const float* scale, const float* shift, float* y, int B, int Cin,
                               int Cout, int cout_real, int D, int H, int W, int act, int out_ndhwc, osb_stream_t stream) {
  return deconv3d_k4_tc_h16_impl(x_ndhwc, w_split, scale, shift, y, B, Cin, Cout, cout_real, D, H, W, act, out_ndhwc, 0, stream);
}

int osb_deconv3d_k4_tc_cs_h16_fwd(const void* x_ndhwc, const void* w_split, const float* scale, const float* shift, float* y, int B,
                                  int Cin, int Cout, int D, int H, int W, int act, int ystride, osb_stream_t stream) {
  return deconv3d_k4_tc_h16_impl(x_ndhwc, w_split, scale, shift, y, B, Cin, Cout, Cout, D, H, W, act, 1, ystride, stream);
}

int osb_deconv3d_k3_tc_fwd(const float* x_ndhwc, const void* w_split, const float* scale, const float* shift,
                           const float* residual, float* y, int B, int Cin, int Cout, int D, int H, int W, int act,
                           int out_ndhwc, int res_ndhwc, osb_stream_t stream) {
  using namespace osb;
  OSB_REQUIRE(x_ndhwc && w_split && y, "deconv3d_k3_tc: null pointer");
  OSB_REQUIRE(B > 0 && D > 0 && H > 0, "deconv3d_k3_tc: empty shape");
  OSB_REQUIRE(osb_deconv3d_tc_supported(Cin, Cout, W), "deconv3d_k3_tc: unsupported shape Cin=%d Cout=%d W=%d", Cin, Cout, W);
  OSB_REQUIRE(act >= 0 && act <= 2, "deconv3d_k3_tc: unknown activation %d", act);
  TcdcParams p{};
  p.x = x_ndhwc, p.w = w_split, p.scale = scale, p.shift = shift, p.residual = residual, p.y = y;
  p.B = B, p.D = D, p.H = H, p.Cin = Cin, p.act = act, p.out_ndhwc = out_ndhwc, p.res_ndhwc = res_ndhwc;
  p.kappa = rz_kappa(), p.overflow = tc_overflow_flag();
  OSB_REQUIRE(p.overflow, "tensor-core conv: cannot allocate the overflow flag");
  cudaStream_t s = (cudaStream_t)stream;
  {
    // conv6 (64 -> 32 at W' = 64), channels-last: the parity-quad kernel stages 4 units where this file's kernel stages 9
    static const int quad = [] { const char* e = getenv("OSB_TCDQ"); return e ? atoi(e) : 1; }();
    if (quad && W == 64 && Cout == 32 && out_ndhwc && (!residual || res_ndhwc)) {
      const int rc = launch_tcdq(x_ndhwc, w_split, scale, shift, residual, y, B, Cin, Cout, D, H, W, act, s);
      if (rc >= 0) return rc;
    }
  }
  if (W == 32 && Cout == 64) return launch_tcdc<64, 16, 32, 2>(p, s);
  if (W == 64 && Cout == 32) return launch_tcdc<32, 16, 64, 5>(p, s);
  p.Wr = W;
  if (Cout == 64) return launch_tcdc<64, 16, 128, 2, true>(p, s);
  return launch_tcdc<32, 16, 128, 5, true>(p, s);
}
}
