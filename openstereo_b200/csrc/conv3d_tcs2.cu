// Tensor-core (tcgen05) Conv3d 3x3x3 STRIDE 2, pad 1: the down-sampling convs of the hourglasses
//   conv1 32->64 (1/4 -> 1/8 res) and conv3 64->128 / 64->64 (1/8 -> 1/16 res): gwcnet/hourglass.py:19-29,
//   psmnet/psmnet_cost_processor.py:79-94.
// Same machinery as conv3d_tcg.cu (3xFP16 split, LDG-staged swizzled operands, warp-specialised persistent CTA, taps
// stacked along N and recombined in the epilogue); what changes is the gather:
//   out[ow] = in[2ow-1].W0 + in[2ow].W1 + in[2ow+1].W2.  With E[j] = in[2j] (even columns) and O[j] = in[2j+1] (odd columns)
//   this is  out[ow] = E[ow].W1 + O[ow].W2 + O[ow-1].W0 ,  so per (output tile, kd, kh) the loaders stage TWO operand tiles
//   -- the even and the odd columns of the RO = 128/Wo input rows 2*oh + kh - 1 -- and the issuer runs
//   E x W1 (N = Cout) into accumulator columns [0,Cout) and O x [W0 | W2] (N = 2 Cout) into [Cout, 3 Cout); the epilogue
//   adds P1[ow] + P2[ow] + P0[ow-1] (a single left shift, zero at ow = 0 = the conv's left padding).
// Weight slices are packed with the kw order (1, 0, 2) so both MMAs read contiguous rows.
// GENERAL WIDTHS (GW = true, W = 128 instantiations; see conv3d_tcg.cu): an M tile is a 128-column segment of one OUTPUT row of
// runtime width Wr starting at output column ct * 127 - 1; tile column 0 is the halo that provides O[ow-1] (zero at ow = -1) and is
// not stored.
#include "tc_common.cuh"

namespace osb {

struct Tcs2Params {
  const float* x;          // (B, D, H, W, Cin) channels-last (fp16 in the H16 instantiations)
  const void* w;           // fp16 [3 kd][Cin/KC][3 kh][3*Cout][KC hi | KC lo]  (ops.pack_tc_weight)
  const float* scale;
  const float* shift;
  const float* residual;
  float* y;                // fp16 in the H16 instantiations (channels-last only)
  int B, D, H, Cin;        // INPUT extent D x H x (2*WO); output is D/2 x H/2 x WO
  int act;
  float kappa;       // expected round-towards-zero loss per accumulating MMA (tc_common.cuh)
  unsigned int* overflow;  // sticky fp16-range flag (tc_common.cuh)
  int out_ndhwc, res_ndhwc;
  int items, hblocks;
  int Wr, ctiles;          // general-width instantiations: OUTPUT width and column tiles per row (whole-row kernels: W, 1)
  int ystride;             // channels per voxel of the channels-last y / residual (0 = COUT); > COUT: this launch writes a channel slice
};

template <int COUT, int KC, int W, int TILES, bool GW = false>     // W = OUTPUT width
struct Tcs2Cfg {
  static_assert(!GW || W == 128, "general-width tiles are 128-column segments of one output row");
  static constexpr int HALO = GW ? 1 : 0;                   // halo columns on the LEFT of a column tile
  static constexpr int CSTEP = 128 - HALO;                  // output columns a column tile produces
  static constexpr int R = 128 / W;                         // OUTPUT image rows per M tile
  static constexpr int ROWB = KC * 4;                       // bytes per K-major operand row: [KC fp16 hi | KC fp16 lo]
  static constexpr int UNIT_BYTES = 128 * ROWB;
  static constexpr int N3 = 3 * COUT;
  static constexpr int B_SLICE = N3 * ROWB;                 // one kh weight slice (hi and lo halves of every row)
  // A-unit ring.  NLW loader warps (1-4 and 10) fill the units round-robin (unit u belongs to warp u mod NLW) into a ring as deep as
  // shared memory allows (at most 10 units).  Each loader warp enumerates ONLY ITS OWN units: when every warp walked the whole
  // (tile, tap) sequence and picked every NLW-th unit, that scalar control flow was the bound of these kernels -- a conv6 run with
  // loads, conversions, MMAs and stores all disabled still took 0.37 of 0.69 ms, two thirds of the loader warps' stall samples on
  // the loop lines (profiles/r2_conv6_barrier_skeleton_stalls.txt).
  static constexpr int NLW = 5;
  static constexpr int FIXED_SMEM = 1024 + TC_BSLOTS * 3 * B_SLICE + 1024 + 2 * 4 * 2 * 32 * 4 + 3 * COUT * 4 + TP_BYTES;
  static constexpr int STAGES = (232448 - FIXED_SMEM) / UNIT_BYTES < 10 ? (232448 - FIXED_SMEM) / UNIT_BYTES : 10;
  static_assert(STAGES >= NLW, "the ring must hold at least one unit per loader warp");
  static constexpr int NU = TILES * 3 * 2;                   // units of one (kd, chunk) phase: (tile, kh, column parity)
  static constexpr int HBLK = TILES * R;                    // output rows per work item
  static constexpr int KSTEPS = KC / 16;                    // K = 16 fp16 channels per MMA
  static constexpr int LO = KC / 8;                         // descriptor offset (16-byte units) of the lo half of a row
  static constexpr int A_OFF = 0;
  static constexpr int B_OFF = A_OFF + STAGES * UNIT_BYTES;
  static constexpr int BAR_OFF = B_OFF + TC_BSLOTS * 3 * B_SLICE;
  static constexpr int THREADS = 32 + 128 + 128 + 64;       // MMA | A loaders | epilogue | weight loaders (11 warps)
  static constexpr size_t SMEM = 1024 + (size_t)BAR_OFF + 1024 + 2 * 4 * 2 * 32 * 4 + 3 * COUT * 4 + TP_BYTES;
  static_assert(SMEM <= 232448, "shared memory budget of one CTA exceeded");
  static_assert(TILES * N3 <= 512, "accumulators exceed TMEM");
  static_assert(B_SLICE % 1024 == 0 && UNIT_BYTES % 1024 == 0, "operand tiles must stay 1024-byte aligned");
  static_assert(COUT % 16 == 0 && 2 * COUT <= 256, "invalid UMMA N");
};

// H16: fp16 activations in and out, one hi x hi MMA per k-step (see conv3d_tcg.cu)
template <int COUT, int KC, int W, int TILES, bool GW = false, bool H16 = false>
__global__ void __launch_bounds__(Tcs2Cfg<COUT, KC, W, TILES, GW>::THREADS, 1) conv3d_tcs2_kernel(const Tcs2Params p) {
  using C = Tcs2Cfg<COUT, KC, W, TILES, GW>;
  using A = TcAct<H16>;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* a_buf = smem + C::A_OFF;
  uint8_t* b_buf = smem + C::B_OFF;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::BAR_OFF);
  uint64_t* a_ready = bars;                         // [STAGES] loaders -> MMA        (32 arrivals: one warp)
  uint64_t* a_empty = a_ready + C::STAGES;          // [STAGES] MMA -> loaders        (tcgen05.commit)
  uint64_t* b_full = a_empty + C::STAGES;           // [2][3]   weight producer -> MMA (expect_tx + TMA bytes)
  uint64_t* b_empty = b_full + TC_BSLOTS * 3;       // [2][3]   MMA -> weight producer (tcgen05.commit)
  uint64_t* acc_full = b_empty + TC_BSLOTS * 3;                 // [TILES]
  uint64_t* acc_empty = acc_full + TILES;           // [TILES]  (128 arrivals)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + TILES);
  float* xchg = reinterpret_cast<float*>(smem + C::BAR_OFF + 1024);   // [2][4 quadrants][2 sides][32]
  float* s_scale = xchg + 2 * 4 * 2 * 32;
  float* s_shift = s_scale + COUT;
  float* zeros = s_shift + COUT;
  float* tpose = zeros + COUT;                      // [4 warps][32][TP_STRIDE] transpose tiles of the epilogue

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nchunk = p.Cin / KC;
  const int Wp = GW ? p.Wr : W;                     // OUTPUT width (the input is 2 * Wp wide)
  const int YS = (W < 32 && p.ystride) ? p.ystride : COUT;   // (compile-time COUT in the wide instantiations: slices exist at W' = 16 only)      // channel stride of the channels-last output / residual
  const int ctiles = GW ? p.ctiles : 1;             // work item = (b, od, row block, column tile), column tile fastest

  if (threadIdx.x == 0) {
    for (int s = 0; s < C::STAGES; ++s) {
      mbar_init(&a_ready[s], 32);                     // one loader warp fills a unit
      mbar_init(&a_empty[s], 1);
    }
    for (int k = 0; k < TC_BSLOTS * 3; ++k) {
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
    const uint32_t idesc_e = idesc_f16(128, COUT), idesc_o = idesc_f16(128, 2 * COUT);
    const uint64_t dbase = (KC == 32) ? desc_sw128_base() : desc_sw64_base();
    const uint32_t b16 = (smem_u32(b_buf) & 0x3FFFF) >> 4;
    const int Do = p.D / 2, Ho = p.H / 2;
    uint32_t unitc = 0, phc = 0, itc = 0;
    for (int it = blockIdx.x; it < p.items; it += gridDim.x, ++itc) {
      const int hb = (it / ctiles) % p.hblocks;
      const int od = (it / (ctiles * p.hblocks)) % Do;
      const int ntiles = min(TILES, (Ho - hb * C::HBLK + C::R - 1) / C::R);
      uint32_t started = 0;
      for (int kd = 0; kd < 3; ++kd) {
        const int din = 2 * od + kd - 1;
        if (din < 0 || din >= p.D) continue;
        for (int ch = 0; ch < nchunk; ++ch, ++phc) {
          const bool last_phase = (kd == 2) && (ch == nchunk - 1);     // din = 2*od+1 always exists (even D)
#pragma unroll
          for (int t = 0; t < TILES; ++t) {
#pragma unroll
            for (int kh = 0; kh < 3; ++kh) {
#pragma unroll
              for (int par = 0; par < 2; ++par) {       // par 0: even input columns (kw = 1); par 1: odd columns (kw = 0, 2)
                const uint32_t slot = unitc % C::STAGES, ph = (unitc / C::STAGES) & 1;
                mbar_wait(&a_ready[slot], ph);
                if (t == 0 && par == 0) mbar_wait(&b_full[(phc & 1) * 3 + kh], (phc >> 1) & 1);   // first use of slice kh in this phase
                tc_fence_after();
                const uint32_t accum = (started >> (2 * t + par)) & 1;
                if (((started >> (2 * t)) & 3u) == 0u) {     // first touch of this tile in this item (unused tiles too)
                  mbar_wait(&acc_empty[t], (itc & 1) ^ 1);
                  tc_fence_after();
                }
                started |= 1u << (2 * t + par);
                if (t < ntiles) {
                  if (elect_one()) {
                    const uint64_t da0 = dbase | (uint64_t)((smem_u32(a_buf + slot * C::UNIT_BYTES) & 0x3FFFF) >> 4);
                    // slice rows: [W1 (Cout) | W0 (Cout) | W2 (Cout)]; accumulator columns: [P1 | P0 | P2]
                    const uint32_t acc = tmem + t * C::N3 + (par ? COUT : 0);
                    const uint64_t db0 = dbase | (uint64_t)(b16 + (((phc & 1) * 3 + kh) * C::B_SLICE + (par ? COUT * C::ROWB : 0)) / 16);
                    const uint32_t idesc = par ? idesc_o : idesc_e;
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
                  if (t == TILES - 1 && par == 1) mma_commit(&b_empty[(phc & 1) * 3 + kh]);   // last user of slice kh in this phase
                  if (last_phase && kh == 2 && par == 1) mma_commit(&acc_full[t]); // tile t has received its last tap
                }
                __syncwarp();
                ++unitc;
              }
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
    const int WI = 2 * Wp;                           // input width
    const int Do = p.D / 2;
    uint32_t ubase = 0;                              // global index of the current phase's first unit
    int first = lw;                                  // this warp's first local unit index in the current phase: (ubase + first) % NLW == lw
    auto fill = [&](const typename A::T* base, size_t rstride, size_t cstride, int h_first, int h_step, uint32_t u, int col0) {
      // base: this lane's address for load 0; load j covers operand rows VPL*j .. VPL*j + VPL - 1 = columns (VPL*j) % W ..
      // of tile row (VPL*j) / W, read from image row h_first + h_step * tile row (rstride / cstride floats per tile row / column).
      // General widths: col0 = OUTPUT column of load 0 (-1 = the left halo; columns outside [0, Wp) are zero padding).
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
      const int ct = it % ctiles;
      const int hb = (it / ctiles) % p.hblocks;
      const int od = (it / (ctiles * p.hblocks)) % Do;
      const int b = it / (ctiles * p.hblocks * Do);
      const int h0 = hb * C::HBLK;                   // first OUTPUT row of the block
      const int col0 = ct * C::CSTEP - C::HALO + v0; // OUTPUT column of this lane's first load (whole-row kernels: v0)
      for (int kd = 0; kd < 3; ++kd) {
        const int din = 2 * od + kd - 1;
        if (din < 0 || din >= p.D) continue;
        const typename A::T* plane = reinterpret_cast<const typename A::T*>(p.x) + ((size_t)b * p.D + din) * p.H * (size_t)WI * p.Cin;
        for (int ch = 0; ch < nchunk; ++ch) {
#pragma unroll 1
          for (int j = first; j < C::NU; j += C::NLW) {       // local unit index = (t * 3 + kh) * 2 + par
            const int t = j / 6, kh = (j >> 1) % 3, par = j & 1;
            // operand row v = output voxel (row h0 + t*R + v / W, column v % W) reading input (2*row + kh - 1, 2*col + par)
            const int h_first = 2 * (h0 + t * C::R) + kh - 1;
            const typename A::T* base = plane + ((ptrdiff_t)h_first * WI + 2 * col0 + par) * p.Cin + ch * KC + c * 4;
            fill(base, (size_t)2 * WI * p.Cin, (size_t)2 * p.Cin, h_first, 2, ubase + j, col0);
          }
          ubase += C::NU;
          first = (first + C::NLW - C::NU % C::NLW) % C::NLW;
        }
      }
    }
    tc_report_overflow(p.overflow, amax);
  }
  // ---------------------------------------------------------------------------------------------- epilogue
  else if (warp < 9) {
    const int q = warp & 3;                          // TMEM lane quadrant this warp may read
    const int m = q * 32 + lane;                     // operand row owned by this thread
    const int rr = m / W, wcol = m % W;              // image row inside the tile, image column
    const bool has_left_q = ((q * 32) % W) != 0;     // the quadrant to the left continues the same image row
    const int Do = p.D / 2, Ho = p.H / 2;
    uint32_t itc = 0, exc = 0;
    float yamax = 0.f;                               // H16: largest stored magnitude (fp16 saturation at 65504)
    for (int it = blockIdx.x; it < p.items; it += gridDim.x, ++itc) {
      const int ct = it % ctiles;
      const int hb = (it / ctiles) % p.hblocks;
      const int d = (it / (ctiles * p.hblocks)) % Do;
      const int b = it / (ctiles * p.hblocks * Do);
      const int h0 = hb * C::HBLK;
      const int ntiles = min(TILES, (Ho - h0 + C::R - 1) / C::R);
      // general widths: output column of this thread's tile column; the halo column and columns beyond the image are not stored
      const int col = GW ? ct * C::CSTEP - C::HALO + m : wcol;
      const bool cvalid = !GW || (m >= C::HALO && col < Wp);
      const uint32_t vmask = GW ? __ballot_sync(0xffffffffu, cvalid) : 0xffffffffu;
      // input planes 2d-1, 2d, 2d+1: the first is missing for d = 0 (tc_common.cuh: rz_kappa)
      const float corr = 1.f + p.kappa * (float)(((d > 0) + 1 + (2 * d + 1 < p.D)) * nchunk * 3 * C::KSTEPS * A::TERMS);
      for (int t = 0; t < ntiles; ++t) {
        mbar_wait_relaxed(&acc_full[t], itc & 1);
        tc_fence_after();
        const int h = h0 + t * C::R + rr;
        const bool live = h < Ho;
        const ptrdiff_t vox = (((ptrdiff_t)b * Do + d) * Ho + h) * Wp + col;       // NDHWC voxel index (output)
        const size_t plane = (size_t)Do * Ho * Wp;                                 // NCDHW channel stride (output)
        const ptrdiff_t ncdhw0 = (ptrdiff_t)b * COUT * plane + ((ptrdiff_t)d * Ho + h) * Wp + col;
        const uint32_t trow = tmem + ((uint32_t)(q * 32) << 16) + t * C::N3;
#pragma unroll 1
        for (int cg = 0; cg < COUT; cg += 32) {
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
          float* xb = xchg + (exc & 1) * (4 * 2 * 32);
          ++exc;
          // accumulator column groups: raw[0] = P1 (kw=1, even columns), raw[1] = P0 (kw=0), raw[2] = P2 (kw=2)
          if (lane == 31) {
#pragma unroll
            for (int i = 0; i < 32; ++i) xb[(q * 2) * 32 + i] = __uint_as_float(raw[1][i]);
          }
          named_bar_sync(1, 128);
          const float* xl = has_left_q ? xb + ((q - 1) * 2) * 32 : zeros;
          float out[32];
#pragma unroll
          for (int i0 = 0; i0 < 32; i0 += 4) {        // neighbour values loaded unconditionally, merged with selects (no branches)
            const float4 l4 = *reinterpret_cast<const float4*>(xl + i0);
            const float le[4] = {l4.x, l4.y, l4.z, l4.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int i = i0 + k;
              float left = __shfl_up_sync(0xffffffffu, __uint_as_float(raw[1][i]), 1);   // P0 of output column ow-1
              left = (lane == 0) ? le[k] : left;                                        // zero at ow = 0 (left padding)
              if (W < 32) left = (wcol == 0) ? 0.f : left;                              // row seams inside the warp
              out[i] = ((left + __uint_as_float(raw[0][i])) + __uint_as_float(raw[2][i])) * corr;
            }
          }
          const uint32_t vm = (W < 32) ? __ballot_sync(0xffffffffu, live) : (live ? vmask : 0u);   // voxels of this warp that exist
          if (H16 && vm) {                             // channels-last fp16 output, no residual (checked at the entry point)
            store_ndhwc_chunk32(tpose + q * TP_WARP_FLOATS, lane, out, reinterpret_cast<__half*>(p.y) + (vox - lane) * YS + cg, nullptr, YS,
                                s_scale + cg, s_shift + cg, p.act, vm, nullptr, &yamax);
          } else if (!H16 && vm && p.out_ndhwc && (!p.residual || p.res_ndhwc)) {     // coalesced channels-last path (BN/residual/act inside)
            store_ndhwc_chunk32(tpose + q * TP_WARP_FLOATS, lane, out, p.y + (vox - lane) * YS + cg,
                                p.residual ? p.residual + (vox - lane) * YS + cg : nullptr, YS, s_scale + cg, s_shift + cg, p.act,
                                vm);
          } else if (!H16 && live && cvalid) {
#pragma unroll
            for (int i = 0; i < 32; ++i) out[i] = fmaf(out[i], s_scale[cg + i], s_shift[cg + i]);
            if (p.residual) {
              if (p.res_ndhwc) {
                const float4* rp = reinterpret_cast<const float4*>(p.residual + vox * YS + cg);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                  const float4 rv = __ldg(rp + i);
                  out[4 * i] += rv.x, out[4 * i + 1] += rv.y, out[4 * i + 2] += rv.z, out[4 * i + 3] += rv.w;
                }
              } else {
#pragma unroll
                for (int i = 0; i < 32; ++i) out[i] += __ldg(p.residual + ncdhw0 + (size_t)(cg + i) * plane);
              }
            }
            if (p.act == OSB_ACT_RELU) {
#pragma unroll
              for (int i = 0; i < 32; ++i) out[i] = fmaxf(out[i], 0.f);
            } else if (p.act == OSB_ACT_LEAKY) {
#pragma unroll
              for (int i = 0; i < 32; ++i) out[i] = out[i] > 0.f ? out[i] : 0.01f * out[i];
            }
            if (p.out_ndhwc) {
              float4* yp = reinterpret_cast<float4*>(p.y + vox * YS + cg);
#pragma unroll
              for (int i = 0; i < 8; ++i) yp[i] = make_float4(out[4 * i], out[4 * i + 1], out[4 * i + 2], out[4 * i + 3]);
            } else {
#pragma unroll
              for (int i = 0; i < 32; ++i) p.y[ncdhw0 + (size_t)(cg + i) * plane] = out[i];
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
  // One elected lane streams the pre-swizzled (kd, chunk, kh) slices with 1-D TMA bulk copies into the two buffer sets, up to a
  // whole phase ahead of the MMAs (tc_common.cuh: bulk_g2s).
  else if (warp == 9) {
    if (elect_one()) {
      const uint8_t* wsrc = reinterpret_cast<const uint8_t*>(p.w);
      uint32_t phc = 0;
      for (int it = blockIdx.x; it < p.items; it += gridDim.x) {
        const int od = (it / (ctiles * p.hblocks)) % (p.D / 2);
        for (int kd = 0; kd < 3; ++kd) {
          const int din = 2 * od + kd - 1;              // must enumerate the same phases as the MMA warp and the loaders
          if (din < 0 || din >= p.D) continue;
          for (int ch = 0; ch < nchunk; ++ch, ++phc) {
            for (int kh = 0; kh < 3; ++kh) {
              const uint32_t slot = (phc & 1) * 3 + kh;
              const size_t slice = ((size_t)kd * nchunk + ch) * 3 + kh;
              mbar_wait_relaxed(&b_empty[slot], ((phc >> 1) & 1) ^ 1);
              mbar_arrive_expect_tx(&b_full[slot], C::B_SLICE);
              bulk_g2s(b_buf + slot * C::B_SLICE, wsrc + slice * C::B_SLICE, C::B_SLICE, &b_full[slot]);
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

template <int COUT, int KC, int W, int TILES, bool GW = false, bool H16 = false>
static int launch_tcs2(Tcs2Params& p, cudaStream_t stream) {
  using C = Tcs2Cfg<COUT, KC, W, TILES, GW>;
  auto kernel = conv3d_tcs2_kernel<COUT, KC, W, TILES, GW, H16>;
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
    set_error("conv3d_tcs2: channel slices are instantiated for W = 16 only");
    return OSB_EUNSUPPORTED;
  }
  p.hblocks = (p.H / 2 + C::HBLK - 1) / C::HBLK;
  if (GW) p.ctiles = (p.Wr + C::CSTEP - 1) / C::CSTEP;
  else p.Wr = W, p.ctiles = 1;
  const long long items = (long long)p.B * (p.D / 2) * p.hblocks * p.ctiles;
  OSB_REQUIRE(items < (1ll << 31), "conv3d_tcs2: too many work items");
  p.items = (int)items;
  const int sms = sm_count();
  const int grid = p.items < sms ? p.items : sms;
  kernel<<<grid, C::THREADS, C::SMEM, stream>>>(p);
  count_launch();
  cudaError_t le = cudaGetLastError();
  if (le != cudaSuccess) {
    cudaFuncAttributes fa{};
    (void)cudaFuncGetAttributes(&fa, kernel);
    set_error("conv3d_tcs2_kernel<%d,%d,%d,%d>: launch failed: %s (threads %d, kernel maxThreadsPerBlock %d, regs %d, static smem %zu, "
              "dynamic smem %zu, max dynamic %d)", COUT, KC, W, TILES, cudaGetErrorString(le), C::THREADS, fa.maxThreadsPerBlock,
              fa.numRegs, fa.sharedSizeBytes, C::SMEM, fa.maxDynamicSharedSizeBytes);
    return OSB_ECUDA;
  }
  return OSB_OK;
}

}  // namespace osb

extern "C" {

int osb_conv3d_s2_tc_supported(int Cin, int Cout, int D, int H, int W) {
  if (Cin % 16 != 0 || Cin < 16 || D % 2 || H % 2 || W % 2) return 0;
  if ((W == 128 && Cout == 64) || (W == 64 && (Cout == 64 || Cout == 96 || Cout == 128)) || (W == 32 && (Cout == 64 || Cout == 96)))
    return 1;                                                                               // whole-row variants
  return (osb_tc_general_width(W / 2) && (Cout == 64 || Cout == 128)) ? 1 : 0;              // 128-column tiles of the OUTPUT row
}

static int conv3d_k3_s2_tc_impl(const float* x_ndhwc, const void* w_split, const float* scale, const float* shift,
                                const float* residual, float* y, int B, int Cin, int Cout, int D, int H, int W, int act,
                                int out_ndhwc, int res_ndhwc, int ystride, osb_stream_t stream) {
  using namespace osb;
  OSB_REQUIRE(ystride == 0 || (ystride >= Cout && ystride % 4 == 0 && out_ndhwc && (!residual || res_ndhwc)),
              "conv3d_k3_s2_tc: a channel slice (ystride %d) needs channels-last tensors", ystride);
  OSB_REQUIRE(x_ndhwc && w_split && y, "conv3d_k3_s2_tc: null pointer");
  OSB_REQUIRE(B > 0 && D > 0 && H > 0, "conv3d_k3_s2_tc: empty shape");
  OSB_REQUIRE(osb_conv3d_s2_tc_supported(Cin, Cout, D, H, W), "conv3d_k3_s2_tc: unsupported shape Cin=%d Cout=%d D=%d H=%d W=%d", Cin,
              Cout, D, H, W);
  OSB_REQUIRE(act >= 0 && act <= 2, "conv3d_k3_s2_tc: unknown activation %d", act);
  Tcs2Params p{};
  p.x = x_ndhwc, p.w = w_split, p.scale = scale, p.shift = shift, p.residual = residual, p.y = y;
  p.B = B, p.D = D, p.H = H, p.Cin = Cin, p.act = act, p.out_ndhwc = out_ndhwc, p.res_ndhwc = res_ndhwc;
  p.kappa = rz_kappa(), p.overflow = tc_overflow_flag();
  p.ystride = ystride;
  OSB_REQUIRE(p.overflow, "tensor-core conv: cannot allocate the overflow flag");
  cudaStream_t s = (cudaStream_t)stream;
  if (W == 32 && Cout == 96) return launch_tcs2<96, 16, 16, 1>(p, s);           // StereoBase conv3[0]: 4c -> 6c as two channel slices
  if (W == 32 && Cout == 64) return launch_tcs2<64, 16, 16, 2>(p, s);
  if (W == 128 && Cout == 64) return launch_tcs2<64, 16, 64, 2>(p, s);
  if (W == 64 && Cout == 64) return launch_tcs2<64, 16, 32, 2>(p, s);
  if (W == 64 && Cout == 128) return launch_tcs2<128, 16, 32, 1>(p, s);
  if (W == 64 && Cout == 96) return launch_tcs2<96, 16, 32, 1>(p, s);           // StereoBase conv2[0]: 2c -> 4c = 96
  p.Wr = W / 2;
  if (Cout == 64) return launch_tcs2<64, 16, 128, 2, true>(p, s);
  return launch_tcs2<128, 16, 128, 1, true>(p, s);
}

int osb_conv3d_k3_s2_tc_fwd(const float* x_ndhwc, const void* w_split, const float* scale, const float* shift,
                            const float* residual, float* y, int B, int Cin, int Cout, int D, int H, int W, int act,
                            int out_ndhwc, int res_ndhwc, osb_stream_t stream) {
  return conv3d_k3_s2_tc_impl(x_ndhwc, w_split, scale, shift, residual, y, B, Cin, Cout, D, H, W, act, out_ndhwc, res_ndhwc, 0, stream);
}

int osb_conv3d_k3_s2_tc_cs_fwd(const float* x_ndhwc, const void* w_split, const float* scale, const float* shift, float* y, int B,
                               int Cin, int Cout, int D, int H, int W, int act, int ystride, osb_stream_t stream) {
  return conv3d_k3_s2_tc_impl(x_ndhwc, w_split, scale, shift, nullptr, y, B, Cin, Cout, D, H, W, act, 1, 1, ystride, stream);
}

// ---- fp16 activations (H16 instantiations): the whole-row shapes of StereoBase's hourglass, channels-last, no residual
static bool s2_h16_shape(int Cin, int Cout, int W) {
  return Cin % 16 == 0 && Cin >= 16 && ((W == 128 && Cout == 64) || (W == 64 && Cout == 96) || (W == 32 && (Cout == 96 || Cout == 64)));
}

static int conv3d_k3_s2_tc_h16_impl(const void* x_ndhwc, const void* w_split, const float* scale, const float* shift, float* y, int B,
                                    int Cin, int Cout, int D, int H, int W, int act, int ystride, osb_stream_t stream) {
  using namespace osb;
  OSB_REQUIRE(x_ndhwc && w_split && y, "conv3d_k3_s2_tc_h16: null pointer");
  OSB_REQUIRE(B > 0 && D > 0 && H > 0 && D % 2 == 0 && H % 2 == 0, "conv3d_k3_s2_tc_h16: bad shape");
  OSB_REQUIRE(s2_h16_shape(Cin, Cout, W), "conv3d_k3_s2_tc_h16: unsupported shape Cin=%d Cout=%d W=%d", Cin, Cout, W);
  OSB_REQUIRE(act >= 0 && act <= 2, "conv3d_k3_s2_tc_h16: unknown activation %d", act);
  OSB_REQUIRE(ystride == 0 || (W == 32 && ystride >= Cout && ystride % 4 == 0), "conv3d_k3_s2_tc_h16: bad channel stride %d", ystride);
  OSB_REQUIRE((reinterpret_cast<uintptr_t>(x_ndhwc) & 15) == 0 && (reinterpret_cast<uintptr_t>(w_split) & 15) == 0 &&
                  (reinterpret_cast<uintptr_t>(y) & 7) == 0,
              "conv3d_k3_s2_tc_h16: x and w must be 16-byte, y 8-byte aligned");
  Tcs2Params p{};
  p.x = static_cast<const float*>(x_ndhwc), p.w = w_split, p.scale = scale, p.shift = shift, p.y = y;
  p.B = B, p.D = D, p.H = H, p.Cin = Cin, p.act = act, p.out_ndhwc = 1, p.res_ndhwc = 1;
  p.kappa = rz_kappa(), p.overflow = tc_overflow_flag();
  p.ystride = ystride;
  OSB_REQUIRE(p.overflow, "tensor-core conv: cannot allocate the overflow flag");
  cudaStream_t s = (cudaStream_t)stream;
  if (W == 32 && Cout == 96) return launch_tcs2<96, 16, 16, 1, false, true>(p, s);
  if (W == 32) return launch_tcs2<64, 16, 16, 2, false, true>(p, s);
  if (W == 128) return launch_tcs2<64, 16, 64, 2, false, true>(p, s);
  return launch_tcs2<96, 16, 32, 1, false, true>(p, s);
}

int osb_conv3d_s2_tc_h16_supported(int Cin, int Cout, int D, int H, int W) {
  return (D % 2 == 0 && H % 2 == 0 && s2_h16_shape(Cin, Cout, W)) ? 1 : 0;
}

int osb_conv3d_k3_s2_tc_h16_fwd(const void* x_ndhwc, const void* w_split, const float* scale, const float* shift, float* y, int B, int Cin,
                                int Cout, int D, int H, int W, int act, osb_stream_t stream) {
  return conv3d_k3_s2_tc_h16_impl(x_ndhwc, w_split, scale, shift, y, B, Cin, Cout, D, H, W, act, 0, stream);
}

int osb_conv3d_k3_s2_tc_cs_h16_fwd(const void* x_ndhwc, const void* w_split, const float* scale, const float* shift, float* y, int B,
                                   int Cin, int Cout, int D, int H, int W, int act, int ystride, osb_stream_t stream) {
  return conv3d_k3_s2_tc_h16_impl(x_ndhwc, w_split, scale, shift, y, B, Cin, Cout, D, H, W, act, ystride, stream);
}
}
