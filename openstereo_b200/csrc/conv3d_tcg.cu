// Generic tensor-core (tcgen05) Conv3d 3x3x3 stride 1 for the hourglass-interior layers whose image width is below the
// 128-row UMMA tile: an M tile is R = 128 / W consecutive image rows (W = 64 -> 2 rows, W = 32 -> 4 rows).
//   conv2 64->64 @ 1/8 res, conv4 128->128 (GwcNet) / 64->64 (PSMNet) @ 1/16 res:
//   gwcnet/hourglass.py:25-32, psmnet/psmnet_cost_processor.py:86-98.
// Same scheme as conv3d_tc.cu (3xFP16 split, kw taps stacked along N and un-shifted in the epilogue, LDG-staged swizzled
// operands, warp-specialised persistent CTA), generalised:
//   * an A "unit" is R consecutive input rows starting at block row s; tap kh of output tile t reads the unit with
//     s = t*R + kh - 1, so units are shared between taps/tiles whenever those starts coincide;
//   * K chunks are 16 channels (64-byte rows [16 hi | 16 lo] fp16, SWIZZLE_64B: one K = 16 MMA step each) so that the three
//     kh weight slices of a phase fit in shared memory next to the ring for Cout = 64 / 128;
//   * for Cout = 128 the kw-stacked N = 384 exceeds the UMMA maximum and is issued as three N = 128 MMAs;
//   * the epilogue's +-1 column shift never crosses an image-row boundary (tile rows are whole image rows).
// GENERAL WIDTHS (GW = true, W = 128 instantiations): an M tile is a 128-column SEGMENT of one image row of runtime width Wr,
// starting at column ct * (128 - 2 DIL) - DIL: the first / last DIL tile columns are a halo (loaded like any other column, zero
// outside the image -- the conv's padding), the kw-stacked partial sums are un-shifted across the whole tile exactly as before and
// only the 128 - 2 DIL interior columns that exist in the image are stored.  Work items gain a column-tile index (fastest), so
// widths such as 240 (the reference's 544x960 timing shape), 312 (KITTI) or 160 take the tensor-core path with 1.6 % halo overhead.
#include "tc_common.cuh"

namespace osb {

struct TcgParams {
  const float* x;          // (B, D, H, W, Cin) channels-last (fp16 in the H16 instantiations)
  const void* w;           // fp16 [3 kd][Cin/KC][3 kh][3*Cout][KC hi | KC lo]  (ops.pack_tc_weight)
  const float* scale;
  const float* shift;
  const float* residual;
  const float* gate;       // optional (B, H, W, Cout) channels-last multiplier applied after the activation (FeatureAtt), NDHWC output only
  float* y;                // fp16 in the H16 instantiations (channels-last only)
  int B, D, H, Cin;
  int act;
  float kappa;       // expected round-towards-zero loss per accumulating MMA (tc_common.cuh)
  unsigned int* overflow;  // sticky fp16-range flag (tc_common.cuh)
  int out_ndhwc, res_ndhwc;
  int items, hblocks;
  int Wr, ctiles;          // general-width instantiations: image width and column tiles per row (whole-row kernels: W, 1)
  int ystride;             // channels per voxel of the channels-last y / residual / gate tensors (0 = COUT); > COUT when this launch
                           // produces a channel SLICE of a wider tensor (pointers pre-offset to the slice's first channel)
};

template <int COUT, int KC, int W, int TILES, int DIL = 1, bool GW = false>
struct TcgCfg {
  static_assert(!GW || W == 128, "general-width tiles are 128-column segments of one image row");
  static constexpr int HALO = GW ? DIL : 0;                 // halo columns on each side of a column tile
  static constexpr int CSTEP = 128 - 2 * HALO;              // image columns a column tile produces
  // DIL = 2: dilated 2D convs of the backbone (layer4 of gwcnet_backbone.py:38-60, psmnet_backbone.py) as one-plane volumes:
  // tap kh of output row t reads input row t + (kh-1)*DIL, the kw-stacked partial sums are un-shifted by DIL columns.
  static_assert(DIL == 1 || (W == 128 && DIL == 2 && COUT >= 64), "dilation 2 is instantiated for full-width rows only");
  static constexpr int R = 128 / W;                         // image rows per M tile
  static constexpr int ROWB = KC * 4;                       // bytes per K-major operand row: [KC fp16 hi | KC fp16 lo]
  static constexpr int UNIT_BYTES = 128 * ROWB;
  static constexpr int N3 = 3 * COUT;
  static constexpr int NMMA = (N3 <= 256) ? 1 : 3;          // MMAs per (A unit, weight slice, k step)
  static constexpr int NPER = N3 / NMMA;
  static constexpr int B_SLICE = N3 * ROWB;                 // one kh weight slice (hi and lo halves of every row)
  // A-unit ring.  NLW loader warps (1-4 and 10) fill the units round-robin (unit u belongs to warp u mod NLW) into a ring as deep as
  // shared memory allows (at most 10 units).  Each loader warp enumerates ONLY ITS OWN units: when every warp walked the whole
  // (tile, tap) sequence and picked every NLW-th unit, that scalar control flow was the bound of these kernels -- a conv6 run with
  // loads, conversions, MMAs and stores all disabled still took 0.37 of 0.69 ms, two thirds of the loader warps' stall samples on
  // the loop lines (profiles/r2_conv6_barrier_skeleton_stalls.txt).
  static constexpr int NLW = 5;
  static constexpr int FIXED_SMEM = 1024 + TC_BSLOTS * 3 * B_SLICE + 1024 + 2 * 4 * 2 * DIL * 32 * 4 + 3 * COUT * 4 + TP_BYTES;
  static constexpr int STAGES = (232448 - FIXED_SMEM) / UNIT_BYTES < 10 ? (232448 - FIXED_SMEM) / UNIT_BYTES : 10;
  static_assert(STAGES >= NLW, "the ring must hold at least one unit per loader warp");
  static constexpr int S_FIRST = -DIL;                      // unit start rows run from S_FIRST to S_LAST (block-relative)
  static constexpr int S_LAST = (TILES - 1) * R + DIL;
  static constexpr int HBLK = TILES * R;                    // output rows per work item
  static constexpr int KSTEPS = KC / 16;                    // K = 16 fp16 channels per MMA
  static constexpr int LO = KC / 8;                         // descriptor offset (16-byte units) of the lo half of a row
  static constexpr int A_OFF = 0;
  static constexpr int B_OFF = A_OFF + STAGES * UNIT_BYTES;
  static constexpr int BAR_OFF = B_OFF + TC_BSLOTS * 3 * B_SLICE;
  static constexpr int THREADS = 32 + 128 + 128 + 64;       // MMA | A loaders | epilogue | weight loaders (11 warps)
  static constexpr size_t SMEM = 1024 + (size_t)BAR_OFF + 1024 + 2 * 4 * 2 * DIL * 32 * 4 + 3 * COUT * 4 + TP_BYTES;
  static_assert(SMEM <= 232448, "shared memory budget of one CTA exceeded");
  static_assert(TILES * N3 <= 512, "accumulators exceed TMEM");
  static_assert(B_SLICE % 1024 == 0 && UNIT_BYTES % 1024 == 0, "operand tiles must stay 1024-byte aligned");
  static_assert(NPER % 16 == 0 && NPER <= 256, "invalid UMMA N");
  // tile fed by unit s through tap kh, or -1
  static constexpr int tile_of(int s, int kh) {
    const int num = s - (kh - 1) * DIL;
    return (num >= 0 && num % R == 0 && num / R < TILES) ? num / R : -1;
  }
  static constexpr bool used(int s) { return tile_of(s, 0) >= 0 || tile_of(s, 1) >= 0 || tile_of(s, 2) >= 0; }
  // units of one (kd, chunk) phase in issue order: their number and the start row of the j-th one
  static constexpr int units_per_phase() {
    int n = 0;
    for (int s = S_FIRST; s <= S_LAST; ++s) n += used(s) ? 1 : 0;
    return n;
  }
  static constexpr int NU = units_per_phase();
  static constexpr int unit_s(int j) {
    int k = 0;
    for (int s = S_FIRST; s <= S_LAST; ++s)
      if (used(s)) {
        if (k == j) return s;
        ++k;
      }
    return S_LAST;
  }
};

// H16: fp16 activations in and out, one hi x hi MMA per k-step (tc_common.cuh: TcAct); the shared-memory layout is the split
// kernel's, the lo halves of the operand rows are left unused.
template <int COUT, int KC, int W, int TILES, int DIL = 1, bool GW = false, bool GATE = false, bool H16 = false>
__global__ void __launch_bounds__(TcgCfg<COUT, KC, W, TILES, DIL, GW>::THREADS, 1) conv3d_tcg_kernel(const TcgParams p) {
  using C = TcgCfg<COUT, KC, W, TILES, DIL, GW>;
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
  float* xchg = reinterpret_cast<float*>(smem + C::BAR_OFF + 1024);   // [2][4 quadrants][2 sides][DIL columns][32]
  float* s_scale = xchg + 2 * 4 * 2 * DIL * 32;
  float* s_shift = s_scale + COUT;
  float* zeros = s_shift + COUT;
  float* tpose = zeros + COUT;                      // [4 warps][32][TP_STRIDE] transpose tiles of the epilogue

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nchunk = p.Cin / KC;
  const int Wp = GW ? p.Wr : W;                     // image width = row pitch in voxels
  const int YS = (W < 32 && p.ystride) ? p.ystride : COUT;   // (compile-time COUT in the wide instantiations: slices exist at W' = 16 only)      // channel stride of the channels-last output / residual / gate
  const int ctiles = GW ? p.ctiles : 1;             // work item = (b, d, row block, column tile), column tile fastest

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
    const uint32_t idesc = idesc_f16(128, C::NPER);
    const uint64_t dbase = (KC == 32) ? desc_sw128_base() : desc_sw64_base();
    const uint32_t b16 = (smem_u32(b_buf) & 0x3FFFF) >> 4;
    uint32_t unitc = 0, phc = 0, itc = 0;
    for (int it = blockIdx.x; it < p.items; it += gridDim.x, ++itc) {
      const int hb = (it / ctiles) % p.hblocks;
      const int d = (it / (ctiles * p.hblocks)) % p.D;
      const int ntiles = min(TILES, (p.H - hb * C::HBLK + C::R - 1) / C::R);
      const int last_kd = (d + 1 < p.D) ? 2 : 1;
      uint32_t started = 0;
      for (int kd = 0; kd < 3; ++kd) {
        const int din = d + kd - 1;
        if (din < 0 || din >= p.D) continue;
        for (int ch = 0; ch < nchunk; ++ch, ++phc) {
          const bool last_phase = (kd == last_kd) && (ch == nchunk - 1);
#pragma unroll
          for (int s = C::S_FIRST; s <= C::S_LAST; ++s) {
            if (!C::used(s)) continue;
            const uint32_t slot = unitc % C::STAGES, par = (unitc / C::STAGES) & 1;
            mbar_wait(&a_ready[slot], par);
#pragma unroll
            for (int kh = 0; kh < 3; ++kh)
              if (C::tile_of(s, kh) == 0) mbar_wait(&b_full[(phc & 1) * 3 + kh], (phc >> 1) & 1);   // first needed by the unit feeding tile 0
            tc_fence_after();
            const uint64_t da0 = dbase | (uint64_t)((smem_u32(a_buf + slot * C::UNIT_BYTES) & 0x3FFFF) >> 4);
#pragma unroll
            for (int kh = 0; kh < 3; ++kh) {
              const int t = C::tile_of(s, kh);
              if (t < 0) continue;
              const uint32_t accum = (started >> t) & 1;
              if (!accum) {                             // hand-shake taken for unused tiles too (parity must not alias)
                mbar_wait(&acc_empty[t], (itc & 1) ^ 1);
                tc_fence_after();
                started |= 1u << t;
              }
              if (t < ntiles) {
                if (elect_one()) {
#pragma unroll
                  for (int mm = 0; mm < C::NMMA; ++mm) {
                    const uint32_t acc = tmem + t * C::N3 + mm * C::NPER;
                    const uint64_t db0 = dbase | (uint64_t)(b16 + (((phc & 1) * 3 + kh) * C::B_SLICE + mm * C::NPER * C::ROWB) / 16);
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
                }
                __syncwarp();
              }
              if (t == TILES - 1 && elect_one()) mma_commit(&b_empty[(phc & 1) * 3 + kh]);   // last user of slice kh in this phase
            }
            if (elect_one()) {
              mma_commit(&a_empty[slot]);
              const int tdone = C::tile_of(s, 2);       // kh = 2 is the last tap a tile receives in a phase
              if (last_phase && tdone >= 0) mma_commit(&acc_full[tdone]);
            }
            __syncwarp();
            ++unitc;
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
      // General widths: col0 = image column of load 0 (may be -HALO .. or beyond Wr: those columns are zero padding).
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
      const int d = (it / (ctiles * p.hblocks)) % p.D;
      const int b = it / (ctiles * p.hblocks * p.D);
      const int h0 = hb * C::HBLK;
      const int col0 = ct * C::CSTEP - C::HALO + v0;   // image column of this lane's first load (whole-row kernels: v0)
      for (int kd = 0; kd < 3; ++kd) {
        const int din = d + kd - 1;
        if (din < 0 || din >= p.D) continue;
        const typename A::T* plane = reinterpret_cast<const typename A::T*>(p.x) + ((size_t)b * p.D + din) * p.H * (size_t)Wp * p.Cin;
        for (int ch = 0; ch < nchunk; ++ch) {
#pragma unroll 1
          for (int j = first; j < C::NU; j += C::NLW) {
            // unit = R consecutive image rows starting at h0 + s: operand row v is voxel (h0 + s) * W + v of the plane
            const int s = C::unit_s(j);
            const typename A::T* base = plane + ((ptrdiff_t)(h0 + s) * Wp + col0) * p.Cin + ch * KC + c * 4;
            fill(base, (size_t)Wp * p.Cin, (size_t)p.Cin, h0 + s, 1, ubase + j, col0);
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
    const bool has_right_q = (((q + 1) * 32) % W) != 0;
    uint32_t itc = 0, exc = 0;
    float yamax = 0.f;                               // H16: largest stored magnitude (fp16 saturation at 65504)
    for (int it = blockIdx.x; it < p.items; it += gridDim.x, ++itc) {
      const int ct = it % ctiles;
      const int hb = (it / ctiles) % p.hblocks;
      const int d = (it / (ctiles * p.hblocks)) % p.D;
      const int b = it / (ctiles * p.hblocks * p.D);
      const int h0 = hb * C::HBLK;
      const int ntiles = min(TILES, (p.H - h0 + C::R - 1) / C::R);
      // general widths: image column of this thread's tile column; halo columns and columns beyond the image are not stored
      const int col = GW ? ct * C::CSTEP - C::HALO + m : wcol;
      const bool cvalid = !GW || (m >= C::HALO && m < 128 - C::HALO && col < Wp);
      const uint32_t vmask = GW ? __ballot_sync(0xffffffffu, cvalid) : 0xffffffffu;
      const float corr = 1.f + p.kappa * (float)(((d > 0) + 1 + (d + 1 < p.D)) * nchunk * 3 * C::KSTEPS * A::TERMS);   // tc_common.cuh: rz_kappa
      for (int t = 0; t < ntiles; ++t) {
        const int h = h0 + t * C::R + rr;
        const bool live = h < p.H;
        const ptrdiff_t vox = (((ptrdiff_t)b * p.D + d) * p.H + h) * Wp + col;     // NDHWC voxel index
        if (live && cvalid && p.residual && p.res_ndhwc) {
          // the residual streams from HBM / L2: start pulling this thread's voxel into L2 while the tile is still being accumulated
          // (ncu source view of the backbone layers: 9 % of the samples waited on the residual loads after the transpose)
          const float* rp = p.residual + vox * YS;
#pragma unroll
          for (int k = 0; k < COUT; k += 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(rp + k));
        }
        mbar_wait_relaxed(&acc_full[t], itc & 1);
        tc_fence_after();
        const size_t plane = (size_t)p.D * p.H * Wp;                               // NCDHW channel stride
        const ptrdiff_t ncdhw0 = (ptrdiff_t)b * COUT * plane + ((ptrdiff_t)d * p.H + h) * Wp + col;
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
          float* xb = xchg + (exc & 1) * (4 * 2 * DIL * 32);
          ++exc;
          if (lane >= 32 - DIL) {                     // the next quadrant's first DIL columns need these P0 values
#pragma unroll
            for (int i = 0; i < 32; ++i) xb[((q * 2) * DIL + lane - (32 - DIL)) * 32 + i] = __uint_as_float(raw[0][i]);
          }
          if (lane < DIL) {                           // the previous quadrant's last DIL columns need these P2 values
#pragma unroll
            for (int i = 0; i < 32; ++i) xb[((q * 2 + 1) * DIL + lane) * 32 + i] = __uint_as_float(raw[2][i]);
          }
          named_bar_sync(1, 128);
          const float* xl = has_left_q ? xb + (((q - 1) * 2) * DIL + (lane < DIL ? lane : 0)) * 32 : zeros;
          const float* xr = has_right_q ? xb + (((q + 1) * 2 + 1) * DIL + (lane >= 32 - DIL ? lane - (32 - DIL) : 0)) * 32 : zeros;
          float out[32];
#pragma unroll
          for (int i0 = 0; i0 < 32; i0 += 4) {        // neighbour values loaded unconditionally, merged with selects (no branches)
            const float4 l4 = *reinterpret_cast<const float4*>(xl + i0);
            const float4 r4 = *reinterpret_cast<const float4*>(xr + i0);
            const float le[4] = {l4.x, l4.y, l4.z, l4.w}, re[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int i = i0 + k;
              float left = __shfl_up_sync(0xffffffffu, __uint_as_float(raw[0][i]), DIL);
              float right = __shfl_down_sync(0xffffffffu, __uint_as_float(raw[2][i]), DIL);
              left = (lane < DIL) ? le[k] : left;       // column w-DIL (zero at the image edge)
              right = (lane >= 32 - DIL) ? re[k] : right;   // column w+DIL
              if (W < 32) {                             // several image rows per warp: row seams inside the warp are image edges
                left = (wcol < DIL) ? 0.f : left;
                right = (wcol >= W - DIL) ? 0.f : right;
              }
              out[i] = ((left + __uint_as_float(raw[1][i])) + right) * corr;
            }
          }
          // voxels of this warp that exist (W < 32: the warp spans two image rows, the second may lie below the image)
          const uint32_t vm = (W < 32) ? __ballot_sync(0xffffffffu, live) : (live ? vmask : 0u);
          if (H16 && vm) {                             // channels-last fp16 output, no residual (checked at the entry point)
            const ptrdiff_t gvox = GATE ? ((ptrdiff_t)b * p.H + h) * Wp + col - lane : 0;
            store_ndhwc_chunk32(tpose + q * TP_WARP_FLOATS, lane, out, reinterpret_cast<__half*>(p.y) + (vox - lane) * YS + cg, nullptr, YS,
                                s_scale + cg, s_shift + cg, p.act, vm, (GATE && p.gate) ? p.gate + gvox * YS + cg : nullptr, &yamax);
          } else if (!H16 && vm && p.out_ndhwc && (!p.residual || p.res_ndhwc)) {     // coalesced channels-last path (BN/residual/act inside)
            const ptrdiff_t gvox = GATE ? ((ptrdiff_t)b * p.H + h) * Wp + col - lane : 0;   // (B, H, W) index of lane 0's voxel
            store_ndhwc_chunk32(tpose + q * TP_WARP_FLOATS, lane, out, p.y + (vox - lane) * YS + cg,
                                p.residual ? p.residual + (vox - lane) * YS + cg : nullptr, YS, s_scale + cg, s_shift + cg, p.act,
                                vm, (GATE && p.gate) ? p.gate + gvox * YS + cg : nullptr);
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
        const int d = (it / (ctiles * p.hblocks)) % p.D;
        for (int kd = 0; kd < 3; ++kd) {
          const int din = d + kd - 1;
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

template <int COUT, int KC, int W, int TILES, int DIL = 1, bool GW = false, bool GATE = false, bool H16 = false>
static int launch_tcg(TcgParams& p, cudaStream_t stream) {
  using C = TcgCfg<COUT, KC, W, TILES, DIL, GW>;
  auto kernel = conv3d_tcg_kernel<COUT, KC, W, TILES, DIL, GW, GATE, H16>;
  if (!GATE && p.gate) {
    set_error("conv3d_tcg: no gated instantiation for Cout=%d W=%d", COUT, W);
    return OSB_EUNSUPPORTED;
  }
  if (W >= 32 && p.ystride && p.ystride != COUT) {
    set_error("conv3d_tcg: channel slices are instantiated for W = 16 only");
    return OSB_EUNSUPPORTED;
  }
  static PerDeviceFlag configured;
  if (!configured.here()) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM);
    if (e != cudaSuccess) {
      set_error("conv3d_tcg: cannot reserve %zu bytes of shared memory: %s", C::SMEM, cudaGetErrorString(e));
      return OSB_ECUDA;
    }
    configured.here() = true;
  }
  p.hblocks = (p.H + C::HBLK - 1) / C::HBLK;
  if (GW) p.ctiles = (p.Wr + C::CSTEP - 1) / C::CSTEP;
  else p.Wr = W, p.ctiles = 1;
  const long long items = (long long)p.B * p.D * p.hblocks * p.ctiles;
  OSB_REQUIRE(items < (1ll << 31), "conv3d_tcg: too many work items");
  p.items = (int)items;
  const int sms = sm_count();
  const int grid = p.items < sms ? p.items : sms;
  kernel<<<grid, C::THREADS, C::SMEM, stream>>>(p);
  count_launch();
  cudaError_t le = cudaGetLastError();
  if (le != cudaSuccess) {
    cudaFuncAttributes fa{};
    (void)cudaFuncGetAttributes(&fa, kernel);
    set_error("conv3d_tcg_kernel<%d,%d,%d,%d>: launch failed: %s (threads %d, kernel maxThreadsPerBlock %d, regs %d, static smem %zu, "
              "dynamic smem %zu, max dynamic %d)", COUT, KC, W, TILES, cudaGetErrorString(le), C::THREADS, fa.maxThreadsPerBlock,
              fa.numRegs, fa.sharedSizeBytes, C::SMEM, fa.maxDynamicSharedSizeBytes);
    return OSB_ECUDA;
  }
  return OSB_OK;
}

// dispatcher used by conv3d_tc.cu's C entry point; returns -1 when the shape has no generic instantiation
int launch_tcg_dispatch(const float* x, const void* w, const float* scale, const float* shift, const float* residual, float* y,
                        int B, int Cin, int Cout, int D, int H, int W, int act, int out_ndhwc, int res_ndhwc, cudaStream_t stream,
                        const float* gate, int ystride) {
  TcgParams p{};
  p.x = x, p.w = w, p.scale = scale, p.shift = shift, p.residual = residual, p.y = y, p.gate = gate;
  p.ystride = ystride;
  p.B = B, p.D = D, p.H = H, p.Cin = Cin, p.act = act, p.out_ndhwc = out_ndhwc, p.res_ndhwc = res_ndhwc;
  p.kappa = rz_kappa(), p.overflow = tc_overflow_flag();
  if (!p.overflow) return OSB_ECUDA;
  if (Cin % 16 != 0 || Cin < 16) return -1;
  if (W == 64 && Cout == 64 && gate) return launch_tcg<64, 16, 64, 2, 1, false, true>(p, stream);   // StereoBase 1/8 level (FeatureAtt gate)
  if (W == 32 && Cout == 96 && gate) return launch_tcg<96, 16, 32, 1, 1, false, true>(p, stream);   // ... 1/16 level
  if (W == 64 && Cout == 64) return launch_tcg<64, 16, 64, 2>(p, stream);
  if (W == 32 && Cout == 64) return launch_tcg<64, 16, 32, 2>(p, stream);
  if (W == 32 && Cout == 128) return launch_tcg<128, 16, 32, 1>(p, stream);
  if (W == 32 && Cout == 96) return launch_tcg<96, 16, 32, 1>(p, stream);         // StereoBase 1/16 level (4c = 96)
  if (W == 16 && Cout == 96) return launch_tcg<96, 16, 16, 1, 1, false, true>(p, stream);   // StereoBase 1/32 level: 6c = 144 -> 160 channels
  if (W == 16 && Cout == 64) return launch_tcg<64, 16, 16, 2, 1, false, true>(p, stream);   // as two slices (96 + 64), 8 image rows per tile
  if (W == 128 && Cout == 64) return launch_tcg<64, 16, 128, 2>(p, stream);      // 2D backbone stages as one-plane volumes
  if (W == 128 && Cout == 128) return launch_tcg<128, 16, 128, 1>(p, stream);
  // every other width: 128-column tiles with a one-column halo (tc_general_width() is the single source of the W bound)
  p.Wr = W;
  if (Cout == 32) return launch_tcg<32, 16, 128, 5, 1, true>(p, stream);
  if (Cout == 64) return launch_tcg<64, 16, 128, 2, 1, true>(p, stream);
  if (Cout == 128) return launch_tcg<128, 16, 128, 1, 1, true>(p, stream);
  return -1;
}

// fp16 activations (H16 instantiations): the whole-row shapes of StereoBase's hourglass at W' = 128 -- 1/8 level (W = 64, Cout = 64),
// 1/16 level (W = 32, Cout = 96), 1/32 level channel slices (W = 16, Cout = 96 | 64); channels-last in and out, no residual.
bool tcg_h16_shape(int Cin, int Cout, int W) {
  return Cin % 16 == 0 && Cin >= 16 && ((W == 64 && Cout == 64) || (W == 32 && Cout == 96) || (W == 16 && (Cout == 96 || Cout == 64)));
}

int launch_tcg_h16(const void* x, const void* w, const float* scale, const float* shift, const float* gate, float* y, int B, int Cin,
                   int Cout, int D, int H, int W, int act, int ystride, cudaStream_t stream) {
  TcgParams p{};
  p.x = static_cast<const float*>(x), p.w = w, p.scale = scale, p.shift = shift, p.gate = gate, p.y = y;
  p.ystride = ystride;
  p.B = B, p.D = D, p.H = H, p.Cin = Cin, p.act = act, p.out_ndhwc = 1, p.res_ndhwc = 1;
  p.kappa = rz_kappa(), p.overflow = tc_overflow_flag();
  if (!p.overflow) return OSB_ECUDA;
  if (W == 64) return gate ? launch_tcg<64, 16, 64, 2, 1, false, true, true>(p, stream) : launch_tcg<64, 16, 64, 2, 1, false, false, true>(p, stream);
  if (W == 32) return gate ? launch_tcg<96, 16, 32, 1, 1, false, true, true>(p, stream) : launch_tcg<96, 16, 32, 1, 1, false, false, true>(p, stream);
  if (Cout == 96) return launch_tcg<96, 16, 16, 1, 1, false, true, true>(p, stream);
  return launch_tcg<64, 16, 16, 2, 1, false, true, true>(p, stream);
}

// dilated (2) one-plane variant for the 2D backbone: same parameters with D == 1
int launch_tcg_dilated2(const float* x, const void* w, const float* scale, const float* shift, const float* residual, float* y,
                        int B, int Cin, int Cout, int H, int W, int act, int out_ndhwc, int res_ndhwc, cudaStream_t stream) {
  TcgParams p{};
  p.x = x, p.w = w, p.scale = scale, p.shift = shift, p.residual = residual, p.y = y;
  p.B = B, p.D = 1, p.H = H, p.Cin = Cin, p.act = act, p.out_ndhwc = out_ndhwc, p.res_ndhwc = res_ndhwc;
  p.kappa = rz_kappa(), p.overflow = tc_overflow_flag();
  if (!p.overflow) return OSB_ECUDA;
  if (Cin % 16 != 0 || Cin < 16) return -1;
  if (W == 128 && Cout == 128) return launch_tcg<128, 16, 128, 1, 2>(p, stream);
  return -1;
}

}  // namespace osb
