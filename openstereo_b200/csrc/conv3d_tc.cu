// Tensor-core (tcgen05 / TMEM) implicit-GEMM Conv3d 3x3x3, stride 1, pad 1, for the full-resolution layers of the
// hourglass aggregation (W = 128 output columns = one UMMA M tile).  fp32-accurate through 3xFP16 operand splitting
// (tc_common.cuh):   a*b ~= a_lo*b_hi + a_hi*b_lo + a_hi*b_hi   on tcgen05.mma.kind::f16, fp32 accumulation in TMEM.
// Activations are split while they are staged (fp32 in HBM -> [hi | lo] fp16 rows in shared memory); weights are split
// and pre-scaled once on the host.  Plain TF32 / BF16 / FP16 operands break the north star's 1e-3 px EPE bar
// (SURVEY.md section 4.3: 2.2e-2 px for TF32); the split keeps it (tests/test_zz_fullsize_gpu.py).
//
// Replaces the same reference modules as conv3d.cu (convbn_3d + ReLU of gwcnet/hourglass.py:5-16,
// gwcnet_disp_processor.py:40-81; conv3d_bn(_relu) psmnet/submodule.py:68-83,160-177) for layers with W == 128.
//
// GEMM mapping.  Activations are channels-last (B, D, H, W, Cin): an A tile is "the 128 voxels of one image row x 32
// input channels", K-major with 128-byte rows in the canonical SWIZZLE_128B layout.
//   * the three kw taps are NOT realised by shifting A (that would need halo columns and unaligned tiles); instead the
//     three weight slices are stacked along N -- one MMA of N = 3*Cout produces P_kw[m] = A[m] . B_kw for kw = 0,1,2 --
//     and the epilogue forms D[m] = P_0[m-1] + P_1[m] + P_2[m+1] with warp shuffles (zero padding at m = -1 / 128 is
//     implicit because a row tile spans the whole image width).  N = 96 also lifts the MMA above the ~55-cycle floor
//     that small-N tf32 MMAs hit (tools/tc_probe.cu: N=32, 64 and 96 all take 54-56 cycles).
//   * kh taps: output row t of the block needs input rows t-1, t, t+1: input rows stream through a shared-memory ring
//     and each staged row feeds up to three accumulator tiles.
//   * an operand row is 128 bytes = [32 channels hi | 32 channels lo] fp16, SWIZZLE_128B; a K = 16 MMA step is 32 bytes, so
//     the hi k-steps sit at descriptor offsets +0, +2 and the lo ones at +4, +6 (16-byte units) of the SAME tile.
//   * kd taps and 32-channel Cin chunks are phases of one work item; the three kh weight slices of a phase are
//     refilled just in time (slice kh is free after row 4+kh of a phase and needed again at row kh of the next one).
// Work item = (image b, output plane d, block of 5 output rows); 5 accumulator tiles x 96 columns = 480 TMEM columns.
//
// Operand staging.  A first version fed the ring with TMA (cp.async.bulk.tensor, SWIZZLE_64B boxes of 64-byte rows;
// kept as profiles/r1_conv3d_tc_tma_variant.cu.txt): correct, but ncu showed the TMA unit request-rate bound (~9 cycles
// per 64-byte row, 7 B/clk/SM) and the tensor pipe only 34 % busy (profiles/r1_ncu_summary.md) -- and fp32 data needs
// the split anyway.  Here the loader warps read coalesced float4 from global/L2, convert to the hi/lo fp16 pair, write
// both halves of the row with the 128-byte swizzle applied by hand (two conflict-free STS.64) and publish the tile to the
// tensor core through fence.proxy.async + mbarrier; arbitrary gathers (stride 2, multi-row tiles) come for free.
//
// Warp roles (352 threads, 1 CTA/SM, persistent): warp 0 = MMA issuer (+ TMEM allocator), warps 1-4 = A-row loaders,
// warps 5-8 = epilogue (TMEM -> registers -> BN/residual/ReLU -> global), warp 9 = weight-slice producer (one elected lane issuing
// 1-D TMA bulk copies of the pre-swizzled slices into two buffer sets), warp 10 idle.
#include <cstdlib>

#include "tc_common.cuh"

namespace osb {

constexpr int TC_W = 128;          // image width handled (UMMA M)
constexpr int TC_KC = 32;          // input channels per phase: 128-byte K-major rows [32 hi | 32 lo] fp16, SWIZZLE_128B
constexpr int TC_TILES = 5;        // output rows (accumulator tiles) per work item
constexpr int TC_ROWS = TC_TILES + 2;
constexpr int TC_STAGES = 4;       // A-row ring depth (converted fp16 hi|lo tiles)
constexpr int TC_RAW = 4;          // raw fp32 rows staged by 1-D TMA bulk copies ahead of the converters (Cin = 32 channels-last layers)
constexpr int TC_ROW_BYTES = TC_W * TC_KC * 4;     // 16384: one staged input row (hi and lo halves of every voxel)
constexpr int TC_THREADS = 352;

struct TcParams {
  const float* x;          // (B, D, H, W, Cin) channels-last
  const void* w;           // fp16 [3 kd][Cin/32][3 kh][3*Cout][32 hi | 32 lo]  (ops.pack_tc_weight)
  const float* scale;
  const float* shift;
  const float* residual;
  float* y;
  int B, D, H, Cin, Cout;
  int act;
  float kappa;       // expected round-towards-zero loss per accumulating MMA (tc_common.cuh)
  unsigned int* overflow;  // sticky fp16-range flag (tc_common.cuh)
  int out_ndhwc, res_ndhwc;
  int bulk_rows;     // input rows staged by TMA bulk copies, TC_RAW deep: Cin == 32 channels-last (one 16 KB copy per row) or NCDHW
                     // (32 copies of 512 bytes, one per channel plane)
  int in_ncdhw;      // the INPUT is (B, Cin, D, H, W): the first aggregation layer reads the cost volume as the volume kernel wrote it
  int items, hblocks;
};

template <int COUT>
__global__ void __launch_bounds__(TC_THREADS, 1) conv3d_tc_kernel(const TcParams p) {
  constexpr int N3 = 3 * COUT;                      // kw-stacked MMA N
  constexpr int B_SLICE = N3 * TC_KC * 4;           // one kh weight slice, rows [hi | lo] (12288 B for Cout = 32)
  static_assert(B_SLICE % 1024 == 0, "weight slices must stay 1024-byte aligned");
  static_assert(TC_TILES * N3 <= 512, "accumulators exceed TMEM");
  constexpr int A_OFF = 0;
  constexpr int B_OFF = A_OFF + TC_STAGES * TC_ROW_BYTES;      // [3 kh]
  constexpr int RAW_OFF = B_OFF + TC_BSLOTS * 3 * B_SLICE;    // [TC_RAW] raw fp32 input rows
  constexpr int BAR_OFF = RAW_OFF + TC_RAW * TC_ROW_BYTES;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* a_buf = smem + A_OFF;
  uint8_t* b_buf = smem + B_OFF;
  uint8_t* raw_buf = smem + RAW_OFF;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + BAR_OFF);
  uint64_t* a_ready = bars;                         // [STAGES] loaders -> MMA        (128 arrivals)
  uint64_t* a_empty = a_ready + TC_STAGES;          // [STAGES] MMA -> loaders        (tcgen05.commit)
  uint64_t* b_full = a_empty + TC_STAGES;           // [2][3]   weight producer -> MMA (expect_tx + TMA bytes)
  uint64_t* b_empty = b_full + TC_BSLOTS * 3;       // [2][3]   MMA -> weight producer (tcgen05.commit)
  uint64_t* acc_full = b_empty + TC_BSLOTS * 3;     // [TILES]  MMA -> epilogue, one per accumulator tile
  uint64_t* acc_empty = acc_full + TC_TILES;        // [TILES]  epilogue -> MMA       (128 arrivals)
  uint64_t* raw_full = acc_empty + TC_TILES;        // [RAW]    row producer -> converters (expect_tx + TMA bytes, or a plain arrive)
  uint64_t* raw_empty = raw_full + TC_RAW;          // [RAW]    converters -> row producer (128 arrivals)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(raw_empty + TC_RAW);
  float* xchg = reinterpret_cast<float*>(tmem_slot + 4);   // 16-byte aligned
  //   // [2 tile parities][4 warps][2][COUT] boundary exchange
  float* s_scale = xchg + 2 * 4 * 2 * COUT;                // [COUT]
  float* s_shift = s_scale + COUT;
  float* zeros = s_shift + COUT;                           // [COUT] of 0.f (image-edge neighbours)
  float* tpose = zeros + COUT;                      // [4 warps][32][TP_STRIDE] transpose tiles of the epilogue

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nchunk = p.Cin / TC_KC;

  if (threadIdx.x == 0) {
    for (int s = 0; s < TC_STAGES; ++s) {
      mbar_init(&a_ready[s], 128);
      mbar_init(&a_empty[s], 1);
    }
    for (int k = 0; k < TC_BSLOTS * 3; ++k) {
      mbar_init(&b_full[k], 1);
      mbar_init(&b_empty[k], 1);
    }
    for (int t = 0; t < TC_TILES; ++t) {
      mbar_init(&acc_full[t], 1);
      mbar_init(&acc_empty[t], 128);
    }
    for (int k = 0; k < TC_RAW; ++k) {
      mbar_init(&raw_full[k], 1);
      mbar_init(&raw_empty[k], 128);
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
  // The rows a CTA stages form one flat sequence (item, kd, chunk, r).  `RowIter` walks it; loads run TWO rows ahead of
  // the stores (software pipeline in registers) so that a full L2/HBM round trip is always in flight.
  struct RowIter {
    int it, kd, ch, r;
  };
  auto advance = [&](RowIter& s) {                  // -> false when the sequence is exhausted
    for (;;) {
      if (s.it >= p.items) return false;
      if (++s.r < TC_ROWS) return true;
      s.r = -1;
      if (++s.ch < nchunk) continue;
      s.ch = 0;
      const int d = (s.it / p.hblocks) % p.D;
      for (++s.kd; s.kd < 3; ++s.kd) {
        const int din = d + s.kd - 1;
        if (din >= 0 && din < p.D) break;
      }
      if (s.kd < 3) continue;
      s.it += gridDim.x;
      if (s.it >= p.items) return false;
      const int d2 = (s.it / p.hblocks) % p.D;
      s.kd = (d2 == 0) ? 1 : 0;                     // first input plane that exists
    }
  };
  const uint32_t tmem = *tmem_slot;

  // ---------------------------------------------------------------------------------------------- MMA issuer
  if (warp == 0) {
    {
      const uint32_t idesc = idesc_f16(128, N3);
      constexpr uint32_t LO = TcK<TC_KC>::LO_OFF;     // descriptor offset of the lo half of an operand row
      const uint64_t dbase = desc_sw128_base();
      // Descriptors differ only in their 14-bit start-address field (bits 0-13, units of 16 bytes).
      const uint32_t b16 = (smem_u32(b_buf) & 0x3FFFF) >> 4;
      uint32_t rowc = 0, phc = 0, itc = 0;
      for (int it = blockIdx.x; it < p.items; it += gridDim.x, ++itc) {
        const int hb = it % p.hblocks;
        const int d = (it / p.hblocks) % p.D;
        const int ntiles = min(TC_TILES, p.H - hb * TC_TILES);
        const int last_kd = (d + 1 < p.D) ? 2 : 1;    // last input plane that exists for this output plane
        uint32_t started = 0;
        for (int kd = 0; kd < 3; ++kd) {
          const int din = d + kd - 1;
          if (din < 0 || din >= p.D) continue;
          for (int ch = 0; ch < nchunk; ++ch, ++phc) {
            const bool last_phase = (kd == last_kd) && (ch == nchunk - 1);
#pragma unroll
            for (int r = 0; r < TC_ROWS; ++r) {
              const uint32_t s = rowc % TC_STAGES, par = (rowc / TC_STAGES) & 1;
              mbar_wait(&a_ready[s], par);
              const uint32_t bslot = (phc & 1) * 3;           // weight buffers alternate between phases
              if (r < 3) mbar_wait(&b_full[bslot + r], (phc >> 1) & 1);   // slice kh = r is first needed by row r (tile 0)
              tc_fence_after();
              const uint64_t da0 = dbase | (uint64_t)((smem_u32(a_buf + s * TC_ROW_BYTES) & 0x3FFFF) >> 4);
#pragma unroll
              for (int kh = 0; kh < 3; ++kh) {
                const int t = r - kh;                 // output row tile fed by input row r through tap kh (compile time)
                if (t < 0 || t >= TC_TILES) continue;
                const uint32_t accum = (started >> t) & 1;
                if (!accum) {                         // first touch of this tile in this item: the previous item's epilogue
                  mbar_wait(&acc_empty[t], (itc & 1) ^ 1);     // must have drained it.  Taken for UNUSED tiles too: otherwise
                  tc_fence_after();                            // acc_full[t] could complete twice before the epilogue looks
                  started |= 1u << t;                          // and the mbarrier parity would alias (deadlock).
                }
                if (t < ntiles) {
                  const uint32_t acc = tmem + t * N3;
                  const uint64_t db0 = dbase | (uint64_t)(b16 + (bslot + kh) * (B_SLICE / 16));
                  if (elect_one()) {
#pragma unroll
                    for (int ks = 0; ks < TcK<TC_KC>::KSTEPS; ++ks) {
                      mma_f16(acc, da0 + LO + 2 * ks, db0 + 2 * ks, idesc, ks > 0 ? 1u : accum);   // small terms first
                      mma_f16(acc, da0 + 2 * ks, db0 + LO + 2 * ks, idesc, 1);
                      mma_f16(acc, da0 + 2 * ks, db0 + 2 * ks, idesc, 1);
                    }
                  }
                  __syncwarp();
                }
                if (t == TC_TILES - 1 && elect_one()) mma_commit(&b_empty[bslot + kh]);   // row 4+kh: last user of slice kh
              }
              if (elect_one()) {
                mma_commit(&a_empty[s]);              // ring slot reusable once these MMAs have read it
                if (last_phase && r >= 2) mma_commit(&acc_full[r - 2]);   // tile r-2 has received its last tap
              }
              __syncwarp();
              ++rowc;
            }
          }
        }
      }
    }
  }
  // ---------------------------------------------------------------------------------------------- A-row loaders
  else if (warp < 5) {
    const int lt = threadIdx.x - 32;                 // 0..127
    const int vsel = lt >> 3, c16 = lt & 7;          // this thread's voxel (mod 16) and fp32 16-byte chunk of the 32-channel slice
    // voxel order inside a half-warp alternates bit 2 of the column so that the STS.64 pairs of stage_f16_split hit disjoint banks
    const int vcol = ((vsel & 1) << 2) | ((vsel >> 1) & 3) | (vsel & 8);
    float amax = 0.f;
    const size_t row_stride = (size_t)TC_W * p.Cin;  // floats per image row
    auto load_row = [&](const RowIter& s, float4 (&v)[8]) {
      const int hb = s.it % p.hblocks;
      const int d = (s.it / p.hblocks) % p.D;
      const int b = s.it / (p.hblocks * p.D);
      const int hin = hb * TC_TILES - 1 + s.r, din = d + s.kd - 1;
      if (hin >= 0 && hin < p.H && p.in_ncdhw) {
        // NCDHW input: this thread stages voxel (column) lt for all eight channel quads; every LDG.32 of a warp is one
        // contiguous 128-byte row segment of a channel plane.  v[j] holds channels 4*qj .. 4*qj+3, qj = j ^ ((lt >> 3) & 1)
        // (the swap keeps the STS.64 of lanes 8 apart -- same swizzled chunk -- on different 8-byte halves).
        const size_t plane = (size_t)p.D * p.H * TC_W;
        const float* src = p.x + (((size_t)b * p.Cin + s.ch * TC_KC) * p.D + din) * p.H * TC_W + (size_t)hin * TC_W + lt;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float* q = src + (size_t)(4 * (j ^ ((lt >> 3) & 1))) * plane;
          v[j] = make_float4(__ldg(q), __ldg(q + plane), __ldg(q + 2 * plane), __ldg(q + 3 * plane));
        }
      } else if (hin >= 0 && hin < p.H) {             // rows outside the image are the conv's zero padding
        const float* src = p.x + (((size_t)b * p.D + din) * p.H + hin) * row_stride + s.ch * TC_KC + c16 * 4;
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = __ldg(reinterpret_cast<const float4*>(src + (size_t)(vcol + 16 * j) * p.Cin));
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    uint32_t rowc = 0;
    auto store_row = [&](const float4 (&v)[8]) {
      const uint32_t s = rowc % TC_STAGES, par = (rowc / TC_STAGES) & 1;
      mbar_wait_relaxed(&a_empty[s], par ^ 1);        // the MMAs that read this slot last time have completed
      uint8_t* tile = a_buf + s * TC_ROW_BYTES;
      if (p.in_ncdhw) {
#pragma unroll
        for (int j = 0; j < 8; ++j) stage_f16_split<TC_KC>(tile, lt, j ^ ((lt >> 3) & 1), v[j], amax);
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) stage_f16_split<TC_KC>(tile, vcol + 16 * j, c16, v[j], amax);   // tile row = image column
      }
      fence_proxy_async();                            // generic-proxy writes -> visible to the tensor core (async proxy)
      mbar_arrive(&a_ready[s]);
      ++rowc;
    };
    RowIter ld{(int)blockIdx.x, 0, 0, -1};
    if (ld.it < p.items) ld.kd = (((ld.it / p.hblocks) % p.D) == 0) ? 1 : 0;
    if (p.bulk_rows) {
      // The row producer (warp 10) keeps TC_RAW rows of raw fp32 in flight with 16 KB TMA bulk copies; these four warps only
      // convert: LDS.128 (a warp reads 512 contiguous bytes) -> fp16 hi|lo -> swizzled STS.64.  No load latency on this path.
      uint32_t rawc = 0;
      while (advance(ld)) {
        const int hb = ld.it % p.hblocks;
        const int hin = hb * TC_TILES - 1 + ld.r;
        const uint32_t slot = rawc % TC_RAW, par = (rawc / TC_RAW) & 1;
        mbar_wait_relaxed(&raw_full[slot], par);
        float4 v[8];
        if (hin >= 0 && hin < p.H && p.in_ncdhw) {    // raw slot = [32 channels][128 columns]: this thread's column, 8 channel quads
          const float* src = reinterpret_cast<const float*>(raw_buf + slot * TC_ROW_BYTES) + lt;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float* q = src + 4 * (j ^ ((lt >> 3) & 1)) * TC_W;
            v[j] = make_float4(q[0], q[TC_W], q[2 * TC_W], q[3 * TC_W]);
          }
        } else if (hin >= 0 && hin < p.H) {
          const float* src = reinterpret_cast<const float*>(raw_buf + slot * TC_ROW_BYTES) + c16 * 4;
#pragma unroll
          for (int j = 0; j < 8; ++j) v[j] = *reinterpret_cast<const float4*>(src + (vcol + 16 * j) * TC_KC);
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        store_row(v);                                 // consumes v: the reads of the raw slot are complete behind it
        mbar_arrive(&raw_empty[slot]);
        ++rawc;
      }
      tc_report_overflow(p.overflow, amax);
      amax = 0.f;
    }
    float4 va[8], vb[8];
    bool has_a = !p.bulk_rows && advance(ld);
    if (has_a) load_row(ld, va);
    bool has_b = has_a && advance(ld);
    if (has_b) load_row(ld, vb);
    while (has_a) {
      store_row(va);
      has_a = has_b && advance(ld);
      if (has_a) load_row(ld, va);
      if (!has_b) break;
      store_row(vb);
      has_b = has_a && advance(ld);
      if (has_b) load_row(ld, vb);
    }
    tc_report_overflow(p.overflow, amax);
  }
  // ---------------------------------------------------------------------------------------------- epilogue
  else if (warp < 9) {
    const int q = warp & 3;                          // TMEM lane quadrant this warp may read
    const int m = q * 32 + lane;                     // voxel (image column) owned by this thread
    uint32_t itc = 0, tilec = 0;
    for (int it = blockIdx.x; it < p.items; it += gridDim.x, ++itc) {
      const int hb = it % p.hblocks;
      const int d = (it / p.hblocks) % p.D;
      const int b = it / (p.hblocks * p.D);
      const int h0 = hb * TC_TILES;
      const int ntiles = min(TC_TILES, p.H - h0);
      // MMAs each P_kw accumulator received: (existing kd planes) x chunks x 3 kh x k-steps x 3 split terms
      const float corr = 1.f + p.kappa * (float)(((d > 0) + 1 + (d + 1 < p.D)) * nchunk * 3 * TcK<TC_KC>::KSTEPS * 3);
      // D[m] = P0[m-1] + P1[m] + P2[m+1], tile by tile as the MMA warp releases them
      for (int t = 0; t < ntiles; ++t) {
        mbar_wait_relaxed(&acc_full[t], itc & 1);
        tc_fence_after();
        const int h = h0 + t;
        const size_t vox = (((size_t)b * p.D + d) * p.H + h) * TC_W + m;           // NDHWC voxel index
        const size_t plane = (size_t)p.D * p.H * TC_W;                             // NCDHW channel stride
        const size_t ncdhw0 = (size_t)b * p.Cout * plane + ((size_t)d * p.H + h) * TC_W + m;   // p.Cout <= COUT real channels
        const uint32_t trow = tmem + ((uint32_t)(q * 32) << 16) + t * N3;
        // all 3*COUT accumulator columns of this voxel in one go: loads back to back, a single wait
        uint32_t raw[3][COUT];
#pragma unroll
        for (int kw = 0; kw < 3; ++kw)
#pragma unroll
          for (int c0 = 0; c0 < COUT; c0 += 16) tmem_ld16_nowait(trow + kw * COUT + c0, &raw[kw][c0]);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(&acc_empty[t]);                   // the tile is in registers: hand it back to the MMA warp
        // lanes at the warp edges need the neighbour quadrant's values: exchange through shared memory (double-buffered
        // by tile parity so one named barrier per tile suffices)
        float* xb = xchg + (tilec & 1) * (4 * 2 * COUT);
        ++tilec;                                      // running tile count: consecutive tiles never share a buffer
        if (lane == 31) {
#pragma unroll
          for (int i = 0; i < COUT; ++i) xb[(q * 2) * COUT + i] = __uint_as_float(raw[0][i]);
        }
        if (lane == 0) {
#pragma unroll
          for (int i = 0; i < COUT; ++i) xb[(q * 2 + 1) * COUT + i] = __uint_as_float(raw[2][i]);
        }
        named_bar_sync(1, 128);
        const float* xl = (q > 0) ? xb + ((q - 1) * 2) * COUT : zeros;
        const float* xr = (q < 3) ? xb + ((q + 1) * 2 + 1) * COUT : zeros;
        float out[COUT];
        // The neighbour-quadrant values are loaded UNCONDITIONALLY (warp-uniform addresses: broadcast LDS.128) and merged with
        // selects: the `lane == 0 ? xl[i] : left` form compiled to a branch around a load per element -- 32 % of the kernel's
        // stall samples sat on it (branch_resolving; profiles/r2_step_summary.md) and the MMA warp waited for acc_empty.
#pragma unroll
        for (int i0 = 0; i0 < COUT; i0 += 4) {
          const float4 l4 = *reinterpret_cast<const float4*>(xl + i0);
          const float4 r4 = *reinterpret_cast<const float4*>(xr + i0);
          const float le[4] = {l4.x, l4.y, l4.z, l4.w}, re[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int i = i0 + k;
            float left = __shfl_up_sync(0xffffffffu, __uint_as_float(raw[0][i]), 1);
            float right = __shfl_down_sync(0xffffffffu, __uint_as_float(raw[2][i]), 1);
            left = (lane == 0) ? le[k] : left;        // m-1 lives in the previous quadrant (zero at the image edge)
            right = (lane == 31) ? re[k] : right;     // m+1 lives in the next quadrant
            out[i] = ((left + __uint_as_float(raw[1][i])) + right) * corr;
          }
        }
        if constexpr (COUT == 32) {
          if (p.out_ndhwc && (!p.residual || p.res_ndhwc)) {     // coalesced channels-last path (BN/residual/act inside)
            store_ndhwc_chunk32(tpose + q * TP_WARP_FLOATS, lane, out, p.y + (vox - lane) * COUT,
                                p.residual ? p.residual + (vox - lane) * COUT : nullptr, COUT, s_scale, s_shift, p.act);
            continue;
          }
        }
#pragma unroll
        for (int i = 0; i < COUT; ++i) out[i] = fmaf(out[i], s_scale[i], s_shift[i]);
        if (p.residual) {
          if (p.res_ndhwc) {
            const float4* rp = reinterpret_cast<const float4*>(p.residual + vox * COUT);
#pragma unroll
            for (int i = 0; i < COUT / 4; ++i) {
              const float4 rv = __ldg(rp + i);
              out[4 * i] += rv.x, out[4 * i + 1] += rv.y, out[4 * i + 2] += rv.z, out[4 * i + 3] += rv.w;
            }
          } else {
#pragma unroll
            for (int i = 0; i < COUT; ++i)
              if (i < p.Cout) out[i] += __ldg(p.residual + ncdhw0 + (size_t)i * plane);
          }
        }
        if (p.act == OSB_ACT_RELU) {
#pragma unroll
          for (int i = 0; i < COUT; ++i) out[i] = fmaxf(out[i], 0.f);
        } else if (p.act == OSB_ACT_LEAKY) {
#pragma unroll
          for (int i = 0; i < COUT; ++i) out[i] = out[i] > 0.f ? out[i] : 0.01f * out[i];
        }
        if (p.out_ndhwc) {
          float4* yp = reinterpret_cast<float4*>(p.y + vox * COUT);
#pragma unroll
          for (int i = 0; i < COUT / 4; ++i) yp[i] = make_float4(out[4 * i], out[4 * i + 1], out[4 * i + 2], out[4 * i + 3]);
        } else {
#pragma unroll
          for (int i = 0; i < COUT; ++i)
            if (i < p.Cout) p.y[ncdhw0 + (size_t)i * plane] = out[i];                 // 128-byte rows per warp
        }
      }
      // tiles this (short) block never used still take part in the hand-shake so barrier phases stay in step
      for (int t = ntiles; t < TC_TILES; ++t) {
        mbar_wait(&acc_full[t], itc & 1);
        mbar_arrive(&acc_empty[t]);
      }
    }
  }
  // ---------------------------------------------------------------------------------------------- weight-slice producer
  // One elected lane streams the pre-swizzled (kd, chunk, kh) slices with 1-D TMA bulk copies into the two buffer sets; it runs up
  // to a whole phase ahead of the MMAs (the other 63 threads of warps 9-10 idle: the slot they used to fill by LDG/STS is gone).
  else if (warp == 9) {
    if (elect_one()) {
      const uint8_t* wsrc = reinterpret_cast<const uint8_t*>(p.w);
      uint32_t phc = 0;
      for (int it = blockIdx.x; it < p.items; it += gridDim.x) {
        const int d = (it / p.hblocks) % p.D;
        for (int kd = 0; kd < 3; ++kd) {
          const int din = d + kd - 1;
          if (din < 0 || din >= p.D) continue;
          for (int ch = 0; ch < nchunk; ++ch, ++phc) {
            for (int kh = 0; kh < 3; ++kh) {
              const uint32_t slot = (phc & 1) * 3 + kh;
              const size_t slice = ((size_t)kd * nchunk + ch) * 3 + kh;
              mbar_wait_relaxed(&b_empty[slot], ((phc >> 1) & 1) ^ 1);   // the MMAs that read this buffer two phases ago are done
              mbar_arrive_expect_tx(&b_full[slot], B_SLICE);
              bulk_g2s(b_buf + slot * B_SLICE, wsrc + slice * B_SLICE, B_SLICE, &b_full[slot]);
            }
          }
        }
      }
    }
    __syncwarp();
  }
  // ---------------------------------------------------------------------------------------------- raw-row producer
  else if (warp == 10 && p.bulk_rows) {
    if (elect_one()) {
      RowIter ld{(int)blockIdx.x, 0, 0, -1};
      if (ld.it < p.items) ld.kd = (((ld.it / p.hblocks) % p.D) == 0) ? 1 : 0;
      uint32_t rawc = 0;
      while (advance(ld)) {
        const int hb = ld.it % p.hblocks;
        const int d = (ld.it / p.hblocks) % p.D;
        const int b = ld.it / (p.hblocks * p.D);
        const int hin = hb * TC_TILES - 1 + ld.r, din = d + ld.kd - 1;
        const uint32_t slot = rawc % TC_RAW, par = (rawc / TC_RAW) & 1;
        mbar_wait_relaxed(&raw_empty[slot], par ^ 1);
        if (hin >= 0 && hin < p.H && p.in_ncdhw) {      // NCDHW: 32 channel planes, each contributes one 512-byte image row
          const size_t plane = (size_t)p.D * p.H * TC_W;
          const float* src = p.x + (((size_t)b * p.Cin + ld.ch * TC_KC) * p.D + din) * p.H * TC_W + (size_t)hin * TC_W;
          mbar_arrive_expect_tx(&raw_full[slot], TC_ROW_BYTES);
          for (int c = 0; c < TC_KC; ++c)
            bulk_g2s(raw_buf + slot * TC_ROW_BYTES + c * (TC_W * 4), src + c * plane, TC_W * 4, &raw_full[slot]);
        } else if (hin >= 0 && hin < p.H) {             // one image row = 128 voxels x 32 channels x 4 B, contiguous
          const float* src = p.x + (((size_t)b * p.D + din) * p.H + hin) * (size_t)(TC_W * TC_KC);
          mbar_arrive_expect_tx(&raw_full[slot], TC_ROW_BYTES);
          bulk_g2s(raw_buf + slot * TC_ROW_BYTES, src, TC_ROW_BYTES, &raw_full[slot]);
        } else {
          mbar_arrive(&raw_full[slot]);                 // zero-padding row: nothing to copy, the converters write zeros
        }
        ++rawc;
      }
    }
    __syncwarp();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
}

// ---------------------------------------------------------------------------------------- layout conversion kernels
// NCDHW -> NDHWC through a 32x32 shared-memory transpose (both sides coalesced).
template <typename T = float>       // float, or __half for the fp16 route (osb_ncdhw_to_ndhwc_pad_h16)
__global__ void __launch_bounds__(256) ncdhw_to_ndhwc_kernel(const T* __restrict__ x, T* __restrict__ y, int C, int Cp,
                                                             size_t vol) {
  __shared__ T tile[32][33];
  const int b = blockIdx.z;
  const size_t v0 = (size_t)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;       // 32 x 8
  for (int i = ty; i < 32; i += 8) {
    const int c = c0 + i;
    const size_t v = v0 + tx;
    tile[i][tx] = (c < C && v < vol) ? __ldg(x + ((size_t)b * C + c) * vol + v) : T(0.f);
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const size_t v = v0 + i;
    const int c = c0 + tx;
    if (c < Cp && v < vol) y[((size_t)b * vol + v) * Cp + c] = tile[tx][i];      // channels C .. Cp-1: zero padding
  }
}

template <int COUT>
static int launch_tc(const TcParams& p, cudaStream_t stream) {
  constexpr int N3 = 3 * COUT;
  const size_t smem = 1024 + (size_t)(TC_STAGES + TC_RAW) * TC_ROW_BYTES + TC_BSLOTS * 3 * (size_t)(N3 * TC_KC * 4) + 512 + 2 * 4 * 2 * COUT * 4 +
                      3 * COUT * 4 + TP_BYTES;
  auto kernel = conv3d_tc_kernel<COUT>;
  static PerDeviceFlag configured;
  if (!configured.here()) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      set_error("conv3d_tc: cannot reserve %zu bytes of shared memory: %s", smem, cudaGetErrorString(e));
      return OSB_ECUDA;
    }
    configured.here() = true;
  }
  const int sms = sm_count();
  const int grid = p.items < sms ? p.items : sms;   // persistent: one CTA per SM (it owns all 512 TMEM columns)
  kernel<<<grid, TC_THREADS, smem, stream>>>(p);
  count_launch();
  return check_launch("conv3d_tc_kernel");
}

int launch_tcg_dispatch(const float* x, const void* w, const float* scale, const float* shift, const float* residual, float* y,
                        int B, int Cin, int Cout, int D, int H, int W, int act, int out_ndhwc, int res_ndhwc, cudaStream_t stream,
                        const float* gate = nullptr, int ystride = 0);
int launch_tcg_dilated2(const float* x, const void* w, const float* scale, const float* shift, const float* residual, float* y,
                        int B, int Cin, int Cout, int H, int W, int act, int out_ndhwc, int res_ndhwc, cudaStream_t stream);
bool tcg_h16_shape(int Cin, int Cout, int W);
int launch_tcg_h16(const void* x, const void* w, const float* scale, const float* shift, const float* gate, float* y, int B, int Cin,
                   int Cout, int D, int H, int W, int act, int ystride, cudaStream_t stream);

}  // namespace osb

extern "C" {

// Widths served by the general-width (column-tile) instantiations of conv3d_tcg.cu / conv3d_tcs2.cu / conv3d_tcdc.cu: any row of
// at least OSB_TC_MIN_WIDTH voxels (below that a 128-column tile is mostly padding and the fp32 CUDA-core kernels win).
int osb_tc_general_width(int W) { return W >= OSB_TC_MIN_WIDTH ? 1 : 0; }

// K-chunk (input channels per operand tile) of the kernel variant that serves a shape; 0 = no tensor-core variant.
int osb_conv3d_tc_kc(int Cin, int Cout, int W, int stride) {
  if (stride != 1) return 0;
  if (W == osb::TC_W && (Cout == 32 || (Cout >= 1 && Cout <= 16)) && Cin % 32 == 0 && Cin >= 32) return 32;   // conv3d_tc.cu (narrow
                                                                                               // heads: weights zero-padded to 16 rows)
  if (Cin % 16 == 0 && Cin >= 16 &&
      ((W == 64 && Cout == 64) || (W == 32 && (Cout == 64 || Cout == 96 || Cout == 128)) || (W == 16 && (Cout == 64 || Cout == 96)) ||
       (W == osb::TC_W && (Cout == 64 || Cout == 128))))
    return 16;                                                                                  // conv3d_tcg.cu
  if (Cin % 16 == 0 && Cin >= 16 && osb_tc_general_width(W) && (Cout == 32 || Cout == 64 || Cout == 128))
    return 16;                                                                                  // conv3d_tcg.cu, column tiles
  return 0;
}

int osb_conv3d_tc_supported(int Cin, int Cout, int W, int stride) { return osb_conv3d_tc_kc(Cin, Cout, W, stride) != 0; }

int osb_ncdhw_to_ndhwc_pad(const float* x, float* y, int B, int C, int Cpad, int D, int H, int W, osb_stream_t stream) {
  using namespace osb;
  OSB_REQUIRE(x && y, "ncdhw_to_ndhwc: null pointer");
  OSB_REQUIRE(B > 0 && C > 0 && Cpad >= C && D > 0 && H > 0 && W > 0 && B <= 65535, "ncdhw_to_ndhwc: bad shape");
  const size_t vol = (size_t)D * H * W;
  dim3 grid((unsigned)((vol + 31) / 32), (Cpad + 31) / 32, B);
  ncdhw_to_ndhwc_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, y, C, Cpad, vol);
  count_launch();
  return check_launch("ncdhw_to_ndhwc_kernel");
}

int osb_ncdhw_to_ndhwc_pad_h16(const void* x, float* y, int B, int C, int Cpad, int D, int H, int W, osb_stream_t stream) {
  using namespace osb;
  OSB_REQUIRE(x && y, "ncdhw_to_ndhwc_h16: null pointer");
  OSB_REQUIRE(B > 0 && C > 0 && Cpad >= C && D > 0 && H > 0 && W > 0 && B <= 65535, "ncdhw_to_ndhwc_h16: bad shape");
  const size_t vol = (size_t)D * H * W;
  dim3 grid((unsigned)((vol + 31) / 32), (Cpad + 31) / 32, B);
  ncdhw_to_ndhwc_kernel<__half><<<grid, 256, 0, (cudaStream_t)stream>>>(static_cast<const __half*>(x), reinterpret_cast<__half*>(y), C, Cpad, vol);
  count_launch();
  return check_launch("ncdhw_to_ndhwc_kernel<half>");
}

int osb_ncdhw_to_ndhwc(const float* x, float* y, int B, int C, int D, int H, int W, osb_stream_t stream) {
  return osb_ncdhw_to_ndhwc_pad(x, y, B, C, C, D, H, W, stream);
}

static int conv3d_k3_tc_impl(const float* x_ndhwc, const void* w_split, const float* scale, const float* shift,
                             const float* residual, float* y, int B, int Cin, int Cout, int D, int H, int W, int act,
                             int out_ndhwc, int res_ndhwc, int in_ncdhw, osb_stream_t stream, const float* gate = nullptr,
                             int ystride = 0) {
  using namespace osb;
  OSB_REQUIRE(x_ndhwc && w_split && y, "conv3d_k3_tc: null pointer");
  OSB_REQUIRE(B > 0 && D > 0 && H > 0, "conv3d_k3_tc: empty shape");
  OSB_REQUIRE(osb_conv3d_tc_supported(Cin, Cout, W, 1), "conv3d_k3_tc: unsupported shape Cin=%d Cout=%d W=%d", Cin, Cout, W);
  OSB_REQUIRE(act >= 0 && act <= 2, "conv3d_k3_tc: unknown activation %d", act);
  OSB_REQUIRE((reinterpret_cast<uintptr_t>(x_ndhwc) & 15) == 0 && (reinterpret_cast<uintptr_t>(w_split) & 15) == 0 &&
                  (reinterpret_cast<uintptr_t>(y) & 15) == 0 && (reinterpret_cast<uintptr_t>(residual) & 15) == 0,
              "conv3d_k3_tc: pointers must be 16-byte aligned");
  OSB_REQUIRE(!in_ncdhw || osb_conv3d_tc_kc(Cin, Cout, W, 1) == 32, "conv3d_k3_tc: NCDHW input is served by the W = 128 kernel only");
  OSB_REQUIRE(ystride == 0 || (ystride >= Cout && ystride % 4 == 0 && osb_conv3d_tc_kc(Cin, Cout, W, 1) == 16 && out_ndhwc &&
                                (!residual || res_ndhwc)),
              "conv3d_k3_tc: a channel slice (ystride %d) needs channels-last tensors on the 16-channel-chunk kernels", ystride);
  OSB_REQUIRE(!gate || (osb_conv3d_tc_kc(Cin, Cout, W, 1) == 16 && out_ndhwc && (!residual || res_ndhwc) &&
                        (reinterpret_cast<uintptr_t>(gate) & 15) == 0),
              "conv3d_k3_tc: the gate operand needs a channels-last output (and residual) on the 16-channel-chunk kernels");
  if (osb_conv3d_tc_kc(Cin, Cout, W, 1) == 16)
    return launch_tcg_dispatch(x_ndhwc, w_split, scale, shift, residual, y, B, Cin, Cout, D, H, W, act, out_ndhwc, res_ndhwc,
                               (cudaStream_t)stream, gate, ystride);
  TcParams p{};
  p.x = x_ndhwc, p.w = w_split, p.scale = scale, p.shift = shift, p.residual = residual, p.y = y;
  p.B = B, p.D = D, p.H = H, p.Cin = Cin, p.Cout = Cout, p.act = act;
  p.kappa = rz_kappa(), p.overflow = tc_overflow_flag();
  OSB_REQUIRE(p.overflow, "conv3d_k3_tc: cannot allocate the overflow flag");
  p.out_ndhwc = out_ndhwc, p.res_ndhwc = res_ndhwc, p.in_ncdhw = in_ncdhw;
  {
    static const int bulk = [] { const char* e = getenv("OSB_TC_BULK"); return e ? atoi(e) : 1; }();   // 0: register-staged rows (A/B)
    p.bulk_rows = (bulk && (in_ncdhw || Cin == TC_KC)) ? 1 : 0;   // channels-last Cin = 64 rows are strided: register path
  }
  p.hblocks = (H + TC_TILES - 1) / TC_TILES;
  const long long items = (long long)B * D * p.hblocks;
  OSB_REQUIRE(items < (1ll << 31), "conv3d_k3_tc: too many work items");
  p.items = (int)items;
  if (Cout <= 16) {                                  // classifier heads (32 -> 1): COUT = 16 instantiation, NCDHW output only
    OSB_REQUIRE(!out_ndhwc && (!residual || !res_ndhwc), "conv3d_k3_tc: Cout <= 16 writes (and adds) NCDHW tensors only");
    return launch_tc<16>(p, (cudaStream_t)stream);
  }
  return launch_tc<32>(p, (cudaStream_t)stream);
}

int osb_conv3d_k3_tc_fwd(const float* x_ndhwc, const void* w_split, const float* scale, const float* shift,
                         const float* residual, float* y, int B, int Cin, int Cout, int D, int H, int W, int act,
                         int out_ndhwc, int res_ndhwc, osb_stream_t stream) {
  return conv3d_k3_tc_impl(x_ndhwc, w_split, scale, shift, residual, y, B, Cin, Cout, D, H, W, act, out_ndhwc, res_ndhwc, 0, stream);
}

int osb_conv3d_k3_tc_gate_fwd(const float* x_ndhwc, const void* w_split, const float* scale, const float* shift,
                              const float* residual, const float* gate_nhwc, float* y, int B, int Cin, int Cout, int D, int H, int W,
                              int act, osb_stream_t stream) {
  OSB_REQUIRE(gate_nhwc, "conv3d_k3_tc_gate: null gate");
  return conv3d_k3_tc_impl(x_ndhwc, w_split, scale, shift, residual, y, B, Cin, Cout, D, H, W, act, 1, 1, 0, stream, gate_nhwc);
}

int osb_conv3d_k3_tc_cs_fwd(const float* x_ndhwc, const void* w_split, const float* scale, const float* shift, const float* residual,
                            const float* gate_nhwc, float* y, int B, int Cin, int Cout, int D, int H, int W, int act, int ystride,
                            osb_stream_t stream) {
  return conv3d_k3_tc_impl(x_ndhwc, w_split, scale, shift, residual, y, B, Cin, Cout, D, H, W, act, 1, 1, 0, stream, gate_nhwc, ystride);
}

// ---- fp16 activations (H16 instantiations of conv3d_tcg.cu): channels-last fp16 x and y, fp32 gate, no residual
static int conv3d_k3_tc_h16_impl(const void* x_ndhwc, const void* w_split, const float* scale, const float* shift, const float* gate,
                                 float* y, int B, int Cin, int Cout, int D, int H, int W, int act, int ystride, osb_stream_t stream) {
  using namespace osb;
  OSB_REQUIRE(x_ndhwc && w_split && y, "conv3d_k3_tc_h16: null pointer");
  OSB_REQUIRE(B > 0 && D > 0 && H > 0, "conv3d_k3_tc_h16: empty shape");
  OSB_REQUIRE(tcg_h16_shape(Cin, Cout, W), "conv3d_k3_tc_h16: unsupported shape Cin=%d Cout=%d W=%d", Cin, Cout, W);
  OSB_REQUIRE(act >= 0 && act <= 2, "conv3d_k3_tc_h16: unknown activation %d", act);
  OSB_REQUIRE(ystride == 0 || (W == 16 && ystride >= Cout && ystride % 4 == 0), "conv3d_k3_tc_h16: bad channel stride %d", ystride);
  OSB_REQUIRE((reinterpret_cast<uintptr_t>(x_ndhwc) & 15) == 0 && (reinterpret_cast<uintptr_t>(w_split) & 15) == 0 &&
                  (reinterpret_cast<uintptr_t>(y) & 7) == 0 && (reinterpret_cast<uintptr_t>(gate) & 15) == 0,
              "conv3d_k3_tc_h16: x, w and gate must be 16-byte, y 8-byte aligned");
  return launch_tcg_h16(x_ndhwc, w_split, scale, shift, gate, y, B, Cin, Cout, D, H, W, act, ystride, (cudaStream_t)stream);
}

int osb_conv3d_tc_h16_supported(int Cin, int Cout, int W) { return osb::tcg_h16_shape(Cin, Cout, W) ? 1 : 0; }

int osb_conv3d_k3_tc_h16_fwd(const void* x_ndhwc, const void* w_split, const float* scale, const float* shift, float* y, int B, int Cin,
                             int Cout, int D, int H, int W, int act, osb_stream_t stream) {
  return conv3d_k3_tc_h16_impl(x_ndhwc, w_split, scale, shift, nullptr, y, B, Cin, Cout, D, H, W, act, 0, stream);
}

int osb_conv3d_k3_tc_gate_h16_fwd(const void* x_ndhwc, const void* w_split, const float* scale, const float* shift, const float* gate_nhwc,
                                  float* y, int B, int Cin, int Cout, int D, int H, int W, int act, osb_stream_t stream) {
  OSB_REQUIRE(gate_nhwc, "conv3d_k3_tc_gate_h16: null gate");
  return conv3d_k3_tc_h16_impl(x_ndhwc, w_split, scale, shift, gate_nhwc, y, B, Cin, Cout, D, H, W, act, 0, stream);
}

int osb_conv3d_k3_tc_cs_h16_fwd(const void* x_ndhwc, const void* w_split, const float* scale, const float* shift, const float* gate_nhwc,
                                float* y, int B, int Cin, int Cout, int D, int H, int W, int act, int ystride, osb_stream_t stream) {
  return conv3d_k3_tc_h16_impl(x_ndhwc, w_split, scale, shift, gate_nhwc, y, B, Cin, Cout, D, H, W, act, ystride, stream);
}

int osb_conv3d_k3_tc_ncdhw_fwd(const float* x_ncdhw, const void* w_split, const float* scale, const float* shift,
                               const float* residual, float* y, int B, int Cin, int Cout, int D, int H, int W, int act,
                               int out_ndhwc, int res_ndhwc, osb_stream_t stream) {
  return conv3d_k3_tc_impl(x_ncdhw, w_split, scale, shift, residual, y, B, Cin, Cout, D, H, W, act, out_ndhwc, res_ndhwc, 1, stream);
}

int osb_conv2d_tc_kc(int Cin, int Cout, int W, int dilation) {
  if (dilation == 1) return osb_conv3d_tc_kc(Cin, Cout, W, 1);
  if (dilation == 2 && W == osb::TC_W && Cout == 128 && Cin % 16 == 0 && Cin >= 16) return 16;
  return 0;
}

int osb_conv2d_k3_tc_fwd(const float* x_nhwc, const void* w_split, const float* scale, const float* shift, const float* residual,
                         float* y, int B, int Cin, int Cout, int H, int W, int dilation, int act, int out_nhwc, int res_nhwc,
                         osb_stream_t stream) {
  using namespace osb;
  if (dilation == 1)
    return osb_conv3d_k3_tc_fwd(x_nhwc, w_split, scale, shift, residual, y, B, Cin, Cout, 1, H, W, act, out_nhwc, res_nhwc, stream);
  OSB_REQUIRE(x_nhwc && w_split && y, "conv2d_k3_tc: null pointer");
  OSB_REQUIRE(B > 0 && H > 0, "conv2d_k3_tc: empty shape");
  OSB_REQUIRE(osb_conv2d_tc_kc(Cin, Cout, W, dilation) != 0, "conv2d_k3_tc: unsupported shape Cin=%d Cout=%d W=%d dilation=%d", Cin, Cout,
              W, dilation);
  OSB_REQUIRE(act >= 0 && act <= 2, "conv2d_k3_tc: unknown activation %d", act);
  OSB_REQUIRE((reinterpret_cast<uintptr_t>(x_nhwc) & 15) == 0 && (reinterpret_cast<uintptr_t>(w_split) & 15) == 0 &&
                  (reinterpret_cast<uintptr_t>(y) & 15) == 0 && (reinterpret_cast<uintptr_t>(residual) & 15) == 0,
              "conv2d_k3_tc: pointers must be 16-byte aligned");
  return launch_tcg_dilated2(x_nhwc, w_split, scale, shift, residual, y, B, Cin, Cout, H, W, act, out_nhwc, res_nhwc,
                             (cudaStream_t)stream);
}
}
