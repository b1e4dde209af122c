// Shared device helpers of the tcgen05 convolution kernels (conv3d_tc.cu: W = 128 specialisation; conv3d_tcg.cu: generic
// multi-row tiles).  See conv3d_tc.cu for the design notes.
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"

namespace osb {

// ------------------------------------------------------------------------------------------------ small PTX wrappers
// Wait used by the helper roles (loaders, epilogue): they run AHEAD of the MMA warp and would otherwise burn issue
// slots of the shared schedulers in a tight try_wait loop; back off between probes.
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  for (;;) {
    asm volatile(
        "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (done) return;
    __nanosleep(64);
  }
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// K-major, SWIZZLE_128B shared-memory matrix descriptor: 8-row atoms of 1024 bytes (SBO), version 1, address 0.
__device__ __forceinline__ uint64_t desc_sw128_base() {
  uint64_t d = 0;
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// Instruction descriptor of a dense kind::f16 MMA: fp16 A and B (formats 0), fp32 accumulator, both operands K-major.
__device__ __forceinline__ uint32_t idesc_f16(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 1-D bulk copy global -> shared through the TMA engine (SASS UBLKCP), completion counted in bytes on an mbarrier.  The weight
// slices are stored PRE-SWIZZLED in global memory (ops.pack_tc_weight), so one elected thread can stream them with no register
// staging, any number of slices in flight -- the LDG/STS weight loaders exposed one full L2 round trip per 12-24 KB slice
// (12 slices per work item of the backbone layers: ~10 us of the 25 us an item took, profiles/r2_step_ncu_summary.md).
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// 16-byte asynchronous copy global -> shared (LDGSTS) with zero fill when !valid: the A-unit loaders keep several units of raw
// fp32 rows in flight per warp WITHOUT holding them in registers (each lane later reads back exactly the bytes it copied, so no
// cross-lane synchronisation beyond cp.async.wait_group is needed).
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, bool valid) {
  const uint32_t n = valid ? 16u : 0u;
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
constexpr int TC_BSLOTS = 2;       // weight-slice buffers per kh tap: the producer runs one (kd, chunk) phase ahead of the MMAs
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}
// One lane of a fully converged warp (the tcgen05 issue idiom: control flow stays warp-uniform so descriptors live in
// uniform registers; only the MMA / commit instructions are predicated on the elected lane).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\nselp.u32 %0, 1, 0, p;\n}\n" : "=r"(pred));
  return pred != 0;
}
// 3xFP16 operand split (fp32-accurate products on the 16-bit tensor-core rate).
//   x * s  =  hi + lo + r,   hi = fp16_rn(x*s),  lo = fp16_rn(x*s - hi),   |r| <= max(2^-22 |x*s|, 2^-25)
// and every product is issued as  a_lo*b_hi + a_hi*b_lo + a_hi*b_hi  on tcgen05.mma.kind::f16 with fp32 accumulation in TMEM
// (the dropped lo*lo term is <= 2^-22 of the product; both roundings are to nearest, so the residual is zero-mean).  fp16
// carries the same 11 significant bits as TF32, so the accuracy equals the 3xTF32 scheme this replaces (round 1 / early round 2)
// while an MMA instruction covers K = 16 channels instead of 8: half the MMAs, half the operand bytes in shared memory --
// the two resources that bounded the TF32 kernels (DESIGN.md section 4.3).  What fp16 lacks is exponent range, hence the
// power-of-two scales: activations are staged as x * TC_ACT_SCALE (|x| < 65504 / TC_ACT_SCALE = 4094 is representable; smaller
// magnitudes keep 22 significant bits down to |x| ~ 2^-7 and an ABSOLUTE error of 2^-29 below that), weights are pre-scaled per
// output channel on the host so that max |w| lands in [2^14, 2^15) (ops.pack_tc_weight), and the epilogue's folded-BN scale
// carries the exact inverse 2^-(e_c + 4).  Conversions saturate (no inf/NaN poisoning) and a sticky device flag records any
// |x * s| > 65504 (osb_tc_overflow_count; the Python engines check it and refuse to return silently wrong results).
constexpr float TC_ACT_SCALE = 16.f;
constexpr float TC_F16_MAX = 65504.f;
// {lo 16 bits: fp16(a), hi 16 bits: fp16(b)}, round to nearest even, saturating to +-65504
__device__ __forceinline__ uint32_t cvt_f16x2_sat(float a, float b) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
__device__ __forceinline__ float2 f16x2_to_float2(uint32_t h) {
  float2 f;
  asm("{\n.reg .b16 l, u;\nmov.b32 {l, u}, %2;\ncvt.f32.f16 %0, l;\ncvt.f32.f16 %1, u;\n}\n" : "=f"(f.x), "=f"(f.y) : "r"(h));
  return f;
}
// four fp32 channels -> 4 fp16 hi parts + 4 fp16 lo parts of x * TC_ACT_SCALE; amax tracks max |x * s| for the overflow flag
__device__ __forceinline__ void f16_split4(const float4 v, uint2& hi, uint2& lo, float& amax) {
  const float x0 = v.x * TC_ACT_SCALE, x1 = v.y * TC_ACT_SCALE, x2 = v.z * TC_ACT_SCALE, x3 = v.w * TC_ACT_SCALE;
  amax = fmaxf(amax, fmaxf(fmaxf(fabsf(x0), fabsf(x1)), fmaxf(fabsf(x2), fabsf(x3))));
  hi.x = cvt_f16x2_sat(x0, x1);
  hi.y = cvt_f16x2_sat(x2, x3);
  const float2 h01 = f16x2_to_float2(hi.x), h23 = f16x2_to_float2(hi.y);
  lo.x = cvt_f16x2_sat(x0 - h01.x, x1 - h01.y);
  lo.y = cvt_f16x2_sat(x2 - h23.x, x3 - h23.y);
}
unsigned int* tc_overflow_flag();      // api.cu: device address of the sticky overflow counter of the CURRENT device
__device__ __forceinline__ void tc_report_overflow(unsigned int* flag, float amax) {
  if (amax > TC_F16_MAX) atomicAdd(flag, 1u);
}

// The TMEM accumulator of tcgen05.mma rounds TOWARDS ZERO (tools/tc_probe.cu acc, profiles/r2_acc_probe.log: accumulating the same
// positive product block n times loses n * 2^-24 of the sum, where round-to-nearest would lose ~sqrt(n) * 2^-25).  Each MMA
// therefore shrinks the running sum by ~c * ulp, and because E[partial sum after i of n MMAs | final] = (i/n) * final, an
// accumulator that received n MMAs comes out as final * (1 - kappa * n) plus zero-mean noise.  The shrink is coherent from
// layer to layer (round 1: -4e-5 on the GwcNet logits, 2.3e-3 px EPE), the noise is not -- so the epilogue undoes the EXPECTED
// loss: raw sum * (1 + kappa * n), n = MMAs issued into that accumulator for this work item.  kappa is measured
// (tools/parity_bisect.py --layers: every kernel variant agrees within 10 %); osb_set_rz_kappa() overrides it for calibration.
float rz_kappa();           // api.cu


// K-major SWIZZLE_64B descriptor base (64-byte rows, 512-byte 8-row atoms)
__device__ __forceinline__ uint64_t desc_sw64_base() {
  uint64_t d = 0;
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(512 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)4 << 61;
  return d;
}
// byte offset of 16-byte chunk `c` of K-major row `row` inside a swizzled operand tile
template <int KC>
__device__ __forceinline__ int swz_offset(int row, int c) {
  if constexpr (KC == 32) return row * 128 + ((c ^ (row & 7)) << 4);          // SWIZZLE_128B
  else return row * 64 + ((c ^ ((row >> 1) & 3)) << 4);                        // SWIZZLE_64B
}


// Stage four fp32 channels (fp32 16-byte chunk `q` of the KC-channel slice of operand row `row`) into a swizzled operand tile whose
// K-major rows hold [KC fp16 hi | KC fp16 lo] = 4*KC bytes: hi part to 16-byte chunk q/2, lo part to chunk KC/8 + q/2, 8 bytes each.
template <int KC>
__device__ __forceinline__ void stage_f16_split(uint8_t* tile, int row, int q, const float4 v, float& amax) {
  uint2 hi, lo;
  f16_split4(v, hi, lo, amax);
  const int sub = (q & 1) << 3;
  *reinterpret_cast<uint2*>(tile + swz_offset<KC>(row, q >> 1) + sub) = hi;
  *reinterpret_cast<uint2*>(tile + swz_offset<KC>(row, KC / 8 + (q >> 1)) + sub) = lo;
}
// 16-bit activation route (H16 instantiations, DESIGN.md section 4.11): the activations already ARE fp16 (the caller ran the model
// under autocast and asked for 16-bit arithmetic), so four channels arrive as 8 bytes and go to the hi half of the row unchanged --
// no TC_ACT_SCALE, no split, the lo half of the row is never read (one MMA per k-step, A hi x B hi).
template <int KC>
__device__ __forceinline__ void stage_f16_hi(uint8_t* tile, int row, int q, const uint2 v) {
  *reinterpret_cast<uint2*>(tile + swz_offset<KC>(row, q >> 1) + ((q & 1) << 3)) = v;
}
// activation element / 4-channel load type of the loaders and products per k-step of the two routes
template <bool H16>
struct TcAct {
  using T = float;
  using V = float4;
  static constexpr int TERMS = 3;      // lo*hi + hi*lo + hi*hi
};
template <>
struct TcAct<true> {
  using T = __half;
  using V = uint2;
  static constexpr int TERMS = 1;      // hi*hi
};

// Lane -> operand row inside a warp-wide load of VPL = 128 / KC voxels (KC/4 lanes each), permuted so that the two STS.64 of
// stage_f16_split are bank-conflict free per half-warp: SWIZZLE_128B rows (KC = 32) must differ in bit 2, SWIZZLE_64B rows
// (KC = 16) must be {r, r+1, r+4, r+5}.  Global loads stay whole 16-byte chunks of whole voxels either way.
template <int KC>
__device__ __forceinline__ int lane_voxel(int lane) {
  if constexpr (KC == 32) return (((lane >> 3) & 1) << 2) | (lane >> 4);                       // 4 voxels: 0,4 | 1,5 (caller adds the rest)
  else return ((lane >> 2) & 1) | (((lane >> 3) & 1) << 2) | ((lane >> 4) << 1);               // 8 voxels: 0,1,4,5 | 2,3,6,7
}
// MMAs issued per accumulator per staged (unit, weight slice): k-steps of 16 channels x 3 split terms
template <int KC>
struct TcK {
  static constexpr int KSTEPS = KC / 16;
  static constexpr int LO_OFF = KC / 8;           // descriptor start-address offset (16-byte units) of the lo half of a row
};

// ------------------------------------------------------------------------------- coalesced channels-last epilogue output
// An epilogue thread owns ONE voxel and all of its channels.  Storing those directly makes every STG.128 of a warp touch
// 32 different 128-byte lines (16 B of each) -- 8x the L1 wavefronts of a coalesced store, on the data pipe the tensor
// core's operand reads also use (ncu r1_conv3d_tc_v7: tc 49 % + lsu 43 % of that pipe).  Instead the warp transposes its
// 32 voxels x 32 channels through a private shared-memory tile so one instruction covers 4 voxels x 128 contiguous bytes;
// folded BN, the channels-last residual and the activation are applied after the transpose, where a lane's four channels
// are the same for every voxel (scale/shift sit in registers instead of one LDS per channel).
constexpr int TP_STRIDE = 36;                       // floats per tile row: 144 B keeps STS.128 / LDS.128 conflict-free
constexpr int TP_WARP_FLOATS = 32 * TP_STRIDE;      // 4608 B per epilogue warp
constexpr int TP_BYTES = 4 * TP_WARP_FLOATS * 4;    // four epilogue warps

// sum[32]: raw accumulator sums of this lane's voxel for channels [c, c+32).  y0 / res0 point at channel c of the voxel
// owned by lane 0; lane k's voxel lies vstride floats further per lane.  sc / sh point at channel c of the folded BN.
// vmask: bit k set = the voxel of lane k exists in the output (general-width column tiles mask their halo columns and the part of
// the last tile beyond the image; whole-row tiles pass all ones and the tests fold away).
// gate0: optional channels-last multiplier of lane 0's voxel (same voxel stride), applied AFTER the activation -- FeatureAtt's
// sigmoid(att) * cv of stereobase/hourglass.py:80-99 / igev_blocks.py:35-48 with the gate stored as (B, H, W, C).
// T = __half (H16 instantiations): the fp32 results are stored with cvt.rn.satfinite; *amax tracks their largest magnitude so the
// caller can count values that saturated at +-65504 (tc_report_overflow).
template <typename T = float>
__device__ __forceinline__ void store_ndhwc_chunk32(float* tbuf, int lane, const float (&sum)[32], T* y0, const float* res0,
                                                    size_t vstride, const float* sc, const float* sh, int act,
                                                    uint32_t vmask = 0xffffffffu, const float* gate0 = nullptr,
                                                    float* amax = nullptr) {
  const int c4 = 4 * (lane & 7), sub = lane >> 3;
  __syncwarp();                                     // the previous chunk's readers are done with the tile
  float4* row = reinterpret_cast<float4*>(tbuf + lane * TP_STRIDE);
#pragma unroll
  for (int i = 0; i < 8; ++i) row[i] = make_float4(sum[4 * i], sum[4 * i + 1], sum[4 * i + 2], sum[4 * i + 3]);
  __syncwarp();
  const float4 a = *reinterpret_cast<const float4*>(sc + c4);
  const float4 b = *reinterpret_cast<const float4*>(sh + c4);
  float4 o[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    o[j] = *reinterpret_cast<const float4*>(tbuf + (4 * j + sub) * TP_STRIDE + c4);
    o[j].x = fmaf(o[j].x, a.x, b.x), o[j].y = fmaf(o[j].y, a.y, b.y), o[j].z = fmaf(o[j].z, a.z, b.z), o[j].w = fmaf(o[j].w, a.w, b.w);
  }
  if (res0) {
    float4 r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j)
      r[j] = ((vmask >> (4 * j + sub)) & 1u) ? __ldg(reinterpret_cast<const float4*>(res0 + (size_t)(4 * j + sub) * vstride + c4))
                                             : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j].x += r[j].x, o[j].y += r[j].y, o[j].z += r[j].z, o[j].w += r[j].w;
  }
  if (act == OSB_ACT_RELU) {
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j].x = fmaxf(o[j].x, 0.f), o[j].y = fmaxf(o[j].y, 0.f), o[j].z = fmaxf(o[j].z, 0.f), o[j].w = fmaxf(o[j].w, 0.f);
  } else if (act == OSB_ACT_LEAKY) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      o[j].x = o[j].x > 0.f ? o[j].x : 0.01f * o[j].x, o[j].y = o[j].y > 0.f ? o[j].y : 0.01f * o[j].y;
      o[j].z = o[j].z > 0.f ? o[j].z : 0.01f * o[j].z, o[j].w = o[j].w > 0.f ? o[j].w : 0.01f * o[j].w;
    }
  }
  if (gate0) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (!((vmask >> (4 * j + sub)) & 1u)) continue;
      const float4 g = __ldg(reinterpret_cast<const float4*>(gate0 + (size_t)(4 * j + sub) * vstride + c4));
      o[j].x *= g.x, o[j].y *= g.y, o[j].z *= g.z, o[j].w *= g.w;
    }
  }
  if constexpr (sizeof(T) == 2) {
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if ((vmask >> (4 * j + sub)) & 1u) {
        *amax = fmaxf(*amax, fmaxf(fmaxf(fabsf(o[j].x), fabsf(o[j].y)), fmaxf(fabsf(o[j].z), fabsf(o[j].w))));
        *reinterpret_cast<uint2*>(y0 + (size_t)(4 * j + sub) * vstride + c4) =
            make_uint2(cvt_f16x2_sat(o[j].x, o[j].y), cvt_f16x2_sat(o[j].z, o[j].w));
      }
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if ((vmask >> (4 * j + sub)) & 1u) *reinterpret_cast<float4*>(y0 + (size_t)(4 * j + sub) * vstride + c4) = o[j];
  }
}

}  // namespace osb
