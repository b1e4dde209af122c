// Direct (im2col-free) fp32 3D convolutions for the hourglass aggregation, sm_100a.
//
//   Conv3d k3 s1/s2 + BN + act (+residual, +gate)   convbn_3d gwcnet/hourglass.py:5-16, gwcnet_disp_processor.py:8-19
//                                                   conv3d_bn(_relu) psmnet/submodule.py:68-83,160-177
//                                                   BasicConv3d common/basic_block_3d.py:5-20
//   ConvTranspose3d k3 s2 p1 op1 / k4 s2 p1 + BN    gwcnet/hourglass.py:35-41, psmnet deconv3d_bn submodule.py:86-100,
//                                                   BasicDeconv3d stereobase/hourglass.py:39-49
//   Conv3d k1 (+ channel concat of two inputs)      redir1/2 gwcnet/hourglass.py:43-44, agg_0/agg_1 stereobase/hourglass.py:51-66
//
// Numerics: IEEE fp32 FMA accumulation on the CUDA cores.  TF32/BF16 tensor-core operands break the 1e-3 px EPE bar
// of the north star (SURVEY.md section 4.3: 2.2e-2 / 1.8e-1 px), so the 3x3x3 path stays on the fp32 pipe.
//
// Register tiling: one thread owns 8 consecutive output voxels along W x 8 output channels (64 accumulators).  Per
// (input channel, kd, kh) it reads a 10-float input row segment and 3x8 weights from shared memory and issues 192 FMAs
// (~22 FMA per shared-memory load instruction), so the kernel is bound by the fp32 FMA pipe, not by LDS or HBM.
// BatchNorm (eval) is folded into a per-channel scale/shift epilogue together with the residual add, the activation
// and StereoBase's sigmoid channel gate, so no elementwise pass ever touches HBM.
#include <algorithm>

#include <cuda_fp16.h>

#include "common.cuh"

namespace osb {

struct ConvParams {
  const float* x;
  const float* x1;       // second channel slab (1x1 only)
  const float* w;        // packed (Cin, taps, Cout)
  const float* scale;
  const float* shift;
  const float* residual;
  const float* gate;
  float* y;
  int B, Cin, Cin0, Cout;
  int D, H, W;           // input extent
  int Do, Ho, Wo;        // output extent
  int tiles_w, tiles_h, tiles_d;
  int act, sigmoid_out, vec_ok;
};

__device__ __forceinline__ float activate(float v, int act) {
  if (act == OSB_ACT_RELU) return fmaxf(v, 0.f);
  if (act == OSB_ACT_LEAKY) return v > 0.f ? v : 0.01f * v;
  if (act == OSB_ACT_RELU6) return fminf(fmaxf(v, 0.f), 6.f);
  return v;
}

// Shared epilogue: acc[c][v] -> y for TCO channels x 8 consecutive output columns.
template <int TCO>
__device__ __forceinline__ void epilogue(const ConvParams& p, float (&acc)[TCO][8], int b, int co_first, int od, int oh,
                                         int ow_first) {
  if (od >= p.Do || oh >= p.Ho || ow_first >= p.Wo) return;
#pragma unroll
  for (int c = 0; c < TCO; ++c) {
    const int co = co_first + c;
    if (co >= p.Cout) break;
    const float sc = p.scale ? __ldg(p.scale + co) : 1.f;
    const float sh = p.shift ? __ldg(p.shift + co) : 0.f;
    const size_t row = (((size_t)(b * p.Cout + co) * p.Do + od) * p.Ho + oh) * p.Wo + ow_first;
    const float* grow = p.gate ? p.gate + ((size_t)(b * p.Cout + co) * p.Ho + oh) * p.Wo + ow_first : nullptr;
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = fmaf(acc[c][i], sc, sh);
    if (p.vec_ok && ow_first + 7 < p.Wo) {
      if (p.residual) {
        const float4 r0 = __ldg(reinterpret_cast<const float4*>(p.residual + row));
        const float4 r1 = __ldg(reinterpret_cast<const float4*>(p.residual + row + 4));
        v[0] += r0.x, v[1] += r0.y, v[2] += r0.z, v[3] += r0.w, v[4] += r1.x, v[5] += r1.y, v[6] += r1.z, v[7] += r1.w;
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = activate(v[i], p.act);
      if (grow) {
        const float4 g0 = __ldg(reinterpret_cast<const float4*>(grow));
        const float4 g1 = __ldg(reinterpret_cast<const float4*>(grow + 4));
        v[0] *= g0.x, v[1] *= g0.y, v[2] *= g0.z, v[3] *= g0.w, v[4] *= g1.x, v[5] *= g1.y, v[6] *= g1.z, v[7] *= g1.w;
      }
      if (p.sigmoid_out) {
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = 1.f / (1.f + expf(-v[i]));
      }
      *reinterpret_cast<float4*>(p.y + row) = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<float4*>(p.y + row + 4) = make_float4(v[4], v[5], v[6], v[7]);
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (ow_first + i < p.Wo) {
          float t = v[i];
          if (p.residual) t += __ldg(p.residual + row + i);
          t = activate(t, p.act);
          if (grow) t *= __ldg(grow + i);
          if (p.sigmoid_out) t = 1.f / (1.f + expf(-t));
          p.y[row + i] = t;
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ 3x3x3, stride S
// CTA tile: TD x TH x 32 output voxels, NCG*TCO output channels; threads = NCG * TD*TH*4.
template <int S, int TCO, int NCG, int TD, int TH, int CI>
struct ConvCfg {
  static constexpr int TW = 32;
  static constexpr int VG = TD * TH * 4;               // voxel groups (8 columns each)
  static constexpr int THREADS = NCG * VG;
  static constexpr int COB = TCO * NCG;
  static constexpr int ID = (TD - 1) * S + 3, IH = (TH - 1) * S + 3, IW = (TW - 1) * S + 3;
  static constexpr int PITCH = (IW + 3) / 4 * 4;       // 36 (S=1) / 68 (S=2)
  static constexpr int XS = CI * ID * IH * PITCH;      // floats
  static constexpr int WS = CI * 27 * COB;
  static constexpr size_t SMEM = (size_t)(XS + WS) * sizeof(float);
};

template <int S, int TCO, int NCG, int TD, int TH, int CI>
__global__ void __launch_bounds__(NCG* TD* TH * 4) conv3d_k3_kernel(const ConvParams p) {
  using C = ConvCfg<S, TCO, NCG, TD, TH, CI>;
  extern __shared__ __align__(16) float smem[];
  float* xs = smem;
  float* ws = smem + C::XS;
  const int tid = threadIdx.x;
  const int cg = tid / C::VG, vg = tid % C::VG;
  const int wg = vg & 3, th = (vg >> 2) % TH, td = vg / (4 * TH);
  int t = blockIdx.x;
  const int tw = t % p.tiles_w;
  t /= p.tiles_w;
  const int thh = t % p.tiles_h;
  const int tdd = t / p.tiles_h;
  const int b = blockIdx.z;
  const int co0 = blockIdx.y * C::COB;
  const int od0 = tdd * TD, oh0 = thh * TH, ow0 = tw * C::TW;
  const int id0 = od0 * S - 1, ih0 = oh0 * S - 1, iw0 = ow0 * S - 1;  // input coordinate of xs[.][0][0][0]

  float acc[TCO][8];
#pragma unroll
  for (int c = 0; c < TCO; ++c)
#pragma unroll
    for (int v = 0; v < 8; ++v) acc[c][v] = 0.f;

  const size_t in_plane = (size_t)p.H * p.W;
  const size_t in_vol = (size_t)p.D * in_plane;
  for (int c0 = 0; c0 < p.Cin; c0 += CI) {
    __syncthreads();                                   // previous chunk fully consumed
    // ---- stage the input halo tile (zero padding = the conv's padding=1) ----
    for (int idx = tid; idx < C::XS; idx += C::THREADS) {
      const int wx = idx % C::PITCH;
      int r = idx / C::PITCH;
      const int hy = r % C::IH;
      r /= C::IH;
      const int dz = r % C::ID;
      const int ci = r / C::ID;
      const int gd = id0 + dz, gh = ih0 + hy, gw = iw0 + wx, gc = c0 + ci;
      float v = 0.f;
      if (wx < C::IW && gc < p.Cin && gd >= 0 && gd < p.D && gh >= 0 && gh < p.H && gw >= 0 && gw < p.W)
        v = __ldg(p.x + (size_t)(b * p.Cin + gc) * in_vol + (size_t)gd * in_plane + (size_t)gh * p.W + gw);
      xs[idx] = v;
    }
    // ---- stage the weight slab (CI, 27, COB) ----
    for (int idx = tid; idx < C::WS; idx += C::THREADS) {
      const int c = idx % C::COB;
      const int r = idx / C::COB;                      // ci*27 + tap
      const int ci = r / 27;
      float v = 0.f;
      if (c0 + ci < p.Cin && co0 + c < p.Cout) v = __ldg(p.w + ((size_t)(c0 * 27 + r)) * p.Cout + co0 + c);
      ws[idx] = v;
    }
    __syncthreads();
    // ---- 192 FMAs per (ci, kd, kh) ----
#pragma unroll 1
    for (int ci = 0; ci < CI; ++ci) {
#pragma unroll
      for (int kd = 0; kd < 3; ++kd) {
#pragma unroll
        for (int kh = 0; kh < 3; ++kh) {
          const float* xr = xs + ((ci * C::ID + td * S + kd) * C::IH + th * S + kh) * C::PITCH + wg * 8 * S;
          constexpr int NX = 7 * S + 3;                // 10 (S=1) / 17 (S=2)
          float xv[NX + 3];
#pragma unroll
          for (int q = 0; q < (NX + 3) / 4; ++q) {
            const float4 t4 = *reinterpret_cast<const float4*>(xr + 4 * q);
            xv[4 * q + 0] = t4.x, xv[4 * q + 1] = t4.y, xv[4 * q + 2] = t4.z, xv[4 * q + 3] = t4.w;
          }
          const float* wr = ws + (ci * 27 + (kd * 3 + kh) * 3) * C::COB + cg * TCO;
#pragma unroll
          for (int kw = 0; kw < 3; ++kw) {
            float wv[TCO];
            if constexpr (TCO % 4 == 0) {
#pragma unroll
              for (int q = 0; q < TCO / 4; ++q) {
                const float4 t4 = *reinterpret_cast<const float4*>(wr + kw * C::COB + 4 * q);
                wv[4 * q + 0] = t4.x, wv[4 * q + 1] = t4.y, wv[4 * q + 2] = t4.z, wv[4 * q + 3] = t4.w;
              }
            } else {
#pragma unroll
              for (int c = 0; c < TCO; ++c) wv[c] = wr[kw * C::COB + c];
            }
#pragma unroll
            for (int c = 0; c < TCO; ++c)
#pragma unroll
              for (int v = 0; v < 8; ++v) acc[c][v] = fmaf(wv[c], xv[v * S + kw], acc[c][v]);
          }
        }
      }
    }
  }
  epilogue<TCO>(p, acc, b, co0 + cg * TCO, od0 + td, oh0 + th, ow0 + wg * 8);
}

// ------------------------------------------------------------------------------------- transposed conv, stride 2
// Output voxel o gathers input i = m + off where m = o>>1 and, per dimension, the taps of parity p = o&1 are
//   p=0: k=1 (off 0), k=3 (off -1, KS=4 only);   p=1: k=0 (off +1), k=2 (off 0).
// CTA tile: 4 x 4 x 64 output voxels x 16 channels; threads are laid out so that every warp has one (pd, ph) parity
// class and therefore executes exactly its own taps (no divergence).
template <int KS, int CI>
struct DeconvCfg {
  static constexpr int TD = 4, TH = 4, TW = 64, TCO = 8, NCG = 2;
  static constexpr int THREADS = 256, COB = 16;
  static constexpr int ID = TD / 2 + 2, IH = TH / 2 + 2, IW = TW / 2 + 2, PITCH = 36;
  static constexpr int XS = CI * ID * IH * PITCH;
  static constexpr int TAPS = KS * KS * KS;
  static constexpr int WS = CI * TAPS * COB;
  static constexpr size_t SMEM = (size_t)(XS + WS) * sizeof(float);
};

template <int KS, int CI>
__global__ void __launch_bounds__(256) deconv3d_kernel(const ConvParams p) {
  using C = DeconvCfg<KS, CI>;
  extern __shared__ __align__(16) float smem[];
  float* xs = smem;
  float* ws = smem + C::XS;
  const int tid = threadIdx.x;
  const int cg = tid >> 7, vg = tid & 127;
  const int cls = vg >> 5, pd = cls >> 1, ph = cls & 1;
  const int r5 = (vg & 31) >> 3, dd = r5 >> 1, hh = r5 & 1, wg = vg & 7;
  int t = blockIdx.x;
  const int tw = t % p.tiles_w;
  t /= p.tiles_w;
  const int thh = t % p.tiles_h;
  const int tdd = t / p.tiles_h;
  const int b = blockIdx.z;
  const int co0 = blockIdx.y * C::COB;
  const int od0 = tdd * C::TD, oh0 = thh * C::TH, ow0 = tw * C::TW;
  const int id0 = od0 / 2 - 1, ih0 = oh0 / 2 - 1, iw0 = ow0 / 2 - 1;

  float acc[8][8];
#pragma unroll
  for (int c = 0; c < 8; ++c)
#pragma unroll
    for (int v = 0; v < 8; ++v) acc[c][v] = 0.f;

  const size_t in_plane = (size_t)p.H * p.W;
  const size_t in_vol = (size_t)p.D * in_plane;
  for (int c0 = 0; c0 < p.Cin; c0 += CI) {
    __syncthreads();
    for (int idx = tid; idx < C::XS; idx += C::THREADS) {
      const int wx = idx % C::PITCH;
      int r = idx / C::PITCH;
      const int hy = r % C::IH;
      r /= C::IH;
      const int dz = r % C::ID;
      const int ci = r / C::ID;
      const int gd = id0 + dz, gh = ih0 + hy, gw = iw0 + wx, gc = c0 + ci;
      float v = 0.f;
      if (wx < C::IW && gc < p.Cin && gd >= 0 && gd < p.D && gh >= 0 && gh < p.H && gw >= 0 && gw < p.W)
        v = __ldg(p.x + (size_t)(b * p.Cin + gc) * in_vol + (size_t)gd * in_plane + (size_t)gh * p.W + gw);
      xs[idx] = v;
    }
    for (int idx = tid; idx < C::WS; idx += C::THREADS) {
      const int c = idx % C::COB;
      const int r = idx / C::COB;                      // ci*TAPS + tap
      const int ci = r / C::TAPS;
      float v = 0.f;
      if (c0 + ci < p.Cin && co0 + c < p.Cout) v = __ldg(p.w + ((size_t)c0 * C::TAPS + r) * p.Cout + co0 + c);
      ws[idx] = v;
    }
    __syncthreads();
#pragma unroll 1
    for (int ci = 0; ci < CI; ++ci) {
#pragma unroll
      for (int kd = 0; kd < KS; ++kd) {
        if ((pd + 1 - kd) & 1) continue;               // warp-uniform
        const int offd = (pd + 1 - kd) >> 1;           // -1, 0 or +1
#pragma unroll
        for (int kh = 0; kh < KS; ++kh) {
          if ((ph + 1 - kh) & 1) continue;
          const int offh = (ph + 1 - kh) >> 1;
          // xs row holds input columns m0-1 .. m0+4 for this thread's m0 = ow0/2 + 4*wg
          const float* xr = xs + ((ci * C::ID + dd + 1 + offd) * C::IH + hh + 1 + offh) * C::PITCH + wg * 4;
          const float4 xa = *reinterpret_cast<const float4*>(xr);
          const float2 xb = *reinterpret_cast<const float2*>(xr + 4);
          const float xv[6] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y};
          const float* wr = ws + ((ci * KS + kd) * KS + kh) * KS * C::COB + cg * 8;
          float wv[KS][8];
#pragma unroll
          for (int kw = 0; kw < KS; ++kw) {
            const float4 a = *reinterpret_cast<const float4*>(wr + kw * C::COB);
            const float4 c4 = *reinterpret_cast<const float4*>(wr + kw * C::COB + 4);
            wv[kw][0] = a.x, wv[kw][1] = a.y, wv[kw][2] = a.z, wv[kw][3] = a.w;
            wv[kw][4] = c4.x, wv[kw][5] = c4.y, wv[kw][6] = c4.z, wv[kw][7] = c4.w;
          }
#pragma unroll
          for (int c = 0; c < 8; ++c) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              // even column 2(m0+u): k=1 <- x[m0+u] (= xv[u+1]); KS=4 also k=3 <- x[m0+u-1] (= xv[u])
              acc[c][2 * u] = fmaf(wv[1][c], xv[u + 1], acc[c][2 * u]);
              if constexpr (KS == 4) acc[c][2 * u] = fmaf(wv[3][c], xv[u], acc[c][2 * u]);
              // odd column 2(m0+u)+1: k=0 <- x[m0+u+1] (= xv[u+2]), k=2 <- x[m0+u] (= xv[u+1])
              acc[c][2 * u + 1] = fmaf(wv[0][c], xv[u + 2], acc[c][2 * u + 1]);
              acc[c][2 * u + 1] = fmaf(wv[2][c], xv[u + 1], acc[c][2 * u + 1]);
            }
          }
        }
      }
    }
  }
  epilogue<8>(p, acc, b, co0 + cg * 8, od0 + 2 * dd + pd, oh0 + 2 * hh + ph, ow0 + wg * 8);
}

// --------------------------------------------------------------------------------------------------- 1x1x1 conv
// CTA: 64 voxel-octets (512 voxels of the flattened D*H*W axis... per row of W) x 32 output channels.
// The weight slab (<=128 input channels at a time) lives in shared memory; inputs stream from global.
constexpr int kPwChunk = 128;
__global__ void __launch_bounds__(256) conv3d_1x1_kernel(const ConvParams p) {
  __shared__ __align__(16) float ws[kPwChunk * 32];
  const int tid = threadIdx.x;
  const int cg = tid >> 6, vq = tid & 63;
  const int b = blockIdx.z;
  const int co0 = blockIdx.y * 32;
  const size_t vol = (size_t)p.D * p.H * p.W;
  // voxel octet = 8 consecutive columns of one (d,h) row
  const int octs_per_row = (p.W + 7) / 8;
  const size_t oct = (size_t)blockIdx.x * 64 + vq;
  const size_t rows = (size_t)p.D * p.H;
  const bool live = oct < rows * octs_per_row;
  const size_t row = live ? oct / octs_per_row : 0;
  const int ow = live ? (int)(oct % octs_per_row) * 8 : 0;
  const size_t off = row * p.W + ow;
  const bool vec = p.vec_ok && (ow + 7 < p.W);

  float acc[8][8];
#pragma unroll
  for (int c = 0; c < 8; ++c)
#pragma unroll
    for (int v = 0; v < 8; ++v) acc[c][v] = 0.f;

  for (int c0 = 0; c0 < p.Cin; c0 += kPwChunk) {
    const int nci = min(kPwChunk, p.Cin - c0);
    __syncthreads();
    for (int idx = tid; idx < nci * 32; idx += 256) {
      const int c = idx & 31, ci = idx >> 5;
      ws[idx] = (co0 + c < p.Cout) ? __ldg(p.w + (size_t)(c0 + ci) * p.Cout + co0 + c) : 0.f;
    }
    __syncthreads();
    if (live) {
#pragma unroll 2
      for (int ci = 0; ci < nci; ++ci) {
        const int gc = c0 + ci;
        const float* src = (gc < p.Cin0) ? p.x + ((size_t)b * p.Cin0 + gc) * vol
                                         : p.x1 + ((size_t)b * (p.Cin - p.Cin0) + (gc - p.Cin0)) * vol;
        float xv[8];
        if (vec) {
          const float4 a = __ldg(reinterpret_cast<const float4*>(src + off));
          const float4 c4 = __ldg(reinterpret_cast<const float4*>(src + off + 4));
          xv[0] = a.x, xv[1] = a.y, xv[2] = a.z, xv[3] = a.w, xv[4] = c4.x, xv[5] = c4.y, xv[6] = c4.z, xv[7] = c4.w;
        } else {
#pragma unroll
          for (int v = 0; v < 8; ++v) xv[v] = (ow + v < p.W) ? __ldg(src + off + v) : 0.f;
        }
        const float4 wa = *reinterpret_cast<const float4*>(ws + ci * 32 + cg * 8);
        const float4 wb = *reinterpret_cast<const float4*>(ws + ci * 32 + cg * 8 + 4);
        const float wv[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
#pragma unroll
        for (int c = 0; c < 8; ++c)
#pragma unroll
          for (int v = 0; v < 8; ++v) acc[c][v] = fmaf(wv[c], xv[v], acc[c][v]);
      }
    }
  }
  if (live) {
    const int od = (int)(row / p.H), oh = (int)(row % p.H);
    epilogue<8>(p, acc, b, co0 + cg * 8, od, oh, ow);
  }
}

// --------------------------------------------------------------------------------- channels-last 1x1x1 conv
// x (V, Cin) -> y (V, Cout), y = act(x.W * scale + shift): the redir1/redir2 branches of the GwcNet hourglass
// (gwcnet/hourglass.py:43-44, :53-54) when the aggregation runs channels-last for the tensor-core kernels.
// A warp owns 32 consecutive voxels: it reads their 32 x Cin block with fully coalesced LDG.128 (a thread-per-voxel read
// touches 32 different lines per instruction), transposes it through a private shared-memory tile so that each lane then
// holds one voxel's Cin inputs in registers, multiplies by the (Cin x Cout) matrix broadcast from shared memory, and writes
// the result back through the same tile, again coalesced.  Memory-bound: Cin + Cout floats per voxel.
template <int CIN, int COUT>
__global__ void __launch_bounds__(64) conv1x1_ndhwc_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                           const float* __restrict__ scale, const float* __restrict__ shift,
                                                           float* __restrict__ y, size_t V, int act) {
  static_assert(CIN == COUT, "the in/out tiles share one buffer");
  constexpr int TS = CIN + 4;                       // tile row stride (floats): 16-byte aligned, conflict-free per quarter warp
  constexpr int F4 = CIN / 4;                       // float4 per voxel
  __shared__ __align__(16) float ws[CIN * COUT];
  __shared__ __align__(16) float tile[2][32 * TS];
  __shared__ __align__(16) float s_sc[COUT];
  __shared__ __align__(16) float s_sh[COUT];
  for (int i = threadIdx.x; i < CIN * COUT; i += 64) ws[i] = __ldg(w + i);           // packed (Cin, Cout)
  for (int i = threadIdx.x; i < COUT; i += 64) {
    s_sc[i] = scale ? __ldg(scale + i) : 1.f;
    s_sh[i] = shift ? __ldg(shift + i) : 0.f;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* tl = tile[warp];
  const size_t ngroups = (V + 31) / 32;
  // software pipeline: the NEXT group's 32 x Cin block is already on its way from HBM while this one is multiplied (without it
  // every warp sat on one full DRAM round trip per group: 0.38 ms for the 806 MB of a full-resolution redir, 2.1 TB/s)
  float4 nxt[F4];
  auto fetch = [&](size_t g) {
    const size_t v0 = g * 32;
    const int nv = (int)min((size_t)32, V - v0);
    const float4* src = reinterpret_cast<const float4*>(x + v0 * CIN);
#pragma unroll
    for (int j = 0; j < F4; ++j) {                  // coalesced: 512 contiguous bytes per instruction
      const int f = lane + 32 * j;
      nxt[j] = (f / F4 < nv) ? __ldg(src + f) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  const size_t g0 = (size_t)blockIdx.x * 2 + warp, gstep = (size_t)gridDim.x * 2;
  if (g0 < ngroups) fetch(g0);
  for (size_t g = g0; g < ngroups; g += gstep) {
    const size_t v0 = g * 32;
    const int nv = (int)min((size_t)32, V - v0);
    __syncwarp();
#pragma unroll
    for (int j = 0; j < F4; ++j) {
      const int f = lane + 32 * j, vox = f / F4, ch = f % F4;
      *reinterpret_cast<float4*>(tl + vox * TS + 4 * ch) = nxt[j];
    }
    __syncwarp();
    float xin[CIN];
#pragma unroll
    for (int i = 0; i < F4; ++i) {
      const float4 t = *reinterpret_cast<const float4*>(tl + lane * TS + 4 * i);
      xin[4 * i] = t.x, xin[4 * i + 1] = t.y, xin[4 * i + 2] = t.z, xin[4 * i + 3] = t.w;
    }
    __syncwarp();                                   // everyone has its row: the tile can take the outputs
    if (g + gstep < ngroups) fetch(g + gstep);
#pragma unroll 1
    for (int c0 = 0; c0 < COUT; c0 += 16) {
      float acc[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) acc[j] = 0.f;
#pragma unroll
      for (int ci = 0; ci < CIN; ++ci) {
        const float4* wr = reinterpret_cast<const float4*>(ws + ci * COUT + c0);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 t = wr[q];
          acc[4 * q + 0] = fmaf(xin[ci], t.x, acc[4 * q + 0]);
          acc[4 * q + 1] = fmaf(xin[ci], t.y, acc[4 * q + 1]);
          acc[4 * q + 2] = fmaf(xin[ci], t.z, acc[4 * q + 2]);
          acc[4 * q + 3] = fmaf(xin[ci], t.w, acc[4 * q + 3]);
        }
      }
#pragma unroll
      for (int j = 0; j < 16; ++j) acc[j] = activate(fmaf(acc[j], s_sc[c0 + j], s_sh[c0 + j]), act);
#pragma unroll
      for (int q = 0; q < 4; ++q)
        *reinterpret_cast<float4*>(tl + lane * TS + c0 + 4 * q) = make_float4(acc[4 * q], acc[4 * q + 1], acc[4 * q + 2], acc[4 * q + 3]);
    }
    __syncwarp();
    float4* dst = reinterpret_cast<float4*>(y + v0 * COUT);
#pragma unroll
    for (int j = 0; j < F4; ++j) {
      const int f = lane + 32 * j, vox = f / F4, ch = f % F4;
      if (vox < nv) dst[f] = *reinterpret_cast<const float4*>(tl + vox * TS + 4 * ch);
    }
  }
}

// 32 -> 32 specialisation (redir1 at full resolution: 806 MB per launch, the bigger of the two redirs).  ncu on the generic
// kernel above: l1tex throughput 85 % -- every FMA quadruple needed one broadcast LDS.128 of weights.  Here a lane keeps the weights
// of FOUR output channels for all 32 inputs in registers (32 float4) and walks the 8 voxels of its sub-row: one LDS.128 of inputs
// feeds 16 FMAs, and the results leave as coalesced STG.128 without a second transpose.
__global__ void __launch_bounds__(64) conv1x1_ndhwc_32_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                               const float* __restrict__ scale, const float* __restrict__ shift,
                                                               float* __restrict__ y, size_t V, int act) {
  constexpr int C = 32, TS = C + 4, F4 = C / 4;
  __shared__ __align__(16) float tile[2][32 * TS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c4 = 4 * (lane & 7), sub = lane >> 3;
  float4 wr[C];                                     // w[ci][c4 .. c4+3]
#pragma unroll
  for (int ci = 0; ci < C; ++ci) wr[ci] = __ldg(reinterpret_cast<const float4*>(w + ci * C + c4));
  const float4 sc = scale ? __ldg(reinterpret_cast<const float4*>(scale + c4)) : make_float4(1.f, 1.f, 1.f, 1.f);
  const float4 sh = shift ? __ldg(reinterpret_cast<const float4*>(shift + c4)) : make_float4(0.f, 0.f, 0.f, 0.f);
  float* tl = tile[warp];
  const size_t ngroups = (V + 31) / 32;
  float4 nxt[F4];
  auto fetch = [&](size_t g) {
    const size_t v0 = g * 32;
    const int nv = (int)min((size_t)32, V - v0);
    const float4* src = reinterpret_cast<const float4*>(x + v0 * C);
#pragma unroll
    for (int j = 0; j < F4; ++j) {
      const int f = lane + 32 * j;
      nxt[j] = (f / F4 < nv) ? __ldg(src + f) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  const size_t g0 = (size_t)blockIdx.x * 2 + warp, gstep = (size_t)gridDim.x * 2;
  if (g0 < ngroups) fetch(g0);
  for (size_t g = g0; g < ngroups; g += gstep) {
    const size_t v0 = g * 32;
    const int nv = (int)min((size_t)32, V - v0);
    __syncwarp();                                   // the previous group's readers are done with the tile
#pragma unroll
    for (int j = 0; j < F4; ++j) {
      const int f = lane + 32 * j;
      *reinterpret_cast<float4*>(tl + (f / F4) * TS + 4 * (f % F4)) = nxt[j];
    }
    __syncwarp();
    if (g + gstep < ngroups) fetch(g + gstep);      // next group's loads fly while this one is multiplied
    float4* dst = reinterpret_cast<float4*>(y + v0 * C);
#pragma unroll 2
    for (int j = 0; j < 8; ++j) {
      const int vox = 4 * j + sub;
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int i = 0; i < F4; ++i) {
        const float4 xv = *reinterpret_cast<const float4*>(tl + vox * TS + 4 * i);     // 8-lane broadcast, 4 rows per instruction
        const float xs[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float4 wv = wr[4 * i + k];
          acc.x = fmaf(xs[k], wv.x, acc.x), acc.y = fmaf(xs[k], wv.y, acc.y);
          acc.z = fmaf(xs[k], wv.z, acc.z), acc.w = fmaf(xs[k], wv.w, acc.w);
        }
      }
      acc.x = activate(fmaf(acc.x, sc.x, sh.x), act), acc.y = activate(fmaf(acc.y, sc.y, sh.y), act);
      acc.z = activate(fmaf(acc.z, sc.z, sh.z), act), acc.w = activate(fmaf(acc.w, sc.w, sh.w), act);
      if (vox < nv) dst[vox * F4 + (lane & 7)] = acc;                                   // 4 voxels x 128 B per instruction
    }
  }
}

// --------------------------------------------------------------------- channels-last 3x3x3 conv to ONE output channel
// The classifier head `classif*[2]` = Conv3d(32, 1, 3, 1, 1, bias=False) (gwcnet_disp_processor.py:60-70,
// psmnet_cost_processor.py:106-124) on a channels-last input: with one output channel there is no GEMM N dimension to
// feed the tensor cores, and the NCDHW CUDA-core kernel spends its time on 8-channel register tiles that are 7/8 empty.
// Here a CTA stages a (2+2) x (4+2) x (32+2) voxel halo with all 32 channels (coalesced 128-byte voxel rows, 144-byte
// padded in shared memory so LDS.128 is conflict-free) and each thread forms one output voxel's 27 x 32 dot product.
constexpr int C1_TD = 2, C1_TH = 4, C1_TW = 32;
template <int CIN>
__global__ void __launch_bounds__(256) conv3d_k3_c1_ndhwc_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                                 const float* __restrict__ scale, const float* __restrict__ shift,
                                                                 float* __restrict__ y, int D, int H, int W, int tiles_w, int tiles_h,
                                                                 int tiles_d) {
  constexpr int HD = C1_TD + 2, HH = C1_TH + 2, HW = C1_TW + 2, VS = CIN + 4, F4 = CIN / 4;
  extern __shared__ __align__(16) float c1_smem[];
  float* xs = c1_smem;                              // [HD][HH][HW][VS]
  float* ws = xs + HD * HH * HW * VS;               // [27][CIN]
  int bid = blockIdx.x;
  const int tw0 = (bid % tiles_w) * C1_TW;
  bid /= tiles_w;
  const int th0 = (bid % tiles_h) * C1_TH;
  bid /= tiles_h;
  const int td0 = (bid % tiles_d) * C1_TD;
  const int b = bid / tiles_d;
  for (int i = threadIdx.x; i < 27 * CIN; i += 256) ws[i] = __ldg(w + i);
  const float* xb = x + (size_t)b * D * H * W * CIN;
  for (int i = threadIdx.x; i < HD * HH * HW * F4; i += 256) {
    const int ch = i % F4, vox = i / F4;
    const int wx = vox % HW, hy = (vox / HW) % HH, dz = vox / (HW * HH);
    const int d = td0 - 1 + dz, h = th0 - 1 + hy, ww = tw0 - 1 + wx;
    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
    if (d >= 0 && d < D && h >= 0 && h < H && ww >= 0 && ww < W)
      t = __ldg(reinterpret_cast<const float4*>(xb + (((size_t)d * H + h) * W + ww) * CIN) + ch);
    *reinterpret_cast<float4*>(xs + vox * VS + 4 * ch) = t;
  }
  __syncthreads();
  const int tw = threadIdx.x % C1_TW, th = (threadIdx.x / C1_TW) % C1_TH, td = threadIdx.x / (C1_TW * C1_TH);
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
  for (int kd = 0; kd < 3; ++kd)
#pragma unroll
    for (int kh = 0; kh < 3; ++kh)
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        const float* xp = xs + (((td + kd) * HH + th + kh) * HW + tw + kw) * VS;
        const float* wp = ws + ((kd * 3 + kh) * 3 + kw) * CIN;
#pragma unroll
        for (int q = 0; q < F4; ++q) {
          const float4 xv = *reinterpret_cast<const float4*>(xp + 4 * q);
          const float4 wv = *reinterpret_cast<const float4*>(wp + 4 * q);
          a0 = fmaf(xv.x, wv.x, a0), a1 = fmaf(xv.y, wv.y, a1), a2 = fmaf(xv.z, wv.z, a2), a3 = fmaf(xv.w, wv.w, a3);
        }
      }
  const int d = td0 + td, h = th0 + th, ww = tw0 + tw;
  if (d < D && h < H && ww < W) {
    float r = (a0 + a1) + (a2 + a3);
    r = fmaf(r, scale ? __ldg(scale) : 1.f, shift ? __ldg(shift) : 0.f);
    y[(((size_t)b * D + d) * H + h) * W + ww] = r;
  }
}

// ------------------------------------------------------------------------------------------------------- launchers
template <typename K>
static int set_smem(K kernel, size_t bytes, const char* what) {
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) {
    set_error("%s: cannot reserve %zu bytes of shared memory: %s", what, bytes, cudaGetErrorString(e));
    return OSB_ECUDA;
  }
  return OSB_OK;
}

template <int S, int TCO, int NCG, int TD, int TH, int CI>
static int launch_conv_k3(ConvParams& p, cudaStream_t stream) {
  using C = ConvCfg<S, TCO, NCG, TD, TH, CI>;
  auto kernel = conv3d_k3_kernel<S, TCO, NCG, TD, TH, CI>;
  static PerDeviceFlag configured;
  if (!configured.here()) {
    if (int rc = set_smem(kernel, C::SMEM, "conv3d_k3")) return rc;
    configured.here() = true;
  }
  p.tiles_w = (p.Wo + C::TW - 1) / C::TW;
  p.tiles_h = (p.Ho + TH - 1) / TH;
  p.tiles_d = (p.Do + TD - 1) / TD;
  dim3 grid(p.tiles_w * p.tiles_h * p.tiles_d, (p.Cout + C::COB - 1) / C::COB, p.B);
  OSB_REQUIRE(grid.y <= 65535 && grid.z <= 65535, "conv3d_k3: grid too large");
  kernel<<<grid, C::THREADS, C::SMEM, stream>>>(p);
  count_launch();
  return check_launch("conv3d_k3_kernel");
}

template <int KS, int CI>
static int launch_deconv(ConvParams& p, cudaStream_t stream) {
  using C = DeconvCfg<KS, CI>;
  auto kernel = deconv3d_kernel<KS, CI>;
  static PerDeviceFlag configured;
  if (!configured.here()) {
    if (int rc = set_smem(kernel, C::SMEM, "deconv3d")) return rc;
    configured.here() = true;
  }
  p.tiles_w = (p.Wo + C::TW - 1) / C::TW;
  p.tiles_h = (p.Ho + C::TH - 1) / C::TH;
  p.tiles_d = (p.Do + C::TD - 1) / C::TD;
  dim3 grid(p.tiles_w * p.tiles_h * p.tiles_d, (p.Cout + C::COB - 1) / C::COB, p.B);
  OSB_REQUIRE(grid.y <= 65535 && grid.z <= 65535, "deconv3d: grid too large");
  kernel<<<grid, C::THREADS, C::SMEM, stream>>>(p);
  count_launch();
  return check_launch("deconv3d_kernel");
}

static bool aligned16(const void* q) { return q == nullptr || (reinterpret_cast<uintptr_t>(q) & 15) == 0; }


// ------------------------------------------------------------------------------- channels-last 1x1 conv over two channel slabs
// StereoBase's agg_0[0] / agg_1[0] (stereobase/hourglass.py:91-92,96-97): Conv3d(k=1) on torch.cat((up, skip), 1) without
// materialising the concat, channels-last in and out: x0 (V, C0) and x1 (V, CIN - C0) -> y (V, COUT).  Persistent CTAs of 4 warps;
// the (Cin, Cout) weight matrix sits in shared memory for the CTA's lifetime; a CTA tile is 128 voxels staged by coalesced float4
// loads of both slabs.  Thread (warp w, lane l) owns voxels l, l+32, l+64, l+96 and the output channels [w, w+1) * COUT/4: per
// four input channels it issues 4 LDS.128 of activations and COUT/4 broadcast LDS.128 of weights for 4 * COUT FMAs (FMA-bound, not
// LSU-bound: the first version -- one voxel per thread, weights through L1 -- ran at 2.4 TFLOP/s).  Outputs leave through the tile.
// H16: fp16 slabs in and fp16 out (StereoBase's fp16 hourglass route), fp32 weights and arithmetic; outputs are stored with
// cvt.rn.satfinite and a magnitude beyond 65504 bumps the tensor-core overflow counter `overflow`.
template <int CIN, int COUT, bool H16 = false>
__global__ void __launch_bounds__(128) conv1x1_ndhwc_cat_kernel(const float* __restrict__ x0, const float* __restrict__ x1, int C0,
                                                               const float* __restrict__ w, const float* __restrict__ scale,
                                                               const float* __restrict__ shift, float* __restrict__ y, size_t V,
                                                               int act, unsigned int* overflow) {
  constexpr int TS = CIN + 4;                       // tile row stride (floats): LDS.128 of a quarter warp hit distinct bank groups
  constexpr int F4 = CIN / 4, O4 = COUT / 4;
  constexpr int NC = COUT / 4;                      // output channels per warp
  static_assert(COUT <= CIN && CIN % 4 == 0 && NC % 4 == 0, "the output rides the input tile; a warp owns whole float4s");
  extern __shared__ __align__(16) float cat_smem[];
  float* ws = cat_smem;                             // [CIN][COUT]
  float* tl = cat_smem + CIN * COUT;                // [128][TS]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < CIN * COUT / 4; i += 128) reinterpret_cast<float4*>(ws)[i] = __ldg(reinterpret_cast<const float4*>(w) + i);
  const int c0f4 = C0 / 4, C1 = CIN - C0;
  const int cbase = warp * NC;
  float sc[NC], sh[NC];
#pragma unroll
  for (int j = 0; j < NC; ++j) {
    sc[j] = scale ? __ldg(scale + cbase + j) : 1.f;
    sh[j] = shift ? __ldg(shift + cbase + j) : 0.f;
  }
  const size_t ntiles = (V + 127) / 128;
  for (size_t g = blockIdx.x; g < ntiles; g += gridDim.x) {
    const size_t v0 = g * 128;
    const int nv = (int)min((size_t)128, V - v0);
    __syncthreads();                                // the previous tile's stores have read the tile (first pass: weights staged)
    for (int f = threadIdx.x; f < 128 * F4; f += 128) {
      const int vox = f / F4, ch = f % F4;
      float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
      if constexpr (H16) {
        if (vox < nv) {
          const __half* h0 = reinterpret_cast<const __half*>(x0), *h1 = reinterpret_cast<const __half*>(x1);
          const uint2 u = ch < c0f4 ? __ldg(reinterpret_cast<const uint2*>(h0 + (v0 + vox) * C0) + ch)
                                    : __ldg(reinterpret_cast<const uint2*>(h1 + (v0 + vox) * C1) + (ch - c0f4));
          const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
          t = make_float4(a.x, a.y, b.x, b.y);
        }
      } else if (vox < nv)
        t = ch < c0f4 ? __ldg(reinterpret_cast<const float4*>(x0 + (v0 + vox) * C0) + ch)
                      : __ldg(reinterpret_cast<const float4*>(x1 + (v0 + vox) * C1) + (ch - c0f4));
      *reinterpret_cast<float4*>(tl + vox * TS + 4 * ch) = t;
    }
    __syncthreads();
    float acc[4][NC];
#pragma unroll
    for (int v = 0; v < 4; ++v)
#pragma unroll
      for (int j = 0; j < NC; ++j) acc[v][j] = 0.f;
#pragma unroll 2
    for (int ci = 0; ci < CIN; ci += 4) {
      float xs[4][4];
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const float4 t = *reinterpret_cast<const float4*>(tl + (lane + 32 * v) * TS + ci);
        xs[v][0] = t.x, xs[v][1] = t.y, xs[v][2] = t.z, xs[v][3] = t.w;
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float4* wr = reinterpret_cast<const float4*>(ws + (ci + k) * COUT + cbase);
#pragma unroll
        for (int q = 0; q < NC / 4; ++q) {
          const float4 t = wr[q];
#pragma unroll
          for (int v = 0; v < 4; ++v) {
            acc[v][4 * q + 0] = fmaf(xs[v][k], t.x, acc[v][4 * q + 0]);
            acc[v][4 * q + 1] = fmaf(xs[v][k], t.y, acc[v][4 * q + 1]);
            acc[v][4 * q + 2] = fmaf(xs[v][k], t.z, acc[v][4 * q + 2]);
            acc[v][4 * q + 3] = fmaf(xs[v][k], t.w, acc[v][4 * q + 3]);
          }
        }
      }
    }
    __syncthreads();                                // every warp has read its input rows: the tile can take the outputs
#pragma unroll
    for (int v = 0; v < 4; ++v)
#pragma unroll
      for (int q = 0; q < NC / 4; ++q) {
        float4 o;
        o.x = activate(fmaf(acc[v][4 * q + 0], sc[4 * q + 0], sh[4 * q + 0]), act);
        o.y = activate(fmaf(acc[v][4 * q + 1], sc[4 * q + 1], sh[4 * q + 1]), act);
        o.z = activate(fmaf(acc[v][4 * q + 2], sc[4 * q + 2], sh[4 * q + 2]), act);
        o.w = activate(fmaf(acc[v][4 * q + 3], sc[4 * q + 3], sh[4 * q + 3]), act);
        *reinterpret_cast<float4*>(tl + (lane + 32 * v) * TS + cbase + 4 * q) = o;
      }
    __syncthreads();
    if constexpr (H16) {
      uint2* dst = reinterpret_cast<uint2*>(reinterpret_cast<__half*>(y) + v0 * COUT);
      float amax = 0.f;
      for (int f = threadIdx.x; f < 128 * O4; f += 128) {
        const int vox = f / O4, ch = f % O4;
        if (vox < nv) {
          const float4 o = *reinterpret_cast<const float4*>(tl + vox * TS + 4 * ch);
          amax = fmaxf(amax, fmaxf(fmaxf(fabsf(o.x), fabsf(o.y)), fmaxf(fabsf(o.z), fabsf(o.w))));
          uint32_t lo, hi;
          asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(o.y), "f"(o.x));
          asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(o.w), "f"(o.z));
          dst[f] = make_uint2(lo, hi);
        }
      }
      if (amax > 65504.f) atomicAdd(overflow, 1u);
    } else {
      float4* dst = reinterpret_cast<float4*>(y + v0 * COUT);
      for (int f = threadIdx.x; f < 128 * O4; f += 128) {
        const int vox = f / O4, ch = f % O4;
        if (vox < nv) dst[f] = *reinterpret_cast<const float4*>(tl + vox * TS + 4 * ch);
      }
    }
  }
}

unsigned int* tc_overflow_flag();      // api.cu: sticky fp16-range counter of the tensor-core route (tc_common.cuh)

template <int CIN, int COUT, bool H16 = false>
static int launch_conv1x1_cat(const float* x0, const float* x1, int C0, const float* w, const float* scale, const float* shift, float* y,
                              long long voxels, int act, cudaStream_t s, unsigned int* overflow = nullptr) {
  constexpr size_t smem = ((size_t)CIN * COUT + (size_t)128 * (CIN + 4)) * sizeof(float);
  static_assert(smem <= 232448, "shared memory budget of one CTA exceeded");
  auto kernel = conv1x1_ndhwc_cat_kernel<CIN, COUT, H16>;
  static PerDeviceFlag configured;
  if (!configured.here()) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      set_error("conv1x1_ndhwc_cat: cannot reserve %zu bytes of shared memory: %s", smem, cudaGetErrorString(e));
      return OSB_ECUDA;
    }
    configured.here() = true;
  }
  const long long tiles = (voxels + 127) / 128;
  const int per_sm = smem <= 113 * 1024 ? 2 : 1;
  const unsigned blocks = (unsigned)std::min<long long>(tiles, (long long)sm_count() * per_sm);
  kernel<<<blocks, 128, smem, s>>>(x0, x1, C0, w, scale, shift, y, (size_t)voxels, act, overflow);
  count_launch();
  return check_launch("conv1x1_ndhwc_cat_kernel");
}

}  // namespace osb

extern "C" {

int osb_conv3d_k3_bn_act_fwd(const float* x, const float* w_packed, const float* scale, const float* shift,
                             const float* residual, const float* gate, float* y, int B, int Cin, int Cout, int D, int H,
                             int W, int stride, int act, osb_stream_t stream) {
  using namespace osb;
  OSB_REQUIRE(x && w_packed && y, "conv3d_k3: null pointer");
  OSB_REQUIRE(B > 0 && Cin > 0 && Cout > 0 && D > 0 && H > 0 && W > 0, "conv3d_k3: empty shape");
  OSB_REQUIRE(stride == 1 || stride == 2, "conv3d_k3: stride %d not supported (1 or 2)", stride);
  OSB_REQUIRE(act >= 0 && act <= 2, "conv3d_k3: unknown activation %d", act);
  ConvParams p{};
  p.x = x, p.w = w_packed, p.scale = scale, p.shift = shift, p.residual = residual, p.gate = gate, p.y = y;
  p.B = B, p.Cin = Cin, p.Cin0 = Cin, p.Cout = Cout, p.D = D, p.H = H, p.W = W;
  p.Do = (D - 1) / stride + 1, p.Ho = (H - 1) / stride + 1, p.Wo = (W - 1) / stride + 1;
  p.act = act, p.sigmoid_out = 0;
  p.vec_ok = (p.Wo % 4 == 0) && aligned16(y) && aligned16(residual) && aligned16(gate);
  cudaStream_t s = (cudaStream_t)stream;
  if (Cout < 8) {  // classifier heads (32 -> 1): one channel per thread
    return stride == 1 ? launch_conv_k3<1, 1, 1, 4, 4, 8>(p, s) : launch_conv_k3<2, 1, 1, 2, 4, 4>(p, s);
  }
  if (Cout % 32 != 0 && Cout % 24 == 0) {  // StereoBase widths 24/48/96/144
    return stride == 1 ? launch_conv_k3<1, 8, 3, 4, 4, 8>(p, s) : launch_conv_k3<2, 8, 3, 2, 4, 4>(p, s);
  }
  return stride == 1 ? launch_conv_k3<1, 8, 4, 4, 4, 8>(p, s) : launch_conv_k3<2, 8, 4, 2, 4, 4>(p, s);
}

int osb_deconv3d_bn_act_fwd(const float* x, const float* w_packed, const float* scale, const float* shift,
                            const float* residual, float* y, int B, int Cin, int Cout, int D, int H, int W, int kernel,
                            int act, osb_stream_t stream) {
  using namespace osb;
  OSB_REQUIRE(x && w_packed && y, "deconv3d: null pointer");
  OSB_REQUIRE(B > 0 && Cin > 0 && Cout > 0 && D > 0 && H > 0 && W > 0, "deconv3d: empty shape");
  OSB_REQUIRE(kernel == 3 || kernel == 4, "deconv3d: kernel %d not supported (3 or 4)", kernel);
  OSB_REQUIRE(act >= 0 && act <= 2, "deconv3d: unknown activation %d", act);
  ConvParams p{};
  p.x = x, p.w = w_packed, p.scale = scale, p.shift = shift, p.residual = residual, p.gate = nullptr, p.y = y;
  p.B = B, p.Cin = Cin, p.Cin0 = Cin, p.Cout = Cout, p.D = D, p.H = H, p.W = W;
  p.Do = 2 * D, p.Ho = 2 * H, p.Wo = 2 * W;
  p.act = act, p.sigmoid_out = 0;
  p.vec_ok = (p.Wo % 4 == 0) && aligned16(y) && aligned16(residual);
  cudaStream_t s = (cudaStream_t)stream;
  return kernel == 3 ? launch_deconv<3, 8>(p, s) : launch_deconv<4, 8>(p, s);
}

int osb_conv3d_1x1_bn_act_fwd(const float* x0, const float* x1, int Cin0, const float* w_packed, const float* scale,
                              const float* shift, const float* residual, const float* gate, float* y, int B, int Cin,
                              int Cout, int D, int H, int W, int act, int sigmoid_out, osb_stream_t stream) {
  using namespace osb;
  OSB_REQUIRE(x0 && w_packed && y, "conv3d_1x1: null pointer");
  OSB_REQUIRE(B > 0 && Cin > 0 && Cout > 0 && D > 0 && H > 0 && W > 0, "conv3d_1x1: empty shape");
  OSB_REQUIRE(Cin0 > 0 && Cin0 <= Cin && (Cin0 == Cin || x1 != nullptr), "conv3d_1x1: bad channel split %d of %d", Cin0, Cin);
  OSB_REQUIRE(act >= 0 && act <= 3, "conv3d_1x1: unknown activation %d", act);
  ConvParams p{};
  p.x = x0, p.x1 = x1, p.w = w_packed, p.scale = scale, p.shift = shift, p.residual = residual, p.gate = gate, p.y = y;
  p.B = B, p.Cin = Cin, p.Cin0 = Cin0, p.Cout = Cout, p.D = D, p.H = H, p.W = W;
  p.Do = D, p.Ho = H, p.Wo = W;
  p.act = act, p.sigmoid_out = sigmoid_out;
  p.vec_ok = (W % 4 == 0) && aligned16(y) && aligned16(residual) && aligned16(gate) && aligned16(x0) && aligned16(x1);
  const size_t octs = (size_t)D * H * ((W + 7) / 8);
  dim3 grid((unsigned)((octs + 63) / 64), (Cout + 31) / 32, B);
  OSB_REQUIRE(grid.y <= 65535 && grid.z <= 65535, "conv3d_1x1: grid too large");
  conv3d_1x1_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(p);
  count_launch();
  return check_launch("conv3d_1x1_kernel");
}

int osb_conv1x1_ndhwc_cat_fwd(const float* x0, const float* x1, int C0, int C1, const float* w_packed, const float* scale,
                              const float* shift, float* y, long long voxels, int Cout, int act, osb_stream_t stream) {
  using namespace osb;
  OSB_REQUIRE(x0 && w_packed && y && (x1 || C1 == 0), "conv1x1_ndhwc_cat: null pointer");
  OSB_REQUIRE(voxels > 0 && C0 > 0 && C1 >= 0 && C0 % 4 == 0 && C1 % 4 == 0, "conv1x1_ndhwc_cat: bad shape");
  OSB_REQUIRE(act >= 0 && act <= 2, "conv1x1_ndhwc_cat: unknown activation %d", act);
  OSB_REQUIRE(aligned16(x0) && aligned16(x1) && aligned16(y) && aligned16(w_packed), "conv1x1_ndhwc_cat: pointers must be 16-byte aligned");
  cudaStream_t s = (cudaStream_t)stream;
  const int Cin = C0 + C1;
  if (Cin == 192 && Cout == 96) return launch_conv1x1_cat<192, 96>(x0, x1, C0, w_packed, scale, shift, y, voxels, act, s);
  if (Cin == 128 && Cout == 64) return launch_conv1x1_cat<128, 64>(x0, x1, C0, w_packed, scale, shift, y, voxels, act, s);
  set_error("conv1x1_ndhwc_cat: unsupported channels %d + %d -> %d (192 -> 96 and 128 -> 64 are instantiated)", C0, C1, Cout);
  return OSB_EUNSUPPORTED;
}

int osb_conv1x1_ndhwc_cat_h16_fwd(const void* x0, const void* x1, int C0, int C1, const float* w_packed, const float* scale,
                                  const float* shift, float* y, long long voxels, int Cout, int act, osb_stream_t stream) {
  using namespace osb;
  OSB_REQUIRE(x0 && x1 && w_packed && y, "conv1x1_ndhwc_cat_h16: null pointer");
  OSB_REQUIRE(voxels > 0 && C0 > 0 && C1 > 0 && C0 % 4 == 0 && C1 % 4 == 0, "conv1x1_ndhwc_cat_h16: bad shape");
  OSB_REQUIRE(act >= 0 && act <= 2, "conv1x1_ndhwc_cat_h16: unknown activation %d", act);
  OSB_REQUIRE((reinterpret_cast<uintptr_t>(x0) & 7) == 0 && (reinterpret_cast<uintptr_t>(x1) & 7) == 0 &&
                  (reinterpret_cast<uintptr_t>(y) & 7) == 0 && aligned16(w_packed),
              "conv1x1_ndhwc_cat_h16: x0 / x1 / y must be 8-byte, w 16-byte aligned");
  unsigned int* flag = tc_overflow_flag();
  OSB_REQUIRE(flag, "conv1x1_ndhwc_cat_h16: cannot allocate the overflow flag");
  cudaStream_t s = (cudaStream_t)stream;
  const int Cin = C0 + C1;
  const float* a = static_cast<const float*>(x0);
  const float* b = static_cast<const float*>(x1);
  float* o = y;
  if (Cin == 192 && Cout == 96) return launch_conv1x1_cat<192, 96, true>(a, b, C0, w_packed, scale, shift, o, voxels, act, s, flag);
  if (Cin == 128 && Cout == 64) return launch_conv1x1_cat<128, 64, true>(a, b, C0, w_packed, scale, shift, o, voxels, act, s, flag);
  set_error("conv1x1_ndhwc_cat_h16: unsupported channels %d + %d -> %d (192 -> 96 and 128 -> 64 are instantiated)", C0, C1, Cout);
  return OSB_EUNSUPPORTED;
}

int osb_conv1x1_ndhwc_fwd(const float* x, const float* w_packed, const float* scale, const float* shift, float* y,
                          long long voxels, int Cin, int Cout, int act, osb_stream_t stream) {
  using namespace osb;
  OSB_REQUIRE(x && w_packed && y, "conv1x1_ndhwc: null pointer");
  OSB_REQUIRE(voxels > 0, "conv1x1_ndhwc: empty input");
  OSB_REQUIRE(act >= 0 && act <= 2, "conv1x1_ndhwc: unknown activation %d", act);
  OSB_REQUIRE(aligned16(x) && aligned16(y), "conv1x1_ndhwc: pointers must be 16-byte aligned");
  const long long groups = (voxels + 31) / 32;
  const unsigned blocks = (unsigned)std::min<long long>((groups + 1) / 2, 148ll * 16);   // 2 warps per CTA, grid-stride over 32-voxel groups
  cudaStream_t s = (cudaStream_t)stream;
  if (Cin == 32 && Cout == 32) conv1x1_ndhwc_32_kernel<<<blocks, 64, 0, s>>>(x, w_packed, scale, shift, y, (size_t)voxels, act);
  else if (Cin == 64 && Cout == 64) conv1x1_ndhwc_kernel<64, 64><<<blocks, 64, 0, s>>>(x, w_packed, scale, shift, y, (size_t)voxels, act);
  else {
    set_error("conv1x1_ndhwc: unsupported channels %d -> %d (32->32 and 64->64 are instantiated)", Cin, Cout);
    return OSB_EUNSUPPORTED;
  }
  count_launch();
  return check_launch("conv1x1_ndhwc_kernel");
}

int osb_conv3d_k3_c1_ndhwc_fwd(const float* x_ndhwc, const float* w_taps, const float* scale, const float* shift, float* y, int B,
                               int Cin, int D, int H, int W, osb_stream_t stream) {
  using namespace osb;
  OSB_REQUIRE(x_ndhwc && w_taps && y, "conv3d_k3_c1_ndhwc: null pointer");
  OSB_REQUIRE(B > 0 && D > 0 && H > 0 && W > 0, "conv3d_k3_c1_ndhwc: empty shape");
  OSB_REQUIRE(aligned16(x_ndhwc) && aligned16(w_taps), "conv3d_k3_c1_ndhwc: pointers must be 16-byte aligned");
  if (Cin != 32) {
    set_error("conv3d_k3_c1_ndhwc: Cin = %d unsupported (32 is instantiated)", Cin);
    return OSB_EUNSUPPORTED;
  }
  const int tiles_w = (W + C1_TW - 1) / C1_TW, tiles_h = (H + C1_TH - 1) / C1_TH, tiles_d = (D + C1_TD - 1) / C1_TD;
  const long long blocks = (long long)B * tiles_d * tiles_h * tiles_w;
  OSB_REQUIRE(blocks < (1ll << 31), "conv3d_k3_c1_ndhwc: too many tiles");
  constexpr size_t smem = ((size_t)(C1_TD + 2) * (C1_TH + 2) * (C1_TW + 2) * (32 + 4) + 27 * 32) * sizeof(float);
  auto kernel = conv3d_k3_c1_ndhwc_kernel<32>;
  static PerDeviceFlag configured;
  if (!configured.here()) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      set_error("conv3d_k3_c1_ndhwc: cannot reserve %zu bytes of shared memory: %s", smem, cudaGetErrorString(e));
      return OSB_ECUDA;
    }
    configured.here() = true;
  }
  kernel<<<(unsigned)blocks, 256, smem, (cudaStream_t)stream>>>(x_ndhwc, w_taps, scale, shift, y, D, H, W, tiles_w, tiles_h, tiles_d);
  count_launch();
  return check_launch("conv3d_k3_c1_ndhwc_kernel");
}
}
