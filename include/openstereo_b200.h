/*
 * openstereo_b200.h -- C ABI of the B200-native cost-volume hot path for OpenStereo.
 *
 * Drop-in boundary.  The reference (XiandaGuo/OpenStereo) has no operator registry: the hot path is
 * a set of plain Python callables on torch.Tensor (SURVEY.md section 8b).  The reference's own
 * convention for native ops is "a compiled extension called from a thin Python wrapper on the
 * current CUDA stream" (stereo/libs/AANet/deform_conv/deform_conv.py:9,44-56;
 * stereo/modeling/models/nmrf/ops/functions/ms_deform_attn_func.py:11-47).  This header is that
 * extension's surface, expressed as a C ABI: plain device pointers, sizes and a stream handle --
 * no torch types.  openstereo_b200/ops.py binds it with ctypes; INTEGRATION.md shows the stub a
 * reference maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to dense fp32 data in the reference's layout
 *     (NCHW features, NCDHW volumes), unless the name ends in _host;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream);
 *   - inputs are borrowed and never written; outputs are caller-allocated;
 *   - return value 0 = success, otherwise an OSB_E* code; osb_last_error() returns a
 *     thread-local message.  Nothing falls back to a CPU path: without a CUDA device every
 *     compute entry point fails with OSB_ECUDA.
 */
#ifndef OPENSTEREO_B200_H_
#define OPENSTEREO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OSB_OK 0
#define OSB_EINVAL 1  /* bad shape / argument (the reference raises AssertionError / ValueError) */
#define OSB_ECUDA 2   /* CUDA runtime / driver error, incl. "no device" */
#define OSB_EUNSUPPORTED 3

#define OSB_ACT_NONE 0
#define OSB_ACT_RELU 1
#define OSB_ACT_LEAKY 2 /* LeakyReLU(0.01), nn.LeakyReLU default used by StereoBase */
#define OSB_ACT_RELU6 3 /* nn.ReLU6 of LightStereo's MobileV2Residual; accepted by the CUDA-core 1x1, depthwise and 2D kernels */

typedef void* osb_stream_t;

int osb_abi_version(void);
const char* osb_last_error(void);
/* Number of kernels this library has launched in this process (bench.py reports it). */
uint64_t osb_launch_count(void);
/* fp16 range guard of the tensor-core convolutions.  They compute every fp32 product as three kind::f16 MMAs on operands split
 * into fp16 (hi, lo) pairs (csrc/tc_common.cuh): activations are staged as x * 16, so |x| must stay below 65504 / 16 = 4094
 * (weights are pre-scaled per output channel on the host and cannot overflow).  Conversions saturate and every loader thread
 * that met a larger value increments a sticky per-device counter.  osb_tc_overflow_count copies it to *count (host memory),
 * optionally resets it, and synchronises `stream`; osb_tc_overflow_flag returns its device address (for an asynchronous read). */
int osb_tc_overflow_count(osb_stream_t stream, int reset, unsigned int* count);
/* Asynchronous variant: enqueue a 4-byte copy of the counter into PINNED host memory on `stream` and return at once (the caller
 * reads *host_pinned after an event recorded behind it has completed; the Python engines do that at the start of their next call). */
int osb_tc_overflow_poll(osb_stream_t stream, unsigned int* host_pinned);
const unsigned int* osb_tc_overflow_flag(void);
/* Expected round-towards-zero loss per accumulating tcgen05.mma, undone by the conv epilogues (csrc/tc_common.cuh: rz_kappa;
 * DESIGN.md section 4.3).  Process-wide; returns the previous value; 0 switches the correction off.  The default is the
 * constant measured on B200 (profiles/r2_parity_bisect.md); the setter exists for that calibration. */
float osb_set_rz_kappa(float kappa);

/* ---------------------------------------------------------------- cost-volume constructors --- */

/* build_gwc_volume(refimg_fea, targetimg_fea, maxdisp, num_groups)
 *   stereo/modeling/cost_volume/cost_volume.py:68-78, gwcnet/gwcnet_cost_processor.py:22-39
 * ref,tgt: (B,C,H,W) -> out: (B,G,D,H,W); out[b,g,d,h,w] = mean_k ref[b,gK+k,h,w]*tgt[b,gK+k,h,w-d]
 * for w >= d, exact 0 otherwise.  C % G != 0 -> OSB_EINVAL (reference: assert, cost_volume.py:61). */
int osb_gwc_volume_fwd(const float* ref, const float* tgt, float* out, int B, int C, int H, int W,
                       int D, int G, osb_stream_t stream);

/* build_concat_volume(refimg_fea, targetimg_fea, maxdisp)   cost_volume.py:81-92
 * == cat_fms(start_disp=0, dilation=1)                       psmnet/psmnet_cost_processor.py:9-50
 * out: (B,2C,D,H,W).  mask_left=1: canonical form (left half zero for w<d);
 * mask_left=0: IGEV-family form (igev/submodule.py:216-227). */
int osb_concat_volume_fwd(const float* ref, const float* tgt, float* out, int B, int C, int H,
                          int W, int D, int mask_left, osb_stream_t stream);

/* GwcVolumeCostProcessor.forward: torch.cat((gwc, concat), 1) written in ONE pass
 *   gwcnet/gwcnet_cost_processor.py:55-68, stereobase/stereobase_gru.py:142-160
 * out: (B, G + 2*Cc, D, H, W). */
int osb_gwc_concat_volume_fwd(const float* ref_gwc, const float* tgt_gwc, const float* ref_cat,
                              const float* tgt_cat, float* out, int B, int Cg, int Cc, int H, int W,
                              int D, int G, osb_stream_t stream);

/* correlation_volume(left, right, max_disp)   cost_volume.py:32-41   out: (B,D,H,W) */
int osb_corr_volume_fwd(const float* left, const float* right, float* out, int B, int C, int H,
                        int W, int D, osb_stream_t stream);

/* ------------------------------------------------------------------------ soft-argmin tails --- */

/* softmax over D fused with the expectation (one pass over the cost):
 *   disparity_regression(F.softmax(x,1), D)    disp_pred/disp_regression.py:8-12,
 *                                              gwcnet/gwcnet_disp_processor.py:22-26
 *   FasterSoftArgmin.forward                   psmnet/psmnet_disp_processor.py:51-74
 * cost: (B,D,H,W) -> out: (B,H,W); sample value of bin d is start + d*step; cost is multiplied by
 * alpha first; normalize=0 skips the softmax (sum_d cost*value). */
int osb_softargmin_fwd(const float* cost, float* out, int B, int D, int H, int W, float alpha,
                       float start, float step, int normalize, osb_stream_t stream);

/* F.interpolate(cost,[D,H,W],'trilinear',align_corners) -> softmax(dim=1) -> expectation, fused;
 * the upsampled (B,D,H,W) tensor is never materialised.
 *   gwcnet/gwcnet_disp_processor.py:129-133 (align_corners=0)
 *   psmnet/psmnet_cost_processor.py:203-214 + psmnet_disp_processor.py:64-73 (align_corners=1)
 * cost: (B,1,Dl,Hl,Wl) -> out: (B,H,W). */
int osb_upsample_softargmin_fwd(const float* cost, float* out, int B, int Dl, int Hl, int Wl, int D,
                                int H, int W, int align_corners, osb_stream_t stream);

/* epe_metric partial sums   stereo/evaluation/metric_per_image.py:32-41 with the eval mask of
 * trainer_template.py:288 (0 < gt < maxdisp).  out: (B,2) = {sum |pred-gt| over valid, #valid}. */
int osb_epe_partial_fwd(const float* pred, const float* gt, float* out, int B, int HW, float maxdisp,
                        osb_stream_t stream);

/* ------------------------------------------------------------------------- 3D aggregation ----- */

/* Conv3d(k=3, pad=1, stride in {1,2}, bias=False) + folded eval BatchNorm3d + optional residual +
 * activation + optional channel gate:
 *     y = act( conv(x) * scale[co] + shift[co] + residual ) * gate[b,co,h,w]
 *   convbn_3d gwcnet/hourglass.py:5-16; conv3d_bn(_relu) psmnet/submodule.py:68-83,160-177;
 *   BasicConv3d common/basic_block_3d.py:5-20; FeatureAtt stereobase/igev_blocks.py:35-48.
 * x: (B,Cin,D,H,W); w_packed: (Cin,27,Cout) = weight.permute(1,2,3,4,0) of the (Cout,Cin,3,3,3)
 * parameter; scale/shift: (Cout) or NULL (= 1 / 0); residual: like y or NULL;
 * gate: (B,Cout,Ho,Wo) already sigmoid-ed, or NULL.  y: (B,Cout,Do,Ho,Wo), Do=(D-1)/stride+1. */
int osb_conv3d_k3_bn_act_fwd(const float* x, const float* w_packed, const float* scale,
                             const float* shift, const float* residual, const float* gate, float* y,
                             int B, int Cin, int Cout, int D, int H, int W, int stride, int act,
                             osb_stream_t stream);

/* ConvTranspose3d(stride=2, bias=False) + folded BN + residual + activation.
 *   kernel=3: padding=1, output_padding=1 (gwcnet/hourglass.py:35-41, psmnet deconv3d_bn)
 *   kernel=4: padding=1                   (stereobase/hourglass.py:39-49)
 * x: (B,Cin,D,H,W) -> y: (B,Cout,2D,2H,2W); w_packed: (Cin,k^3,Cout) = weight.permute(0,2,3,4,1)
 * of the (Cin,Cout,k,k,k) parameter. */
int osb_deconv3d_bn_act_fwd(const float* x, const float* w_packed, const float* scale,
                            const float* shift, const float* residual, float* y, int B, int Cin,
                            int Cout, int D, int H, int W, int kernel, int act, osb_stream_t stream);

/* Conv3d(k=1) + folded BN + residual + activation + gate (redir1/2 gwcnet/hourglass.py:43-44,
 * agg_0[0]/agg_1[0] stereobase/hourglass.py:51-66).  Also serves the 2D 1x1 convs of FeatureAtt
 * with D=1.  x may be given as two channel slabs (x0: Cin0 channels, x1: Cin-Cin0 channels) so the
 * torch.cat of stereobase/hourglass.py:91,96 is never materialised; x1 NULL -> single input.
 * w_packed: (Cin,Cout).  sigmoid_out=1 applies a final sigmoid (FeatureAtt gate). */
int osb_conv3d_1x1_bn_act_fwd(const float* x0, const float* x1, int Cin0, const float* w_packed,
                              const float* scale, const float* shift, const float* residual,
                              const float* gate, float* y, int B, int Cin, int Cout, int D, int H,
                              int W, int act, int sigmoid_out, osb_stream_t stream);

/* ------------------------------------------------------- tensor-core (tcgen05) variant of the 3x3x3 conv ----- */

/* Same operator as osb_conv3d_k3_bn_act_fwd (stride 1) for the full-resolution layers, computed on the 5th-gen tensor
 * cores with 3xFP16 operand splitting (fp32-accurate, see csrc/tc_common.cuh, conv3d_tc.cu, conv3d_tcg.cu).  Supported shapes:
 * osb_conv3d_tc_supported / osb_conv3d_tc_kc.  x is CHANNELS-LAST (B,D,H,W,Cin) fp32; w_split is the host-split fp16 weight
 * tensor [3 kd][Cin/kc][3 kh][3*Cout (kw-major)][kc hi | kc lo] of w * 2^e_c (ops.pack_tc_weight; e_c per output channel);
 * `scale` (REQUIRED here, Cout floats) must already contain the exact inverse 2^-(e_c + 4) times the folded-BN scale
 * (TcWeight.eff_scale).  y and residual are fp32, NCDHW or NDHWC according to out_ndhwc / res_ndhwc. */
int osb_conv3d_tc_supported(int Cin, int Cout, int W, int stride);
/* General widths: every W >= OSB_TC_MIN_WIDTH that has no whole-row variant is served by 128-column tiles of one image row with a
 * one-column halo (conv3d_tcg.cu / conv3d_tcs2.cu / conv3d_tcdc.cu, GW instantiations): 240 (the reference's 544x960 timing shape,
 * tools/measure.py:32), 312 (KITTI), 160 (IGEV) ... -- stride 1: Cout 32|64|128; stride 2: Cout 64|128; transposed: Cout 32|64. */
#define OSB_TC_MIN_WIDTH 24
int osb_tc_general_width(int W);
/* K chunk (16 or 32 input channels per operand tile) the weight tensor must be packed with; 0 = unsupported shape.
 * Variants: W=128/Cout=32 (kc 32); W=64/Cout=64, W=32/Cout=64|128 (kc 16, M tile = 128/W image rows); general widths (kc 16). */
int osb_conv3d_tc_kc(int Cin, int Cout, int W, int stride);
int osb_conv3d_k3_tc_fwd(const float* x_ndhwc, const void* w_split, const float* scale, const float* shift,
                         const float* residual, float* y, int B, int Cin, int Cout, int D, int H, int W, int act,
                         int out_ndhwc, int res_ndhwc, osb_stream_t stream);
/* Same with FeatureAtt's gate fused: y = act(bn(conv(x)) + residual) * gate, gate_nhwc (B,H,W,Cout) = sigmoid(att) broadcast over D
 * (stereobase/hourglass.py:80-99, igev_blocks.py:35-48).  Channels-last y / residual, 16-channel-chunk variants only. */
int osb_conv3d_k3_tc_gate_fwd(const float* x_ndhwc, const void* w_split, const float* scale, const float* shift,
                              const float* residual, const float* gate_nhwc, float* y, int B, int Cin, int Cout, int D, int H, int W,
                              int act, osb_stream_t stream);
/* Same, reading an NCDHW input (B,Cin,D,H,W) -- the cost volume exactly as osb_gwc_concat_volume_fwd / build_*_volume return it --
 * so the first aggregation layer needs no layout-conversion pass.  Served by the W = 128 variant (Cout = 32 or <= 16). */
int osb_conv3d_k3_tc_ncdhw_fwd(const float* x_ncdhw, const void* w_split, const float* scale, const float* shift,
                               const float* residual, float* y, int B, int Cin, int Cout, int D, int H, int W, int act,
                               int out_ndhwc, int res_ndhwc, osb_stream_t stream);
/* Stride-2 variant (the down-sampling convs of the hourglasses): x (B,D,H,W,Cin) channels-last with even D,H,W ->
 * y (B,Cout,D/2,H/2,W/2) or channels-last.  w_split like above but with the kw slices stored in the order (1,0,2)
 * (ops.pack_tc_weight(..., kw_order=(1,0,2))), 16-channel K chunks.  Supported: W=128/Cout=64, W=64/Cout=64|128. */
int osb_conv3d_s2_tc_supported(int Cin, int Cout, int D, int H, int W);
int osb_conv3d_k3_s2_tc_fwd(const float* x_ndhwc, const void* w_split, const float* scale, const float* shift,
                            const float* residual, float* y, int B, int Cin, int Cout, int D, int H, int W, int act,
                            int out_ndhwc, int res_ndhwc, osb_stream_t stream);
/* ConvTranspose3d(k=3, stride=2, padding=1, output_padding=1) on the tensor cores: x (B,D,H,W,Cin) channels-last ->
 * y (B,Cout,2D,2H,2W) or channels-last.  w_split = ops.pack_tc_deconv_weight(weight): the (Cin,Cout,3,3,3) parameter split
 * hi/lo (fp16), 16-channel K chunks, kw slices stored as (1,2,0).  Supported: W=32/Cout=64 (conv5), W=64/Cout=32 (conv6). */
int osb_deconv3d_tc_supported(int Cin, int Cout, int W);
int osb_deconv3d_k3_tc_fwd(const float* x_ndhwc, const void* w_split, const float* scale, const float* shift,
                           const float* residual, float* y, int B, int Cin, int Cout, int D, int H, int W, int act,
                           int out_ndhwc, int res_ndhwc, osb_stream_t stream);
/* ConvTranspose3d(k=4, stride=2, padding=1) on the tensor cores -- BasicDeconv3d of StereoBase's hourglass
 * (stereobase/hourglass.py:35-60 conv3_up / conv2_up / conv1_up): x (B,D,H,W,Cin) channels-last -> y (B,2D,2H,2W,Cout) channels-last
 * or (B,cout_real,2D,2H,2W).  w_split = ops.pack_tc_deconv_weight of the (Cin,Cout,4,4,4) parameter, kw slices stored as (1,3,2,0).
 * Cout is the PACKED channel count (zero-padded channel plans: 24 -> 32, 48 -> 64); cout_real <= Cout real channels are written /
 * added when the output / residual is NCDHW.  Supported: W=32/Cout=64, W=64/Cout=32, W=16/Cout=64|32. */
int osb_deconv3d_k4_tc_supported(int Cin, int Cout, int W);
int osb_deconv3d_k4_tc_fwd(const float* x_ndhwc, const void* w_split, const float* scale, const float* shift,
                           const float* residual, float* y, int B, int Cin, int Cout, int cout_real, int D, int H, int W, int act,
                           int out_ndhwc, int res_ndhwc, osb_stream_t stream);
/* Channel-SLICE variants (suffix _cs): the launch computes Cout consecutive channels of a wider channels-last tensor whose voxels
 * hold `ystride` >= Cout floats; y (and residual / gate_nhwc) point at the slice's first channel.  Channel plans whose kw-stacked
 * N = 3*Cout (4*Cout for the k4 transposed conv) exceeds what one CTA can hold -- StereoBase's 6c = 144 (run as 160 = 96 + 64) --
 * are produced by two launches over output-channel slices of separately packed weights.  Channels-last in and out. */
int osb_conv3d_k3_tc_cs_fwd(const float* x_ndhwc, const void* w_split, const float* scale, const float* shift, const float* residual,
                            const float* gate_nhwc, float* y, int B, int Cin, int Cout, int D, int H, int W, int act, int ystride,
                            osb_stream_t stream);
int osb_conv3d_k3_s2_tc_cs_fwd(const float* x_ndhwc, const void* w_split, const float* scale, const float* shift, float* y, int B,
                               int Cin, int Cout, int D, int H, int W, int act, int ystride, osb_stream_t stream);
int osb_deconv3d_k4_tc_cs_fwd(const float* x_ndhwc, const void* w_split, const float* scale, const float* shift, float* y, int B,
                              int Cin, int Cout, int D, int H, int W, int act, int ystride, osb_stream_t stream);
/* Channels-last 1x1x1 conv over the channel concatenation of two tensors (torch.cat((up, skip), 1) -> Conv3d(k=1) of
 * stereobase/hourglass.py:91-92,96-97, never materialised): x0 (voxels,C0), x1 (voxels,C1) or NULL -> y (voxels,Cout);
 * w_packed (C0+C1, Cout).  192 -> 96 and 128 -> 64. */
int osb_conv1x1_ndhwc_cat_fwd(const float* x0, const float* x1, int C0, int C1, const float* w_packed, const float* scale,
                              const float* shift, float* y, long long voxels, int Cout, int act, osb_stream_t stream);
/* ---- fp16 activations (suffix _h16): StereoBase's hourglass under torch.autocast(float16), opt-in (aggregation.StereoBaseAggregation
 * precision="fp16", DESIGN.md section 4.11).  Same operators as the fp32 siblings above, with these differences:
 *   - x / x0 / x1 and y hold fp16 values: inputs are `const void*`, the output keeps the ABI's `float*` spelling but receives
 *     fp16 elements (2 bytes each); scale, shift and gate_nhwc stay fp32, w_split stays the fp16 pack;
 *   - w_split is a hi-only pack (ops.pack_tc_weight(..., h16=True)): the lo halves of its rows are zero and never read, and
 *     `scale` carries 2^-e_c times the folded-BN scale (no activation scale) -- every product is ONE kind::f16 MMA of fp16 operands;
 *   - folded BN, activation and gate are applied in fp32, the result is stored with cvt.rn.satfinite: |y| > 65504 saturates and
 *     increments the sticky counter of osb_tc_overflow_count / osb_tc_overflow_poll;
 *   - channels-last x and y (deconv: NCDHW y with cout_real allowed when out_ndhwc = 0), no residual;
 *   - shapes: the whole-row variants of StereoBase's hourglass at W' = 128, see the _h16_supported queries (W = input width):
 *     stride 1: W=64/Cout=64, W=32/Cout=96, W=16/Cout=96|64 (channel slices); stride 2: W=128/Cout=64, W=64/Cout=96, W=32/Cout=96|64;
 *     k4 transposed conv: osb_deconv3d_k4_tc_supported.  x, w_split and gate_nhwc 16-byte aligned, y 8-byte aligned. */
int osb_conv3d_tc_h16_supported(int Cin, int Cout, int W);
int osb_conv3d_s2_tc_h16_supported(int Cin, int Cout, int D, int H, int W);
int osb_conv3d_k3_tc_h16_fwd(const void* x_ndhwc, const void* w_split, const float* scale, const float* shift, float* y, int B, int Cin,
                             int Cout, int D, int H, int W, int act, osb_stream_t stream);
int osb_conv3d_k3_tc_gate_h16_fwd(const void* x_ndhwc, const void* w_split, const float* scale, const float* shift, const float* gate_nhwc,
                                  float* y, int B, int Cin, int Cout, int D, int H, int W, int act, osb_stream_t stream);
int osb_conv3d_k3_s2_tc_h16_fwd(const void* x_ndhwc, const void* w_split, const float* scale, const float* shift, float* y, int B, int Cin,
                                int Cout, int D, int H, int W, int act, osb_stream_t stream);
int osb_deconv3d_k4_tc_h16_fwd(const void* x_ndhwc, const void* w_split, const float* scale, const float* shift, float* y, int B, int Cin,
                               int Cout, int cout_real, int D, int H, int W, int act, int out_ndhwc, osb_stream_t stream);
/* channel slices (see the _cs_fwd siblings); gate_nhwc (B,H,W,ystride) fp32 pre-offset to the slice, or NULL */
int osb_conv3d_k3_tc_cs_h16_fwd(const void* x_ndhwc, const void* w_split, const float* scale, const float* shift, const float* gate_nhwc,
                                float* y, int B, int Cin, int Cout, int D, int H, int W, int act, int ystride, osb_stream_t stream);
int osb_conv3d_k3_s2_tc_cs_h16_fwd(const void* x_ndhwc, const void* w_split, const float* scale, const float* shift, float* y, int B,
                                   int Cin, int Cout, int D, int H, int W, int act, int ystride, osb_stream_t stream);
int osb_deconv3d_k4_tc_cs_h16_fwd(const void* x_ndhwc, const void* w_split, const float* scale, const float* shift, float* y, int B,
                                  int Cin, int Cout, int D, int H, int W, int act, int ystride, osb_stream_t stream);
/* osb_conv1x1_ndhwc_cat_fwd with fp16 slabs x0, x1 (8-byte aligned) and fp16 y; fp32 weights and arithmetic, saturating stores
 * counted like the tensor-core convs'. */
int osb_conv1x1_ndhwc_cat_h16_fwd(const void* x0, const void* x1, int C0, int C1, const float* w_packed, const float* scale,
                                  const float* shift, float* y, long long voxels, int Cout, int act, osb_stream_t stream);
/* Channels-last 1x1x1 conv + folded BN + activation (the redir branches when the aggregation runs channels-last):
 * x (voxels, Cin) -> y (voxels, Cout); w_packed (Cin, Cout).  32->32 and 64->64. */
int osb_conv1x1_ndhwc_fwd(const float* x, const float* w_packed, const float* scale, const float* shift, float* y,
                          long long voxels, int Cin, int Cout, int act, osb_stream_t stream);
/* Classifier head Conv3d(Cin, 1, 3, 1, 1) (gwcnet_disp_processor.py:60-70 classif*[2]) on a channels-last input:
 * x (B,D,H,W,Cin) -> y (B,1,D,H,W) = (B,D,H,W); w_taps (27, Cin) tap-major [kd][kh][kw][ci]; scale/shift: optional 1-element
 * arrays (folded BN / bias).  Cin = 32. */
int osb_conv3d_k3_c1_ndhwc_fwd(const float* x_ndhwc, const float* w_taps, const float* scale, const float* shift, float* y, int B,
                               int Cin, int D, int H, int W, osb_stream_t stream);
/* 3x3 Conv2d (stride 1, padding = dilation, dilation 1 or 2) + folded BN + residual + activation on the tensor cores, for the
 * residual blocks of the PSMNet-style feature extractor (BasicBlock gwcnet_backbone.py:13-35, layers :38-60;
 * psmnet/submodule.py:219-243): x (B,H,W,Cin) channels-last, w_split = the 3x3x3 tensor-core packing of the 2D weight placed
 * at kd = 1, y (B,H,W,Cout) or (B,Cout,H,W).  dilation 1 = osb_conv3d_k3_tc_fwd with D = 1; dilation 2: W = 128, Cout = 128.
 * osb_conv2d_tc_kc returns the K chunk of the serving kernel (0 = unsupported). */
int osb_conv2d_tc_kc(int Cin, int Cout, int W, int dilation);
int osb_conv2d_k3_tc_fwd(const float* x_nhwc, const void* w_split, const float* scale, const float* shift, const float* residual,
                         float* y, int B, int Cin, int Cout, int H, int W, int dilation, int act, int out_nhwc, int res_nhwc,
                         osb_stream_t stream);
/* ---- SURVEY.md section 8(f) row 4: remaining volume / regression flavours of the model zoo -------------------------------------
 * osb_gwc_volume_sum_fwd: osb_gwc_volume_fwd with a plain SUM over the K channels of a group instead of the mean:
 *   - CoExCostVolume(maxdisp, group)(x, y) (cost_volume/cost_volume.py:9-29) = sum flavour with D = maxdisp + 1, G = group;
 *   - FoundationStereo's L2-normalised volume (foundationstereo/core/submodule.py:422-461) = sum flavour on features that
 *     osb_group_l2_normalize_fwd normalised per group first (y = x / max(||x_group||_2, eps), aten F.normalize, eps 1e-12).
 * osb_sub_volume_fwd: build_sub_volume (cost_volume.py:108-117): out[b,d,h,w] = sum_c |L[..,w] - R[..,w-d]| (R = 0 for w < d).
 * osb_regression_values_fwd: sum_d prob[b,d,h,w] * values[b,d,h,w] -> (B,H,W) (casnet/submodule.py:22-24). */
int osb_gwc_volume_sum_fwd(const float* ref, const float* tgt, float* out, int B, int C, int H, int W, int D, int G,
                           osb_stream_t stream);
int osb_group_l2_normalize_fwd(const float* x, float* y, int B, int C, int H, int W, int G, float eps, osb_stream_t stream);
int osb_sub_volume_fwd(const float* left, const float* right, float* out, int B, int C, int H, int W, int D, osb_stream_t stream);
int osb_regression_values_fwd(const float* prob, const float* values, float* out, int B, int D, int H, int W, osb_stream_t stream);

/* Backward (adjoint) kernels so the volume constructors and the soft-argmin stay differentiable under tools/train.py
 * (openstereo_b200/autograd.py wraps them in torch.autograd.Function).  grad_ref / grad_tgt may be NULL when not needed.
 *   osb_gwc_volume_bwd     adjoint of osb_gwc_volume_fwd (reduce_sum = 0) / osb_gwc_volume_sum_fwd (1): grad_vol (B,G,D,H,W)
 *   osb_concat_volume_bwd  adjoint of osb_concat_volume_fwd: grad_vol (B,2C,D,H,W)
 *   osb_softargmin_bwd     adjoint of osb_softargmin_fwd w.r.t. cost: grad_out (B,H,W) -> grad_cost (B,D,H,W) */
int osb_gwc_volume_bwd(const float* grad_vol, const float* ref, const float* tgt, float* grad_ref, float* grad_tgt, int B, int C,
                       int H, int W, int D, int G, int reduce_sum, osb_stream_t stream);
int osb_concat_volume_bwd(const float* grad_vol, float* grad_ref, float* grad_tgt, int B, int C, int H, int W, int D, int mask_left,
                          osb_stream_t stream);
int osb_softargmin_bwd(const float* cost, const float* grad_out, float* grad_cost, int B, int D, int H, int W, float alpha,
                       float start, float step, int normalize, osb_stream_t stream);

/* ---- SURVEY.md section 8(f) row 2: LightStereo 2D cost aggregation (lightstereo/aggregation.py:7-134) ------------------------------
 * Depthwise Conv2d (groups = C), kernel KH x KW (odd, <= 21), padding (KH/2, KW/2), stride 1 or 2, NCHW fp32:
 *   y[b,c,oh,ow] = act(scale[c] * sum_{i,j} w[c,i,j] * x[b,c,oh*s+i-KH/2,ow*s+j-KW/2] + shift[c] + residual[b,c,oh,ow])
 * the 3x3 dwconv of MobileV2Residual (:80-84, folded BN + ReLU6) and the strip convolutions of AttentionModule
 * (:109-117: 1x7/7x1, 1x11/11x1, 1x21/21x1 with bias = shift; the branch sum `attn + attn_0 + ...` rides on `residual`).
 * w: (C, KH, KW) contiguous; scale/shift/residual optional; y may alias residual. */
int osb_dwconv2d_fwd(const float* x, const float* w, const float* scale, const float* shift, const float* residual, float* y, int B,
                     int C, int H, int W, int KH, int KW, int stride, int act, osb_stream_t stream);
/* ConvTranspose2d(k=3, stride=2, padding=1, output_padding=1, bias=False) + folded BN + residual + activation
 * (lightstereo/aggregation.py:28-34,58-59: conv5 / conv6 with `F.relu(conv5(conv4) + redir2(conv2))`): x (B,Cin,H,W) ->
 * y (B,Cout,2H,2W); w_packed (Cin, 9, Cout) = ops.pack_deconv2d_weight of the (Cin,Cout,3,3) parameter. */
int osb_deconv2d_k3s2_fwd(const float* x, const float* w_packed, const float* scale, const float* shift, const float* residual,
                          float* y, int B, int Cin, int Cout, int H, int W, int act, osb_stream_t stream);

/* ---- SURVEY.md section 8(f) rows 1 and 3: GRU-iteration lookups of IGEV / StereoBase ------------------------------------
 * Pair-average along the middle axis of a (outer, n, inner) array -> (outer, n/2, inner): the F.avg_pool2d(.., [1,2],
 * stride=[1,2]) pyramid of Combined_Geo_Encoding_Volume.__init__ (igev/geometry.py:24-30, stereobase/gru_blocks.py:187-193)
 * on the volume's native (B,C,D,H,W) layout (outer=B*C, n=D, inner=H*W) and on the all-pairs correlation
 * (outer=B*H*W1, n=W2, inner=1). */
int osb_avgpool_pairs_fwd(const float* x, float* y, long long outer, int n, long long inner, osb_stream_t stream);
/* Combined_Geo_Encoding_Volume.__call__ (igev/geometry.py:32-57) == CombinedGeoEncodingVolume.__call__
 * (stereobase/gru_blocks.py:195-220): per pyramid level i < num_levels, 2*radius+1 zero-padded bilinear taps of
 *   geo_i (B, C, D>>i, H, W) at d = disp/2^i + dx            -> channels [i*(C+1)*T + c*T + k]
 *   corr_i (B, H, W, W2>>i) at x = coords/2^i - disp/2^i + dx -> channels [i*(C+1)*T + C*T + k],   T = 2*radius+1
 * disp (B,1,H,W), coords (B,H,W), out (B, num_levels*(C+1)*T, H, W).  Unused level pointers are NULL. */
int osb_geo_lookup_fwd(const float* geo0, const float* geo1, const float* geo2, const float* geo3, const float* corr0,
                       const float* corr1, const float* corr2, const float* corr3, const float* disp, const float* coords,
                       float* out, int B, int C, int D, int H, int W, int W2, int num_levels, int radius, osb_stream_t stream);
/* context_upsample (stereobase/igev_blocks.py:51-63, igev/submodule.py:253-265): disp_low (B,1,h,w), up_weights
 * (B,9,scale*h,scale*w) -> out (B, scale*h, scale*w) = sum over the 3x3 low-resolution neighbourhood (zero padded). */
int osb_context_upsample_fwd(const float* disp_low, const float* up_weights, float* out, int B, int h, int w, int scale,
                             osb_stream_t stream);
/* (B,C,D,H,W) -> (B,D,H,W,C) layout change feeding the tensor-core conv. */
int osb_ncdhw_to_ndhwc(const float* x, float* y, int B, int C, int D, int H, int W, osb_stream_t stream);
/* Same with the channel axis zero-padded to Cpad >= C: y (B,D,H,W,Cpad) -- channel plans that are not multiples of 16 (StereoBase's
 * 24 / 48) run on the tensor-core kernels as 32 / 64 with zero weights on the padding. */
int osb_ncdhw_to_ndhwc_pad(const float* x, float* y, int B, int C, int Cpad, int D, int H, int W, osb_stream_t stream);
/* Same for fp16 tensors: x (B,C,D,H,W) fp16 -> y (B,D,H,W,Cpad) fp16, padding zero. */
int osb_ncdhw_to_ndhwc_pad_h16(const void* x, float* y, int B, int C, int Cpad, int D, int H, int W, osb_stream_t stream);
/* FeatureAtt gate in one launch (igev_blocks.py:35-48 as used by stereobase/hourglass.py:62-99):
 * gate_nhwc (B,H,W,Cpad) = sigmoid(conv1x1(act1(bn(conv1x1(feat_nchw (B,Cf,H,W)))))), channels Cv..Cpad-1 zero.
 * w1_packed (Cf,Ch), w2_packed (Ch,Cv); scale/shift = folded BN / bias (NULL = identity).  HW = H*W. */
int osb_feature_att_gate_fwd(const float* feat_nchw, const float* w1_packed, const float* scale1, const float* shift1,
                             const float* w2_packed, const float* scale2, const float* shift2, float* gate_nhwc, int B,
                             int Cf, int Ch, int Cv, int Cpad, int HW, int act1, osb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* OPENSTEREO_B200_H_ */
