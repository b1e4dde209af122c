"""Reference-facing operators: same names, argument meaning and error behaviour as the OpenStereo
functions they replace, executed by the sm_100a kernels in libopenstereo_b200.so.

PyTorch is plumbing here: it owns device memory (tensor.data_ptr()) and the stream
(torch.cuda.current_stream()).  All arithmetic happens in the hand-written kernels.  There is no
CPU path: a non-CUDA tensor raises, exactly like the reference's own native ops
(stereo/modeling/models/nmrf/ops/src/ms_deform_attn.h:29-38 -> "Not implemented on the CPU").
"""
import math

import torch

from . import _lib

ACT_NONE, ACT_RELU, ACT_LEAKY, ACT_RELU6 = 0, 1, 2, 3
TC_WIDTH = 128      # image width (at 1/4 resolution) handled by the tensor-core conv kernel
TC_KC = 32          # input channels per K chunk of the tensor-core conv (128-byte K-major rows)


_LAUNCH_DEVICE = [None]      # device index of the tensors of the launch being assembled (set by _stream, read by _call)


def _stream(t):
    """cudaStream_t of the CURRENT stream of the device `t` lives on (not of the current device: a model moved to cuda:1 without
    torch.cuda.set_device(1) must still launch on device 1 -- the reference's aten ops are device-guarded the same way)."""
    _LAUNCH_DEVICE[0] = t.device.index
    return torch.cuda.current_stream(t.device).cuda_stream


def _same_device(*tensors):
    devs = {t.device for t in tensors if t is not None}
    if len(devs) > 1:
        raise RuntimeError("openstereo_b200: operands live on different devices: %s" % sorted(str(d) for d in devs))


# Optional live timing: CUDA events recorded on the launching stream around every entry-point call.
_PROFILE = None


def profile_start():
    global _PROFILE
    _PROFILE = {}


def profile_stop():
    """-> {entry point name: [(start_event, stop_event), ...]}; call torch.cuda.synchronize() before reading."""
    global _PROFILE
    out, _PROFILE = _PROFILE, None
    return out or {}


def _call(name, *args):
    dev = _LAUNCH_DEVICE[0]
    if dev is not None and dev != torch.cuda.current_device():
        with torch.cuda.device(dev):                     # device guard: kernels launch where their operands live
            return _call_on_current(name, *args)
    return _call_on_current(name, *args)


def _call_on_current(name, *args):
    if _PROFILE is None:
        return _lib.call(name, *args)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    _lib.call(name, *args)
    stop.record()
    _PROFILE.setdefault(name, []).append((start, stop))


def _prep(t, name):
    """-> (contiguous fp32 CUDA tensor, original dtype).  Half/bf16 inputs (StereoBase under autocast,
    cfgs/stereobase/stereobase_sceneflow.yaml:50) are up-converted on load; outputs are cast back."""
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor" % name)
    if not t.is_cuda:
        raise RuntimeError("%s: not implemented on the CPU (openstereo_b200 has no CPU fallback)" % name)
    if t.dtype not in (torch.float32, torch.float16, torch.bfloat16):
        raise TypeError("%s: unsupported dtype %s" % (name, t.dtype))
    return t.detach().float().contiguous(), t.dtype


def _ptr(t):
    return None if t is None else t.data_ptr()


def _recording(*tensors):
    """True when autograd is recording on one of the operands: the call must go through openstereo_b200.autograd (the plain
    path detaches its inputs)."""
    return torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.requires_grad for t in tensors)


def _grad_operands(*tensors):
    for t in tensors:
        if not t.is_cuda:
            raise RuntimeError("openstereo_b200: not implemented on the CPU (openstereo_b200 has no CPU fallback)")
    return [t.float() for t in tensors]


# --------------------------------------------------------------------------- cost volumes
def build_gwc_volume(refimg_fea, targetimg_fea, maxdisp, num_groups):
    """stereo/modeling/cost_volume/cost_volume.py:68-78 -> (B, num_groups, maxdisp, H, W)."""
    if _recording(refimg_fea, targetimg_fea):
        from .autograd import GwcVolumeFn
        assert refimg_fea.dim() == 4 and refimg_fea.shape == targetimg_fea.shape and refimg_fea.shape[1] % num_groups == 0
        r, t = _grad_operands(refimg_fea, targetimg_fea)
        return GwcVolumeFn.apply(r, t, int(maxdisp), int(num_groups), False).to(refimg_fea.dtype)
    ref, dt = _prep(refimg_fea, "refimg_fea")
    tgt, _ = _prep(targetimg_fea, "targetimg_fea")
    assert ref.dim() == 4 and ref.shape == tgt.shape
    _same_device(ref, tgt)
    b, c, h, w = ref.shape
    assert c % num_groups == 0                       # cost_volume.py:61
    out = torch.empty((b, num_groups, maxdisp, h, w), dtype=torch.float32, device=ref.device)
    if out.numel():
        _call("osb_gwc_volume_fwd", ref.data_ptr(), tgt.data_ptr(), out.data_ptr(), b, c, h, w, maxdisp,
                  num_groups, _stream(out))
    return out.to(dt)


def build_concat_volume(refimg_fea, targetimg_fea, maxdisp, mask_left=True):
    """cost_volume.py:81-92 -> (B, 2C, maxdisp, H, W); mask_left=False is igev/submodule.py:216-227."""
    if _recording(refimg_fea, targetimg_fea):
        from .autograd import ConcatVolumeFn
        assert refimg_fea.dim() == 4 and refimg_fea.shape == targetimg_fea.shape
        r, t = _grad_operands(refimg_fea, targetimg_fea)
        return ConcatVolumeFn.apply(r, t, int(maxdisp), bool(mask_left)).to(refimg_fea.dtype)
    ref, dt = _prep(refimg_fea, "refimg_fea")
    tgt, _ = _prep(targetimg_fea, "targetimg_fea")
    assert ref.dim() == 4 and ref.shape == tgt.shape
    _same_device(ref, tgt)
    b, c, h, w = ref.shape
    out = torch.empty((b, 2 * c, maxdisp, h, w), dtype=torch.float32, device=ref.device)
    if out.numel():
        _call("osb_concat_volume_fwd", ref.data_ptr(), tgt.data_ptr(), out.data_ptr(), b, c, h, w, maxdisp,
                  1 if mask_left else 0, _stream(out))
    return out.to(dt)


def cat_fms(reference_fm, target_fm, max_disp=192, start_disp=0, dilation=1):
    """psmnet/psmnet_cost_processor.py:9-50.  PSMNet only ever calls it with start_disp=0, dilation=1
    (:227-232), where it equals build_concat_volume; other samplings are not on the hot path."""
    if start_disp != 0 or dilation != 1:
        raise NotImplementedError("cat_fms: only start_disp=0, dilation=1 (the PSMNet configuration) is accelerated")
    return build_concat_volume(reference_fm, target_fm, max_disp)


def correlation_volume(left_feature, right_feature, max_disp):
    """cost_volume.py:32-41 -> (B, max_disp, H, W)."""
    if _recording(left_feature, right_feature):
        from .autograd import GwcVolumeFn
        assert left_feature.dim() == 4 and left_feature.shape == right_feature.shape
        l, r = _grad_operands(left_feature, right_feature)
        return GwcVolumeFn.apply(l, r, int(max_disp), 1, False).squeeze(1).to(left_feature.dtype)
    l, dt = _prep(left_feature, "left_feature")
    r, _ = _prep(right_feature, "right_feature")
    assert l.dim() == 4 and l.shape == r.shape
    _same_device(l, r)
    b, c, h, w = l.shape
    out = torch.empty((b, max_disp, h, w), dtype=torch.float32, device=l.device)
    if out.numel():
        _call("osb_corr_volume_fwd", l.data_ptr(), r.data_ptr(), out.data_ptr(), b, c, h, w, max_disp, _stream(out))
    return out.to(dt)


def build_gwc_volume_normalized(refimg_fea, targetimg_fea, maxdisp, num_groups):
    """FoundationStereo's L2-normalised group-wise correlation volume (foundationstereo/core/submodule.py:422-461):
    every group's channel vector is F.normalize'd (eps 1e-12) before the dot product, which is a SUM over the group."""
    ref, dt = _prep(refimg_fea, "refimg_fea")
    tgt, _ = _prep(targetimg_fea, "targetimg_fea")
    assert ref.dim() == 4 and ref.shape == tgt.shape
    _same_device(ref, tgt)
    b, c, h, w = ref.shape
    assert c % num_groups == 0
    out = torch.empty((b, num_groups, maxdisp, h, w), dtype=torch.float32, device=ref.device)
    if out.numel():
        rn, tn = torch.empty_like(ref), torch.empty_like(tgt)
        _call("osb_group_l2_normalize_fwd", ref.data_ptr(), rn.data_ptr(), b, c, h, w, num_groups, 1e-12, _stream(out))
        _call("osb_group_l2_normalize_fwd", tgt.data_ptr(), tn.data_ptr(), b, c, h, w, num_groups, 1e-12, _stream(out))
        _call("osb_gwc_volume_sum_fwd", rn.data_ptr(), tn.data_ptr(), out.data_ptr(), b, c, h, w, maxdisp, num_groups, _stream(out))
    return out.to(dt)


def coex_cost_volume(x, y, maxdisp, group=1):
    """CoExCostVolume(maxdisp, group)(x, y), cost_volume/cost_volume.py:9-29 -> (B, group, maxdisp + 1, H, W):
    cost[b,g,d,h,w] = sum_k x[b,gK+k,h,w] * y[b,gK+k,h,w-d], zero where w < d (the module's left zero padding)."""
    if _recording(x, y):
        from .autograd import GwcVolumeFn
        assert x.dim() == 4 and x.shape == y.shape and x.shape[1] % group == 0
        a, b_ = _grad_operands(x, y)
        return GwcVolumeFn.apply(a, b_, int(maxdisp) + 1, int(group), True).to(x.dtype)
    xs, dt = _prep(x, "x")
    ys, _ = _prep(y, "y")
    assert xs.dim() == 4 and xs.shape == ys.shape
    _same_device(xs, ys)
    b, c, h, w = xs.shape
    assert c % group == 0
    out = torch.empty((b, group, maxdisp + 1, h, w), dtype=torch.float32, device=xs.device)
    if out.numel():
        _call("osb_gwc_volume_sum_fwd", xs.data_ptr(), ys.data_ptr(), out.data_ptr(), b, c, h, w, maxdisp + 1, group, _stream(out))
    return out.to(dt)


def build_sub_volume(feat_l, feat_r, maxdisp):
    """cost_volume/cost_volume.py:108-117 -> (B, maxdisp, H, W): L1 distance between the left features and the right features
    shifted by d; columns w < d see a zero right feature."""
    l, dt = _prep(feat_l, "feat_l")
    r, _ = _prep(feat_r, "feat_r")
    assert l.dim() == 4 and l.shape == r.shape
    _same_device(l, r)
    b, c, h, w = l.shape
    out = torch.empty((b, maxdisp, h, w), dtype=torch.float32, device=l.device)
    if out.numel():
        _call("osb_sub_volume_fwd", l.data_ptr(), r.data_ptr(), out.data_ptr(), b, c, h, w, maxdisp, _stream(out))
    return out.to(dt)


def gwc_concat_volume(ref_gwc, tgt_gwc, ref_cat, tgt_cat, maxdisp, num_groups):
    """GwcVolumeCostProcessor.forward (gwcnet_cost_processor.py:55-68): both volumes and the
    torch.cat in one launch -> (B, G + 2*Cc, maxdisp, H, W)."""
    rg, dt = _prep(ref_gwc, "ref_gwc")
    tg, _ = _prep(tgt_gwc, "tgt_gwc")
    rc, _ = _prep(ref_cat, "ref_cat")
    tc, _ = _prep(tgt_cat, "tgt_cat")
    assert rg.shape == tg.shape and rc.shape == tc.shape and rg.shape[0] == rc.shape[0] and rg.shape[2:] == rc.shape[2:]
    _same_device(rg, tg, rc, tc)
    b, cg, h, w = rg.shape
    cc = rc.shape[1]
    assert cg % num_groups == 0
    out = torch.empty((b, num_groups + 2 * cc, maxdisp, h, w), dtype=torch.float32, device=rg.device)
    if out.numel():
        _call("osb_gwc_concat_volume_fwd", rg.data_ptr(), tg.data_ptr(), rc.data_ptr(), tc.data_ptr(),
                  out.data_ptr(), b, cg, cc, h, w, maxdisp, num_groups, _stream(out))
    return out.to(dt)


# --------------------------------------------------------------------------- soft-argmin tails
def softargmin(cost, maxdisp, keepdim=True, alpha=1.0, start=0.0, step=1.0, normalize=True):
    """disparity_regression(F.softmax(cost, 1), maxdisp) in one pass (stereobase_gru.py:163-164)."""
    if _recording(cost):
        from .autograd import SoftArgminFn
        assert cost.dim() == 4 and cost.shape[1] == maxdisp
        (cg,) = _grad_operands(cost)
        out = SoftArgminFn.apply(cg, float(alpha), float(start), float(step), bool(normalize)).to(cost.dtype)
        return out.unsqueeze(1) if keepdim else out
    c, dt = _prep(cost, "cost")
    assert len(c.shape) == 4                          # disp_regression.py:9
    b, d, h, w = c.shape
    assert d == maxdisp
    out = torch.empty((b, h, w), dtype=torch.float32, device=c.device)
    if out.numel():
        _call("osb_softargmin_fwd", c.data_ptr(), out.data_ptr(), b, d, h, w, float(alpha), float(start),
                  float(step), 1 if normalize else 0, _stream(out))
    out = out.to(dt)
    return out.unsqueeze(1) if keepdim else out


def disparity_regression(x, maxdisp, keepdim=True):
    """disp_pred/disp_regression.py:8-12 (keepdim=True) / gwcnet_disp_processor.py:22-26 (False):
    sum_d x[:, d] * d on an already-normalised x."""
    return softargmin(x, maxdisp, keepdim=keepdim, normalize=False)


def disparity_regression_interval(prob, maxdisp, interval):
    """IGEV++'s strided expectation (igevpp/submodule.py:147-151): sum_k prob[:, k] * (k * interval) over the
    maxdisp // interval hypotheses 0, interval, 2*interval, ...; prob is already normalised.  -> (B, 1, H, W)."""
    assert len(prob.shape) == 4
    return softargmin(prob, maxdisp // interval, keepdim=True, start=0.0, step=float(interval), normalize=False)


def disparity_regression_values(prob, disp_values):
    """CasStereo's expectation over per-pixel hypothesis planes (casnet/submodule.py:22-24): sum_d prob * disp_values -> (B, H, W)."""
    p, dt = _prep(prob, "prob")
    v, _ = _prep(disp_values, "disp_values")
    assert len(p.shape) == 4 and p.shape == v.shape
    _same_device(p, v)
    b, d, h, w = p.shape
    out = torch.empty((b, h, w), dtype=torch.float32, device=p.device)
    if out.numel():
        _call("osb_regression_values_fwd", p.data_ptr(), v.data_ptr(), out.data_ptr(), b, d, h, w, _stream(out))
    return out.to(dt)


def faster_soft_argmin(cost_volume, max_disp, start_disp=0, dilation=1, alpha=1.0, normalize=True):
    """FasterSoftArgmin.forward, psmnet/psmnet_disp_processor.py:51-74 -> (B, H, W)."""
    if cost_volume.dim() != 4:
        raise ValueError('expected 4D input (got {}D input)'.format(cost_volume.dim()))
    n = (max_disp + dilation - 1) // dilation
    end = start_disp + max_disp - 1
    step = (end - start_disp) / (n - 1) if n > 1 else 0.0       # torch.linspace(start, end, n)
    return softargmin(cost_volume, n, keepdim=False, alpha=alpha, start=start_disp, step=step, normalize=normalize)


def upsample_softargmin(cost, maxdisp, out_h, out_w, align_corners=False):
    """F.interpolate(cost, [maxdisp, H, W], 'trilinear') -> squeeze -> softmax -> regression, fused
    (gwcnet_disp_processor.py:129-133; psmnet_cost_processor.py:203-214 with align_corners=True).
    cost: (B, 1, D', H', W') -> (B, H, W)."""
    c, dt = _prep(cost, "cost")
    assert c.dim() == 5 and c.shape[1] == 1
    b, _, dl, hl, wl = c.shape
    out = torch.empty((b, out_h, out_w), dtype=torch.float32, device=c.device)
    if out.numel():
        _call("osb_upsample_softargmin_fwd", c.data_ptr(), out.data_ptr(), b, dl, hl, wl, maxdisp, out_h, out_w,
                  1 if align_corners else 0, _stream(out))
    return out.to(dt)


def epe_partial(disp_pred, disp_gt, maxdisp):
    """Per-image {sum |pred-gt| over 0<gt<maxdisp, #valid} -> (B, 2) fp32
    (metric_per_image.py:32-41 with the mask of trainer_template.py:288)."""
    p, _ = _prep(disp_pred, "disp_pred")
    g, _ = _prep(disp_gt, "disp_gt")
    assert p.shape == g.shape and p.dim() == 3
    b = p.shape[0]
    out = torch.empty((b, 2), dtype=torch.float32, device=p.device)
    _call("osb_epe_partial_fwd", p.data_ptr(), g.data_ptr(), out.data_ptr(), b, p.shape[1] * p.shape[2],
              float(maxdisp), _stream(out))
    return out


def epe_per_image(disp_pred, disp_gt, maxdisp):
    part = epe_partial(disp_pred, disp_gt, maxdisp)
    return torch.where(part[:, 1] > 0, part[:, 0] / part[:, 1], torch.zeros_like(part[:, 0]))


# --------------------------------------------------------------------------- 3D aggregation primitives
def pack_conv_weight(weight):
    """(Cout, Cin, k, k, k) Conv3d parameter -> (Cin, k^3, Cout) contiguous fp32."""
    co, ci = weight.shape[:2]
    return weight.detach().float().permute(1, 2, 3, 4, 0).reshape(ci, -1, co).contiguous()


def pack_deconv_weight(weight):
    """(Cin, Cout, k, k, k) ConvTranspose3d parameter -> (Cin, k^3, Cout) contiguous fp32."""
    ci, co = weight.shape[:2]
    return weight.detach().float().permute(0, 2, 3, 4, 1).reshape(ci, -1, co).contiguous()


def fold_bn(bn):
    """Eval-mode BatchNorm -> (scale, shift) with y = x*scale + shift."""
    scale = (bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps))
    shift = bn.bias.detach().float() - bn.running_mean.detach().float() * scale
    return scale.contiguous(), shift.contiguous()


def conv3d_k3(x, w_packed, scale=None, shift=None, residual=None, gate=None, stride=1, act=ACT_NONE):
    assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous() and x.dim() == 5
    b, cin, d, h, w = x.shape
    assert w_packed.shape[0] == cin and w_packed.shape[1] == 27
    cout = w_packed.shape[2]
    do, ho, wo = (d - 1) // stride + 1, (h - 1) // stride + 1, (w - 1) // stride + 1
    y = torch.empty((b, cout, do, ho, wo), dtype=torch.float32, device=x.device)
    if residual is not None:
        assert residual.shape == y.shape and residual.is_contiguous()
    if gate is not None:
        assert gate.shape == (b, cout, ho, wo) and gate.is_contiguous()
    _call("osb_conv3d_k3_bn_act_fwd", x.data_ptr(), w_packed.data_ptr(), _ptr(scale), _ptr(shift), _ptr(residual),
              _ptr(gate), y.data_ptr(), b, cin, cout, d, h, w, stride, act, _stream(y))
    return y


def deconv3d(x, w_packed, scale=None, shift=None, residual=None, kernel=3, act=ACT_NONE):
    assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous() and x.dim() == 5
    b, cin, d, h, w = x.shape
    assert w_packed.shape[0] == cin and w_packed.shape[1] == kernel ** 3
    cout = w_packed.shape[2]
    y = torch.empty((b, cout, 2 * d, 2 * h, 2 * w), dtype=torch.float32, device=x.device)
    if residual is not None:
        assert residual.shape == y.shape and residual.is_contiguous()
    _call("osb_deconv3d_bn_act_fwd", x.data_ptr(), w_packed.data_ptr(), _ptr(scale), _ptr(shift), _ptr(residual),
              y.data_ptr(), b, cin, cout, d, h, w, kernel, act, _stream(y))
    return y


def conv3d_1x1(x0, w_packed, scale=None, shift=None, residual=None, gate=None, act=ACT_NONE, x1=None,
               sigmoid_out=False):
    """1x1x1 conv over the channel concat of x0 (and x1).  4-D inputs are treated as D=1 volumes."""
    squeeze = x0.dim() == 4
    if squeeze:
        x0 = x0.unsqueeze(2)
        x1 = None if x1 is None else x1.unsqueeze(2)
    assert x0.is_cuda and x0.dtype == torch.float32 and x0.is_contiguous()
    b, c0, d, h, w = x0.shape
    cin = c0 + (0 if x1 is None else x1.shape[1])
    if x1 is not None:
        assert x1.is_contiguous() and x1.shape[0] == b and x1.shape[2:] == x0.shape[2:]
    assert w_packed.shape[0] == cin
    cout = w_packed.shape[-1]
    y = torch.empty((b, cout, d, h, w), dtype=torch.float32, device=x0.device)
    _call("osb_conv3d_1x1_bn_act_fwd", x0.data_ptr(), _ptr(x1), c0, w_packed.data_ptr(), _ptr(scale), _ptr(shift),
              _ptr(residual), _ptr(gate), y.data_ptr(), b, cin, cout, d, h, w, act, 1 if sigmoid_out else 0, _stream(y))
    return y.squeeze(2) if squeeze else y


# --------------------------------------------------------------------------- tensor-core conv (tcgen05, 3xFP16 split)
def conv3d_tc_supported(cin, cout, w, stride=1):
    return bool(_lib.lib.osb_conv3d_tc_supported(int(cin), int(cout), int(w), int(stride)))


def conv3d_tc_kc(cin, cout, w, stride=1):
    """K chunk (16 / 32) of the tensor-core kernel variant serving this shape, 0 if there is none."""
    return int(_lib.lib.osb_conv3d_tc_kc(int(cin), int(cout), int(w), int(stride)))


def tc_operand_kind():
    """MMA kind of the tensor-core convolutions: "f16" (3xFP16 operand split, csrc/tc_common.cuh)."""
    return "f16"


TC_ACT_SCALE_LOG2 = 4        # activations are staged as x * 2^4 (csrc/tc_common.cuh: TC_ACT_SCALE); |x| must stay below 4094
TC_WEIGHT_TOP_LOG2 = 15      # per output channel, weights are scaled so that max |w| * 2^e lies in [2^14, 2^15)


def set_rz_kappa(kappa):
    """Override the accumulator round-towards-zero correction constant of the tensor-core convs (include/openstereo_b200.h:
    osb_set_rz_kappa); returns the previous value.  Calibration / bisect only."""
    return float(_lib.lib.osb_set_rz_kappa(float(kappa)))


def tc_overflow_count(device=None, reset=False):
    """Number of loader threads (since the last reset) that staged an activation outside the fp16 range of the tensor-core
    convolutions (|x| >= 4094).  Synchronises the current stream of `device`.  0 = every result is valid."""
    import ctypes
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    out = ctypes.c_uint(0)
    with torch.cuda.device(dev):
        rc = _lib.lib.osb_tc_overflow_count(torch.cuda.current_stream(dev).cuda_stream, 1 if reset else 0, ctypes.byref(out))
    if rc != 0:
        raise RuntimeError("osb_tc_overflow_count: %s" % (_lib.lib.osb_last_error() or b"").decode())
    return int(out.value)


class TcOverflowMonitor:
    """Asynchronous watch on the fp16-range counter (include/openstereo_b200.h: osb_tc_overflow_poll).  An engine calls poll()
    after its last kernel (a 4-byte device->pinned-host copy on the current stream, no synchronisation) and check() before its
    next forward: once the copy has landed, a non-zero count raises -- an activation left the +-4094 range of the tensor-core
    convolutions and the previous result was computed from saturated operands."""
    _instances = {}

    @classmethod
    def get(cls, device):
        dev = torch.device(device)
        if dev.index not in cls._instances:
            cls._instances[dev.index] = cls(dev)
        return cls._instances[dev.index]

    def __init__(self, device):
        self.device = device
        self.host = torch.zeros(1, dtype=torch.int32).pin_memory()
        self.event = None

    def poll(self):
        stream = torch.cuda.current_stream(self.device)
        with torch.cuda.device(self.device):
            rc = _lib.lib.osb_tc_overflow_poll(stream.cuda_stream, self.host.data_ptr())
        if rc != 0:
            raise RuntimeError("osb_tc_overflow_poll: %s" % (_lib.lib.osb_last_error() or b"").decode())
        self.event = torch.cuda.Event()
        self.event.record(stream)

    def check(self):
        if self.event is not None and self.event.query():
            self.event = None
            n = int(self.host.item()) & 0xFFFFFFFF
            if n:
                tc_overflow_count(self.device, reset=True)
                raise RuntimeError("openstereo_b200: %d loader threads met activations outside the fp16 range of the tensor-core "
                                   "convolutions (|x| >= 4094); the previous result is invalid.  Run those layers with "
                                   "aggregation.USE_TENSOR_CORES = False" % n)


def f16_split(w):
    """fp32 tensor (already scaled into the fp16 range) -> (hi, lo) fp16 with hi = rn(w), lo = rn(w - hi):
    |w - hi - lo| <= 2^-22 |w| while lo stays a normal fp16 number (|w| >= 2^-3), 2^-25 absolute below that."""
    w = w.contiguous()
    hi = w.to(torch.float16)
    lo = (w - hi.float()).to(torch.float16)
    return hi, lo


class TcWeight:
    """A conv weight packed for the tcgen05 kernels: `data` fp16 [3 kd][Cin/kc][3 kh][3*Cout (kw-major)][kc hi | kc lo] of
    w * 2^e_c with the 16-byte chunks of every row stored in UMMA swizzle order (pack_tc_weight), and `inv` = 2^-(e_c + TC_ACT_SCALE_LOG2) per output channel -- the exact factor the epilogue must apply.
    `cout` is the packed row count per kw slice (narrow heads are zero-padded to 16), `cout_real` the layer's channels.
    `h16`: a hi-only pack for the fp16-activation kernels (pack_tc_weight(..., h16=True)): lo halves zero, `inv` = 2^-e_c."""
    __slots__ = ("data", "inv", "kc", "cout", "cout_real", "ksize", "h16", "_eff")

    def __init__(self, data, inv, kc, cout, cout_real=None, ksize=3, h16=False):
        self.data, self.inv, self.kc, self.cout, self._eff = data, inv, kc, cout, None
        self.cout_real = cout if cout_real is None else cout_real
        self.ksize = ksize                                                  # 3, or 4 for the k4-s2 transposed conv
        self.h16 = bool(h16)

    def eff_scale(self, scale):
        """Epilogue scale vector: folded-BN scale (or 1) times the exact power-of-two un-scaling of this weight."""
        key = None if scale is None else (scale.data_ptr(), scale._version)
        if self._eff is None or self._eff[0] != key:
            if scale is not None and scale.numel() < self.inv.numel():            # zero-padded head: pad the BN scale too
                scale = torch.cat((scale.float(), scale.new_ones(self.inv.numel() - scale.numel()).float()))
            eff = self.inv if scale is None else scale.float() * self.inv
            self._eff = (key, eff.contiguous())
        return self._eff[1]


def pack_tc_weight(weight, kc=None, kw_order=(0, 1, 2), pad_cout_to=None, h16=False):
    """(Cout, Cin, k, k, k) fp32 Conv3d parameter (k = 3, or 4 for the k4-s2 transposed conv) -> TcWeight (see there).  Per output
    channel the weights are scaled by the power of two that puts max |w| into [2^14, 2^15) (exact; undone by TcWeight.inv), then
    split with f16_split.  kw_order lists the kw slices in the order the kernel stacks them along N.
    h16=True: the pack of the fp16-activation kernels -- hi = rn_fp16(w * 2^e) only (lo halves zero: one MMA per product), same
    power-of-two scaling (no weight becomes subnormal), inv = 2^-e (the activations are not scaled)."""
    w = weight.detach().float()
    cout_real, cin = w.shape[:2]
    k = int(w.shape[2])
    if pad_cout_to is not None and cout_real < pad_cout_to:             # narrow classifier heads ride the COUT = 16 kernel variant
        w = torch.cat((w, w.new_zeros((pad_cout_to - cout_real,) + tuple(w.shape[1:]))), 0)
    cout = w.shape[0]
    kc = TC_KC if kc is None else kc
    assert kc in (16, 32) and cin % kc == 0 and k in (3, 4) and tuple(w.shape[2:]) == (k, k, k) and len(kw_order) == k
    amax = w.abs().amax(dim=(1, 2, 3, 4))
    _, ex = torch.frexp(amax)                                           # amax = m * 2^ex, m in [0.5, 1)
    e = torch.where(amax > 0, TC_WEIGHT_TOP_LOG2 - ex, torch.zeros_like(ex)).clamp(-40, 40)
    ws = torch.ldexp(w, e.view(-1, 1, 1, 1, 1))
    if h16:
        hi = ws.contiguous().to(torch.float16)
        lo = torch.zeros_like(hi)
    else:
        hi, lo = f16_split(ws)
    both = torch.stack((hi, lo), 0)                                    # (2, co, ci, kd, kh, kw)
    both = both[..., list(kw_order)]                                   # stride-2 kernel wants kw slices as (1, 0, 2)
    both = both.contiguous().view(2, cout, cin // kc, kc, k, k, k)     # (half, co, chunk, ci, kd, kh, kw)
    both = both.permute(4, 2, 5, 6, 1, 0, 3)                           # (kd, chunk, kh, kw, co, half, ci)
    data = both.reshape(k, cin // kc, k, k * cout, 2 * kc).contiguous()
    # Pre-swizzle: the kernels copy a (kd, chunk, kh) slice into shared memory with ONE 1-D TMA bulk copy, so global memory already
    # holds the UMMA K-major swizzled layout: 16-byte chunk c of row n sits at chunk c ^ (n & 7) (128-byte rows, SWIZZLE_128B) or
    # c ^ ((n >> 1) & 3) (64-byte rows, SWIZZLE_64B) -- an XOR within the row, i.e. a gather with an involutive index.
    cpr = (2 * kc) // 8                                                 # 16-byte chunks per row (8 halfs each)
    rows = torch.arange(k * cout, device=data.device)
    key = (rows & 7) if kc == 32 else ((rows >> 1) & 3)
    src = torch.arange(cpr, device=data.device).view(1, cpr) ^ key.view(-1, 1)              # (rows, cpr): chunk stored at position c
    data = data.view(k, cin // kc, k, k * cout, cpr, 8)
    data = torch.gather(data, 4, src.view(1, 1, 1, k * cout, cpr, 1).expand(k, cin // kc, k, k * cout, cpr, 8).contiguous())
    data = data.reshape(k, cin // kc, k, k * cout, 2 * kc).contiguous()
    inv = torch.ldexp(torch.ones_like(amax), -(e if h16 else e + TC_ACT_SCALE_LOG2))
    return TcWeight(data, inv.contiguous(), kc, cout, cout_real, ksize=k, h16=h16)


def _is_h16(x, w_split=None, what="x"):
    """Activation dtype dispatch of the tensor-core ops: True for fp16 (the _h16 entry points, which need an h16 weight pack), False
    for fp32; any other dtype, or a weight pack of the other kind, raises."""
    if x.dtype not in (torch.float32, torch.float16):
        raise TypeError("%s: the tensor-core ops take float32 or float16 activations, got %s" % (what, x.dtype))
    h16 = x.dtype == torch.float16
    if w_split is not None and bool(getattr(w_split, "h16", False)) != h16:
        raise ValueError("%s is %s but the weight pack is %s: pack with pack_tc_weight(..., h16=%s)"
                         % (what, x.dtype, "hi-only (h16=True)" if w_split.h16 else "hi/lo split (h16=False)", h16))
    return h16


def _tc_args(w_split, cin, kc, scale):
    assert isinstance(w_split, TcWeight) and w_split.kc == kc
    k = w_split.ksize
    assert tuple(w_split.data.shape) == (k, cin // kc, k, k * w_split.cout, 2 * kc) and w_split.data.dtype == torch.float16
    assert w_split.data.is_contiguous() and w_split.data.is_cuda
    return w_split.data.data_ptr(), w_split.eff_scale(scale)


def to_ndhwc(x, pad_to=None):
    """(B,C,D,H,W) -> (B,D,H,W,C) contiguous, same dtype (fp32 or fp16), on the device; pad_to > C appends zero channels (channel
    plans that are not multiples of 16 run on the tensor-core kernels zero-padded)."""
    assert x.is_cuda and x.is_contiguous() and x.dim() == 5
    h16 = _is_h16(x)
    b, c, d, h, w = x.shape
    cp = c if pad_to is None else int(pad_to)
    assert cp >= c
    y = torch.empty((b, d, h, w, cp), dtype=x.dtype, device=x.device)
    if h16:
        _call("osb_ncdhw_to_ndhwc_pad_h16", x.data_ptr(), y.data_ptr(), b, c, cp, d, h, w, _stream(y))
    elif cp == c:
        _call("osb_ncdhw_to_ndhwc", x.data_ptr(), y.data_ptr(), b, c, d, h, w, _stream(y))
    else:
        _call("osb_ncdhw_to_ndhwc_pad", x.data_ptr(), y.data_ptr(), b, c, cp, d, h, w, _stream(y))
    return y


def conv3d_k3_tc(x_ndhwc, w_split, scale=None, shift=None, residual=None, act=ACT_NONE, out_ndhwc=True, res_ndhwc=True,
                 in_ncdhw=False, gate=None):
    """3x3x3 stride-1 conv + folded BN + residual + activation on the tensor cores.  x_ndhwc: (B,D,H,W,Cin), or the NCDHW
    tensor (B,Cin,D,H,W) with in_ncdhw=True (W = 128 layers only: the cost volume goes in as the volume kernel wrote it).
    fp16 x (with an h16 weight pack): fp16 channels-last output, no residual, fp32 gate (osb_conv3d_k3_tc_h16_fwd)."""
    assert x_ndhwc.is_cuda and x_ndhwc.is_contiguous() and x_ndhwc.dim() == 5
    if _is_h16(x_ndhwc, w_split):
        if residual is not None or not out_ndhwc or in_ncdhw:
            raise ValueError("conv3d_k3_tc: fp16 activations take channels-last in and out and no residual")
        return _conv3d_k3_tc_h16(x_ndhwc, w_split, scale, shift, act, gate)
    if in_ncdhw:
        b, cin, d, h, w = x_ndhwc.shape
    else:
        b, d, h, w, cin = x_ndhwc.shape
    cout = w_split.cout_real
    kc = conv3d_tc_kc(cin, cout, w)
    assert kc
    wptr, scale = _tc_args(w_split, cin, kc, scale)
    if shift is not None and shift.numel() < w_split.cout:               # zero-padded head
        shift = torch.cat((shift.float(), shift.new_zeros(w_split.cout - shift.numel()).float()))
    shape = (b, d, h, w, cout) if out_ndhwc else (b, cout, d, h, w)
    y = torch.empty(shape, dtype=torch.float32, device=x_ndhwc.device)
    if residual is not None:
        want = (b, d, h, w, cout) if res_ndhwc else (b, cout, d, h, w)
        assert tuple(residual.shape) == want and residual.is_contiguous()
    assert not in_ncdhw or kc == 32
    if gate is not None:                                                     # FeatureAtt: (B,H,W,Cout) multiplier after the activation
        assert kc == 16 and out_ndhwc and res_ndhwc and not in_ncdhw
        assert tuple(gate.shape) == (b, h, w, cout) and gate.is_contiguous() and gate.dtype == torch.float32 and gate.is_cuda
        _call("osb_conv3d_k3_tc_gate_fwd", x_ndhwc.data_ptr(), wptr, _ptr(scale), _ptr(shift), _ptr(residual), gate.data_ptr(),
              y.data_ptr(), b, cin, cout, d, h, w, act, _stream(y))
        return y
    _call("osb_conv3d_k3_tc_ncdhw_fwd" if in_ncdhw else "osb_conv3d_k3_tc_fwd", x_ndhwc.data_ptr(), wptr, _ptr(scale), _ptr(shift), _ptr(residual),
          y.data_ptr(), b, cin, cout, d, h, w, act, 1 if out_ndhwc else 0, 1 if res_ndhwc else 0, _stream(y))
    return y


def _conv3d_k3_tc_h16(x, w_split, scale, shift, act, gate):
    b, d, h, w, cin = x.shape
    cout = w_split.cout
    if not conv3d_tc_h16_supported(cin, cout, w):
        raise NotImplementedError("conv3d_k3_tc: no fp16 kernel for Cin=%d Cout=%d W=%d" % (cin, cout, w))
    wptr, scale = _tc_args(w_split, cin, 16, scale)
    y = torch.empty((b, d, h, w, cout), dtype=torch.float16, device=x.device)
    if gate is not None:
        assert tuple(gate.shape) == (b, h, w, cout) and gate.is_contiguous() and gate.dtype == torch.float32 and gate.is_cuda
        _call("osb_conv3d_k3_tc_gate_h16_fwd", x.data_ptr(), wptr, _ptr(scale), _ptr(shift), gate.data_ptr(), y.data_ptr(), b, cin, cout,
              d, h, w, act, _stream(y))
    else:
        _call("osb_conv3d_k3_tc_h16_fwd", x.data_ptr(), wptr, _ptr(scale), _ptr(shift), y.data_ptr(), b, cin, cout, d, h, w, act, _stream(y))
    return y


def conv3d_tc_h16_supported(cin, cout, w):
    """True when a stride-1 fp16-activation kernel serves this shape (include/openstereo_b200.h: osb_conv3d_tc_h16_supported)."""
    return bool(_lib.lib.osb_conv3d_tc_h16_supported(int(cin), int(cout), int(w)))


def conv3d_s2_tc_h16_supported(cin, cout, d, h, w):
    return bool(_lib.lib.osb_conv3d_s2_tc_h16_supported(int(cin), int(cout), int(d), int(h), int(w)))


def conv3d_s2_tc_supported(cin, cout, d, h, w):
    return bool(_lib.lib.osb_conv3d_s2_tc_supported(int(cin), int(cout), int(d), int(h), int(w)))


def conv3d_k3_s2_tc(x_ndhwc, w_split, scale=None, shift=None, residual=None, act=ACT_NONE, out_ndhwc=False, res_ndhwc=False):
    """3x3x3 STRIDE-2 conv + folded BN + residual + activation on the tensor cores.  x_ndhwc: (B,D,H,W,Cin), even D,H,W;
    w_split = pack_tc_weight(weight, 16, kw_order=(1, 0, 2)).  fp16 x (h16 pack): fp16 channels-last output, no residual."""
    assert x_ndhwc.is_cuda and x_ndhwc.is_contiguous() and x_ndhwc.dim() == 5
    b, d, h, w, cin = x_ndhwc.shape
    cout = w_split.cout
    wptr, scale = _tc_args(w_split, cin, 16, scale)
    do, ho, wo = d // 2, h // 2, w // 2
    if _is_h16(x_ndhwc, w_split):
        if residual is not None or not out_ndhwc:
            raise ValueError("conv3d_k3_s2_tc: fp16 activations take channels-last in and out and no residual")
        y = torch.empty((b, do, ho, wo, cout), dtype=torch.float16, device=x_ndhwc.device)
        _call("osb_conv3d_k3_s2_tc_h16_fwd", x_ndhwc.data_ptr(), wptr, _ptr(scale), _ptr(shift), y.data_ptr(), b, cin, cout, d, h, w, act,
              _stream(y))
        return y
    shape = (b, do, ho, wo, cout) if out_ndhwc else (b, cout, do, ho, wo)
    y = torch.empty(shape, dtype=torch.float32, device=x_ndhwc.device)
    if residual is not None:
        want = (b, do, ho, wo, cout) if res_ndhwc else (b, cout, do, ho, wo)
        assert tuple(residual.shape) == want and residual.is_contiguous()
    _call("osb_conv3d_k3_s2_tc_fwd", x_ndhwc.data_ptr(), wptr, _ptr(scale), _ptr(shift), _ptr(residual),
          y.data_ptr(), b, cin, cout, d, h, w, act, 1 if out_ndhwc else 0, 1 if res_ndhwc else 0, _stream(y))
    return y


def deconv3d_tc_supported(cin, cout, w):
    return bool(_lib.lib.osb_deconv3d_tc_supported(int(cin), int(cout), int(w)))


def pack_tc_deconv_weight(weight, h16=False):
    """(Cin, Cout, 3, 3, 3) ConvTranspose3d parameter -> TcWeight, 16-channel chunks, kw slices ordered (1, 2, 0):
    even output columns come from tap 1, odd ones from taps 2 (same input column) and 0 (next input column).
    (Cin, Cout, 4, 4, 4) (k4 s2 p1): kw slices (1, 3, 2, 0) -- even columns taps 1 (same input column) and 3 (previous one), odd
    columns taps 2 (same) and 0 (next)."""
    w = weight.detach().float().permute(1, 0, 2, 3, 4).contiguous()
    return pack_tc_weight(w, 16, kw_order=(1, 2, 0) if w.shape[2] == 3 else (1, 3, 2, 0), h16=h16)


def deconv3d_k4_tc_supported(cin, cout, w):
    return bool(_lib.lib.osb_deconv3d_k4_tc_supported(int(cin), int(cout), int(w)))


def deconv3d_k4_tc(x_ndhwc, w_split, scale=None, shift=None, residual=None, act=ACT_NONE, out_ndhwc=True, res_ndhwc=True,
                   cout_real=None):
    """ConvTranspose3d(k4, s2, p1) + folded BN + residual + activation on the tensor cores.  x_ndhwc: (B,D,H,W,Cin); cout_real <
    packed Cout (zero-padded channel plan) is allowed for an NCDHW output, which then holds only the real channels.
    fp16 x (h16 pack): fp16 output, no residual."""
    assert x_ndhwc.is_cuda and x_ndhwc.is_contiguous() and x_ndhwc.dim() == 5
    b, d, h, w, cin = x_ndhwc.shape
    cout = w_split.cout
    creal = cout if cout_real is None else int(cout_real)
    assert w_split.ksize == 4 and (out_ndhwc is False or creal == cout)
    wptr, scale = _tc_args(w_split, cin, 16, scale)
    if _is_h16(x_ndhwc, w_split):
        if residual is not None:
            raise ValueError("deconv3d_k4_tc: fp16 activations take no residual")
        shape = (b, 2 * d, 2 * h, 2 * w, cout) if out_ndhwc else (b, creal, 2 * d, 2 * h, 2 * w)
        y = torch.empty(shape, dtype=torch.float16, device=x_ndhwc.device)
        _call("osb_deconv3d_k4_tc_h16_fwd", x_ndhwc.data_ptr(), wptr, _ptr(scale), _ptr(shift), y.data_ptr(), b, cin, cout, creal, d, h, w,
              act, 1 if out_ndhwc else 0, _stream(y))
        return y
    shape = (b, 2 * d, 2 * h, 2 * w, cout) if out_ndhwc else (b, creal, 2 * d, 2 * h, 2 * w)
    y = torch.empty(shape, dtype=torch.float32, device=x_ndhwc.device)
    if residual is not None:
        want = (b, 2 * d, 2 * h, 2 * w, cout) if res_ndhwc else (b, creal, 2 * d, 2 * h, 2 * w)
        assert tuple(residual.shape) == want and residual.is_contiguous()
    _call("osb_deconv3d_k4_tc_fwd", x_ndhwc.data_ptr(), wptr, _ptr(scale), _ptr(shift), _ptr(residual),
          y.data_ptr(), b, cin, cout, creal, d, h, w, act, 1 if out_ndhwc else 0, 1 if res_ndhwc else 0, _stream(y))
    return y


def tc_slice(kind, x_ndhwc, w_split, scale, shift, y, coff, act=ACT_NONE, gate=None):
    """One output-channel SLICE of a tensor-core conv (include/openstereo_b200.h: *_cs_fwd): channels [coff, coff + w_split.cout) of
    the preallocated channels-last `y` (..., Ctot).  kind: "s1" (3x3x3 stride 1, optional (B,H,W,Ctot) gate), "s2" (stride 2) or
    "dc4" (ConvTranspose3d k4 s2 p1).  scale / shift: this slice's folded BN.  fp16 x and y (h16 pack): the _cs_h16 entry points,
    gate stays fp32."""
    assert x_ndhwc.is_cuda and x_ndhwc.is_contiguous() and x_ndhwc.dim() == 5
    assert y.is_contiguous() and y.dim() == 5
    h16 = _is_h16(x_ndhwc, w_split)
    if y.dtype != x_ndhwc.dtype:
        raise ValueError("tc_slice: x is %s but y is %s" % (x_ndhwc.dtype, y.dtype))
    b, d, h, w, cin = x_ndhwc.shape
    cout, ctot = w_split.cout, y.shape[-1]
    assert 0 <= coff and coff + cout <= ctot and coff % 4 == 0
    wptr, scale = _tc_args(w_split, cin, 16, scale)
    yp = y.data_ptr() + y.element_size() * coff
    sfx = "_h16_fwd" if h16 else "_fwd"
    if kind == "s1":
        assert tuple(y.shape[:4]) == (b, d, h, w)
        gp = None
        if gate is not None:
            assert tuple(gate.shape) == (b, h, w, ctot) and gate.is_contiguous() and gate.dtype == torch.float32
            gp = gate.data_ptr() + 4 * coff
        if h16:
            _call("osb_conv3d_k3_tc_cs_h16_fwd", x_ndhwc.data_ptr(), wptr, _ptr(scale), _ptr(shift), gp, yp, b, cin, cout, d, h, w, act,
                  ctot, _stream(y))
        else:
            _call("osb_conv3d_k3_tc_cs_fwd", x_ndhwc.data_ptr(), wptr, _ptr(scale), _ptr(shift), None, gp, yp, b, cin, cout, d, h, w, act,
                  ctot, _stream(y))
    elif kind == "s2":
        assert tuple(y.shape[:4]) == (b, d // 2, h // 2, w // 2) and gate is None
        _call("osb_conv3d_k3_s2_tc_cs" + sfx, x_ndhwc.data_ptr(), wptr, _ptr(scale), _ptr(shift), yp, b, cin, cout, d, h, w, act, ctot,
              _stream(y))
    else:
        assert kind == "dc4" and tuple(y.shape[:4]) == (b, 2 * d, 2 * h, 2 * w) and gate is None and w_split.ksize == 4
        _call("osb_deconv3d_k4_tc_cs" + sfx, x_ndhwc.data_ptr(), wptr, _ptr(scale), _ptr(shift), yp, b, cin, cout, d, h, w, act, ctot,
              _stream(y))
    return y


def feature_att_gate(feat, w1, scale1, shift1, w2, scale2, shift2, pad_to=None, act1=ACT_LEAKY):
    """FeatureAtt's gate (igev_blocks.py:35-48) in one launch: feat (B,Cf,H,W) NCHW -> sigmoid gate (B,H,W,Cpad) channels-last,
    zero beyond the Cv real channels.  w1 (Cf,Ch), w2 (Ch,Cv) packed (Cin, Cout)."""
    assert feat.is_cuda and feat.dtype == torch.float32 and feat.is_contiguous() and feat.dim() == 4
    b, cf, h, w = feat.shape
    ch, cv = w1.shape[1], w2.shape[1]
    assert w1.shape[0] == cf and w2.shape[0] == ch and w1.is_contiguous() and w2.is_contiguous()
    cp = cv if pad_to is None else int(pad_to)
    gate = torch.empty((b, h, w, cp), dtype=torch.float32, device=feat.device)
    _call("osb_feature_att_gate_fwd", feat.data_ptr(), w1.data_ptr(), _ptr(scale1), _ptr(shift1), w2.data_ptr(), _ptr(scale2),
          _ptr(shift2), gate.data_ptr(), b, cf, ch, cv, cp, h * w, act1, _stream(gate))
    return gate


def conv1x1_ndhwc_cat(x0, x1, w_packed, scale=None, shift=None, act=ACT_NONE):
    """Channels-last 1x1x1 conv over torch.cat((x0, x1), -1) without materialising it: (..., C0), (..., C1) -> (..., Cout);
    w_packed (C0 + C1, Cout).  fp16 x0 and x1: fp16 output, fp32 weights and arithmetic."""
    assert x0.is_cuda and x0.is_contiguous() and x1.is_contiguous() and x0.shape[:-1] == x1.shape[:-1]
    h16 = _is_h16(x0, what="x0")
    if x1.dtype != x0.dtype:
        raise ValueError("conv1x1_ndhwc_cat: x0 is %s but x1 is %s" % (x0.dtype, x1.dtype))
    c0, c1 = x0.shape[-1], x1.shape[-1]
    cin, cout = w_packed.shape
    assert cin == c0 + c1 and w_packed.is_contiguous() and w_packed.dtype == torch.float32
    y = torch.empty(x0.shape[:-1] + (cout,), dtype=x0.dtype, device=x0.device)
    _call("osb_conv1x1_ndhwc_cat_h16_fwd" if h16 else "osb_conv1x1_ndhwc_cat_fwd", x0.data_ptr(), x1.data_ptr(), c0, c1, w_packed.data_ptr(), _ptr(scale), _ptr(shift),
          y.data_ptr(), x0.numel() // c0, cout, act, _stream(y))
    return y


def deconv3d_k3_tc(x_ndhwc, w_split, scale=None, shift=None, residual=None, act=ACT_NONE, out_ndhwc=False, res_ndhwc=False):
    """ConvTranspose3d(k3, s2, p1, op1) + folded BN + residual + activation on the tensor cores.  x_ndhwc: (B,D,H,W,Cin)."""
    assert x_ndhwc.is_cuda and x_ndhwc.dtype == torch.float32 and x_ndhwc.is_contiguous() and x_ndhwc.dim() == 5
    b, d, h, w, cin = x_ndhwc.shape
    cout = w_split.cout
    wptr, scale = _tc_args(w_split, cin, 16, scale)
    shape = (b, 2 * d, 2 * h, 2 * w, cout) if out_ndhwc else (b, cout, 2 * d, 2 * h, 2 * w)
    y = torch.empty(shape, dtype=torch.float32, device=x_ndhwc.device)
    if residual is not None:
        want = (b, 2 * d, 2 * h, 2 * w, cout) if res_ndhwc else (b, cout, 2 * d, 2 * h, 2 * w)
        assert tuple(residual.shape) == want and residual.is_contiguous()
    _call("osb_deconv3d_k3_tc_fwd", x_ndhwc.data_ptr(), wptr, _ptr(scale), _ptr(shift), _ptr(residual),
          y.data_ptr(), b, cin, cout, d, h, w, act, 1 if out_ndhwc else 0, 1 if res_ndhwc else 0, _stream(y))
    return y


def conv1x1_ndhwc(x_ndhwc, w_packed, scale=None, shift=None, act=ACT_NONE):
    """Channels-last 1x1x1 conv: x (..., Cin) -> (..., Cout); w_packed (Cin, Cout)."""
    assert x_ndhwc.is_cuda and x_ndhwc.dtype == torch.float32 and x_ndhwc.is_contiguous()
    cin, cout = w_packed.shape
    assert x_ndhwc.shape[-1] == cin
    y = torch.empty(x_ndhwc.shape[:-1] + (cout,), dtype=torch.float32, device=x_ndhwc.device)
    _call("osb_conv1x1_ndhwc_fwd", x_ndhwc.data_ptr(), w_packed.data_ptr(), _ptr(scale), _ptr(shift), y.data_ptr(),
          x_ndhwc.numel() // cin, cin, cout, act, _stream(y))
    return y


def pack_c1_weight(weight):
    """(1, Cin, 3, 3, 3) Conv3d parameter -> (27, Cin) tap-major fp32 for conv3d_k3_c1_ndhwc."""
    assert weight.dim() == 5 and weight.shape[0] == 1 and tuple(weight.shape[2:]) == (3, 3, 3)
    return weight.detach().float()[0].permute(1, 2, 3, 0).reshape(27, -1).contiguous()


def conv3d_k3_c1_ndhwc(x_ndhwc, w_taps, scale=None, shift=None):
    """Single-output-channel 3x3x3 conv (classifier head) on a channels-last volume: (B,D,H,W,Cin) -> (B,1,D,H,W)."""
    assert x_ndhwc.is_cuda and x_ndhwc.dtype == torch.float32 and x_ndhwc.is_contiguous() and x_ndhwc.dim() == 5
    b, d, h, w, cin = x_ndhwc.shape
    assert w_taps.shape == (27, cin) and w_taps.is_contiguous()
    y = torch.empty((b, 1, d, h, w), dtype=torch.float32, device=x_ndhwc.device)
    _call("osb_conv3d_k3_c1_ndhwc_fwd", x_ndhwc.data_ptr(), w_taps.data_ptr(), _ptr(scale), _ptr(shift), y.data_ptr(), b, cin, d, h, w,
          _stream(y))
    return y


# ------------------------------------------------------------------ SURVEY.md section 8(f) row 2: LightStereo 2D aggregation
def dwconv2d(x, weight, scale=None, shift=None, residual=None, stride=1, act=ACT_NONE, out=None):
    """Depthwise Conv2d (groups = C, padding = k // 2) + per-channel scale/shift + residual + activation
    (lightstereo/aggregation.py:80-84 dwconv, :109-117 strip convs).  x (B,C,H,W); weight (C,1,KH,KW) or (C,KH,KW)."""
    assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous() and x.dim() == 4
    b, c, h, w = x.shape
    kh, kw = weight.shape[-2:]
    wt = weight.detach().float().reshape(c, kh, kw).contiguous()
    ho, wo = (h - 1) // stride + 1, (w - 1) // stride + 1
    y = torch.empty((b, c, ho, wo), dtype=torch.float32, device=x.device) if out is None else out
    if residual is not None:
        assert residual.shape == y.shape and residual.is_contiguous()
    _call("osb_dwconv2d_fwd", x.data_ptr(), wt.data_ptr(), _ptr(scale), _ptr(shift), _ptr(residual), y.data_ptr(), b, c, h, w,
          int(kh), int(kw), int(stride), act, _stream(y))
    return y


def pack_deconv2d_weight(weight):
    """(Cin, Cout, 3, 3) ConvTranspose2d parameter -> (Cin, 9, Cout) contiguous fp32."""
    ci, co = weight.shape[:2]
    assert tuple(weight.shape[2:]) == (3, 3)
    return weight.detach().float().permute(0, 2, 3, 1).reshape(ci, 9, co).contiguous()


def deconv2d_k3s2(x, w_packed, scale=None, shift=None, residual=None, act=ACT_NONE):
    """ConvTranspose2d(k3, s2, p1, op1) + folded BN + residual + activation (lightstereo/aggregation.py:28-34,58-59)."""
    assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous() and x.dim() == 4
    b, cin, h, w = x.shape
    assert w_packed.shape[0] == cin and w_packed.shape[1] == 9
    cout = w_packed.shape[2]
    y = torch.empty((b, cout, 2 * h, 2 * w), dtype=torch.float32, device=x.device)
    if residual is not None:
        assert residual.shape == y.shape and residual.is_contiguous()
    _call("osb_deconv2d_k3s2_fwd", x.data_ptr(), w_packed.data_ptr(), _ptr(scale), _ptr(shift), _ptr(residual), y.data_ptr(), b, cin,
          cout, h, w, act, _stream(y))
    return y


# ------------------------------------------------------------------ SURVEY.md section 8(f): GRU-iteration lookups
def avgpool_pairs(x, axis):
    """Average adjacent pairs along `axis` (a trailing odd element is dropped) == F.avg_pool2d(.., [1, 2], stride=[1, 2])
    applied along that axis (igev/geometry.py:24-30)."""
    assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous()
    axis = axis % x.dim()
    n = x.shape[axis]
    outer, inner = math.prod(x.shape[:axis]), math.prod(x.shape[axis + 1:])
    y = torch.empty(x.shape[:axis] + (n // 2,) + x.shape[axis + 1:], dtype=torch.float32, device=x.device)
    _call("osb_avgpool_pairs_fwd", x.data_ptr(), y.data_ptr(), outer, n, inner, _stream(y))
    return y


def geo_lookup(geo_levels, corr_levels, disp, coords, radius):
    """One lookup of the combined geometry-encoding volume (igev/geometry.py:32-57): geo_levels[i] (B,C,D>>i,H,W),
    corr_levels[i] (B,H,W,W2>>i), disp (B,1,H,W), coords (B,H,W[,1]) -> (B, L*(C+1)*(2r+1), H, W)."""
    levels = len(geo_levels)
    assert levels == len(corr_levels) and 1 <= levels <= 4
    b, c, d, h, w = geo_levels[0].shape
    w2 = corr_levels[0].shape[-1]
    for i in range(levels):
        g, cr = geo_levels[i], corr_levels[i]
        assert g.is_cuda and g.dtype == torch.float32 and g.is_contiguous() and tuple(g.shape) == (b, c, d >> i, h, w)
        assert cr.is_cuda and cr.dtype == torch.float32 and cr.is_contiguous() and tuple(cr.shape) == (b, h, w, w2 >> i)
    disp = disp.contiguous().float()
    coords = coords.reshape(b, h, w).contiguous().float()
    assert tuple(disp.shape) == (b, 1, h, w)
    out = torch.empty((b, levels * (c + 1) * (2 * radius + 1), h, w), dtype=torch.float32, device=disp.device)
    gp = [geo_levels[i].data_ptr() if i < levels else None for i in range(4)]
    cp = [corr_levels[i].data_ptr() if i < levels else None for i in range(4)]
    _call("osb_geo_lookup_fwd", *gp, *cp, disp.data_ptr(), coords.data_ptr(), out.data_ptr(), b, c, d, h, w, w2, levels, radius,
          _stream(out))
    return out


def context_upsample(disp_low, up_weights, scale_factor=4):
    """stereobase/igev_blocks.py:51-63: disp_low (B,1,h,w), up_weights (B,9,s*h,s*w) -> (B, s*h, s*w)."""
    assert disp_low.is_cuda and disp_low.dim() == 4 and disp_low.shape[1] == 1
    b, _, h, w = disp_low.shape
    assert tuple(up_weights.shape) == (b, 9, h * scale_factor, w * scale_factor)
    disp_low, up_weights = disp_low.contiguous().float(), up_weights.contiguous().float()
    out = torch.empty((b, h * scale_factor, w * scale_factor), dtype=torch.float32, device=disp_low.device)
    _call("osb_context_upsample_fwd", disp_low.data_ptr(), up_weights.data_ptr(), out.data_ptr(), b, h, w, scale_factor, _stream(out))
    return out


def conv2d_tc_kc(cin, cout, w, dilation=1):
    """K chunk of the tensor-core kernel serving a 3x3 Conv2d of this shape (0 = none)."""
    return int(_lib.lib.osb_conv2d_tc_kc(int(cin), int(cout), int(w), int(dilation)))


def conv2d_k3_tc(x_nhwc, w_split, scale=None, shift=None, residual=None, act=ACT_NONE, dilation=1, out_nhwc=True, res_nhwc=True):
    """3x3 Conv2d (stride 1, padding = dilation) + folded BN + residual + activation on the tensor cores.  x_nhwc (B,H,W,Cin);
    w_split = pack_tc_weight of the 3x3x3 weight that holds the 2D taps at kd = 1."""
    assert x_nhwc.is_cuda and x_nhwc.dtype == torch.float32 and x_nhwc.is_contiguous() and x_nhwc.dim() == 4
    b, h, w, cin = x_nhwc.shape
    cout = w_split.cout
    kc = conv2d_tc_kc(cin, cout, w, dilation)
    assert kc
    wptr, scale = _tc_args(w_split, cin, kc, scale)
    y = torch.empty((b, h, w, cout) if out_nhwc else (b, cout, h, w), dtype=torch.float32, device=x_nhwc.device)
    if residual is not None:
        assert residual.is_contiguous() and residual.numel() == y.numel()
    _call("osb_conv2d_k3_tc_fwd", x_nhwc.data_ptr(), wptr, _ptr(scale), _ptr(shift), _ptr(residual), y.data_ptr(), b, cin,
          cout, h, w, dilation, act, int(out_nhwc), int(res_nhwc), _stream(y))
    return y
