"""Hot-path engines: run the reference's 3D aggregation modules with the sm_100a kernels.

Each engine is built FROM an existing module tree (the reference's own ``GwcDispProcessor`` /
``PSMAggregator`` / StereoBase ``Hourglass``, or the host mirrors in host_models.py): it reads the
module's parameters by the reference's attribute names, pre-packs them once (weights to
(Cin, taps, Cout); eval BatchNorm folded to scale/shift) and then executes the forward graph as a
sequence of fused kernels.  cfg -> constructor -> load_state_dict stay untouched, so unchanged
checkpoints and YAML configs keep working (SURVEY.md section 8b).

Graphs restated (file:line of the reference forward each engine replaces):
  GwcAggregation        gwcnet/gwcnet_disp_processor.py:83-91,128-140 + gwcnet/hourglass.py:46-56
  PSMAggregation        psmnet/psmnet_cost_processor.py:181-221,108-132 + psmnet_disp_processor.py:107-118
  StereoBaseAggregation stereobase/hourglass.py:79-104 + stereobase_gru.py:161-164
  LightStereoAggregation lightstereo/aggregation.py:42-60 (Aggregation.forward), :94-101 (MobileV2Residual), :119-134 (AttentionModule)
"""
import torch

from . import ops
from .ops import ACT_LEAKY, ACT_NONE, ACT_RELU, ACT_RELU6


class _Packed:
    """One conv/deconv (+BN) layer, packed for the kernels."""
    __slots__ = ("w", "scale", "shift", "stride", "kernel", "transposed", "cin", "cout", "_w5", "_tc")

    def __init__(self, conv, bn=None):
        self._tc = {}                                           # K-chunk -> hi/lo split weight for the tcgen05 kernels
        self._w5 = conv.weight.detach() if conv.weight.dim() == 5 else None
        self.cin, self.cout = (conv.in_channels, conv.out_channels)
        self.transposed = isinstance(conv, (torch.nn.ConvTranspose3d, torch.nn.ConvTranspose2d))
        self.kernel = int(conv.kernel_size[0])
        self.stride = int(conv.stride[0])
        self._validate(conv)
        wt = conv.weight
        if wt.dim() == 4:                                       # Conv2d 1x1 (FeatureAtt)
            wt = wt.unsqueeze(2)
        if self.transposed:
            self.w = ops.pack_deconv_weight(wt)
        else:
            self.w = ops.pack_conv_weight(wt)
        if self.kernel == 1:
            self.w = self.w.reshape(self.w.shape[0], self.w.shape[2]).contiguous()
        self.scale, self.shift = (None, None)
        if bn is not None:
            if bn.training:
                raise RuntimeError("BatchNorm folding is only valid in eval mode (call model.eval())")
            self.scale, self.shift = ops.fold_bn(bn)
        if getattr(conv, "bias", None) is not None:
            bias = conv.bias.detach().float()
            self.shift = bias.contiguous() if self.shift is None else (self.shift + bias * self.scale).contiguous()


def _packed_validate(self, conv):
    """The kernels implement exactly the hyper-parameters of the three reference architectures (isotropic k in {1, 3} or the k4
    transposed conv, stride 1/2, padding k // 2, dilation 1, groups 1).  A module tree that deviates would silently compute a
    different convolution: refuse it instead."""
    ks, st = tuple(conv.kernel_size), tuple(conv.stride)
    ok = len(set(ks)) == 1 and len(set(st)) == 1 and tuple(conv.dilation) == (1,) * len(ks) and conv.groups == 1
    if self.transposed:
        op = tuple(conv.output_padding)
        ok = ok and ((ks[0] == 3 and st[0] == 2 and tuple(conv.padding) == (1,) * len(ks) and op == (1,) * len(ks))
                     or (ks[0] == 4 and st[0] == 2 and tuple(conv.padding) == (1,) * len(ks) and op == (0,) * len(ks)))
    else:
        ok = ok and ks[0] in (1, 3) and st[0] in (1, 2) and tuple(conv.padding) == (ks[0] // 2,) * len(ks)
        ok = ok and getattr(conv, "padding_mode", "zeros") == "zeros"
    if not ok:
        raise NotImplementedError("openstereo_b200: no kernel for %r (supported: Conv k1/k3, stride 1/2, padding k//2, dilation 1, "
                                  "groups 1; ConvTranspose k3 s2 p1 op1 or k4 s2 p1)" % (conv,))


_Packed._validate = _packed_validate


def _conv(layer, x, act=ACT_NONE, residual=None, gate=None):
    if layer.kernel == 1:
        return ops.conv3d_1x1(x, layer.w, layer.scale, layer.shift, residual, gate, act)
    return ops.conv3d_k3(x, layer.w, layer.scale, layer.shift, residual, gate, layer.stride, act)


USE_TENSOR_CORES = True      # set False to force every conv onto the fp32 CUDA-core kernels


def _tc_weight(layer, width):
    """hi/lo split weight of a 3x3x3 stride-1 layer for the tensor-core kernel variant serving `width`, or None."""
    if not USE_TENSOR_CORES or layer.transposed or layer.kernel != 3 or layer.stride != 1 or layer._w5 is None:
        return None
    kc = ops.conv3d_tc_kc(layer.cin, layer.cout, width)
    if not kc:
        return None
    if kc not in layer._tc:
        layer._tc[kc] = ops.pack_tc_weight(layer._w5, kc, pad_cout_to=16 if layer.cout < 16 else None)
    return layer._tc[kc]


def _tc_ok(layer, width):
    return _tc_weight(layer, width) is not None


def _conv_tc(layer, x_ndhwc, act=ACT_NONE, residual=None, out_ndhwc=True, res_ndhwc=True, in_ncdhw=False):
    wt = _tc_weight(layer, x_ndhwc.shape[4] if in_ncdhw else x_ndhwc.shape[3])
    return ops.conv3d_k3_tc(x_ndhwc, wt, layer.scale, layer.shift, residual, act, out_ndhwc, res_ndhwc, in_ncdhw)


def _stem_in(layer, volume, act):
    """First aggregation layer on an NCDHW cost volume: the W = 128 kernel reads NCDHW directly, other variants convert once."""
    if ops.conv3d_tc_kc(layer.cin, layer.cout, volume.shape[-1]) == 32:
        return _conv_tc(layer, volume, act, in_ncdhw=True)
    return _conv_tc(layer, ops.to_ndhwc(volume), act)


def _conv_auto(layer, x, act=ACT_NONE, residual=None):
    """3x3x3 conv (stride 1 or 2) on an NCDHW tensor, NCDHW result: tensor cores when a kernel variant exists for the
    shape, the fp32 CUDA-core kernel otherwise."""
    if layer.stride == 1 and _tc_ok(layer, x.shape[-1]):
        return _conv_tc(layer, ops.to_ndhwc(x), act, residual, out_ndhwc=False, res_ndhwc=False)
    if (USE_TENSOR_CORES and layer.stride == 2 and layer.kernel == 3 and not layer.transposed and layer._w5 is not None
            and ops.conv3d_s2_tc_supported(layer.cin, layer.cout, x.shape[2], x.shape[3], x.shape[4])):
        if "s2" not in layer._tc:
            layer._tc["s2"] = ops.pack_tc_weight(layer._w5, 16, kw_order=(1, 0, 2))
        return ops.conv3d_k3_s2_tc(ops.to_ndhwc(x), layer._tc["s2"], layer.scale, layer.shift, residual, act)
    return _conv(layer, x, act, residual)


def _deconv(layer, x, act=ACT_NONE, residual=None):
    if (USE_TENSOR_CORES and layer.transposed and layer.kernel == 3 and layer._w5 is not None
            and ops.deconv3d_tc_supported(layer.cin, layer.cout, x.shape[-1])):
        if "dc" not in layer._tc:
            layer._tc["dc"] = ops.pack_tc_deconv_weight(layer._w5)
        return ops.deconv3d_k3_tc(ops.to_ndhwc(x), layer._tc["dc"], layer.scale, layer.shift, residual, act)
    return ops.deconv3d(x, layer.w, layer.scale, layer.shift, residual, layer.kernel, act)


def _versions(module):
    return tuple(p._version for p in module.parameters()) + tuple(b._version for b in module.buffers())


class _Engine:
    """Pre-pack on first use; re-pack when any parameter/buffer was modified in place or moved."""

    def __init__(self, module):
        self.module = module
        self._stamp = None

    def _watch(self, device):
        """fp16-range guard of the tensor-core convolutions: report a past overflow, schedule the next asynchronous read."""
        if USE_TENSOR_CORES:
            mon = ops.TcOverflowMonitor.get(device)
            mon.check()
            return mon
        return None

    def _ensure(self, device):
        stamp = (str(device), _versions(self.module), tuple(p.data_ptr() for p in self.module.parameters()))
        if stamp != self._stamp:
            if self.module.training:
                raise RuntimeError("openstereo_b200 engines run inference only: call model.eval()")
            with torch.no_grad():
                self._pack()
            self._stamp = stamp

    @staticmethod
    def _check(x, dtype=torch.float32):
        if not x.is_cuda:
            raise RuntimeError("openstereo_b200: not implemented on the CPU (no fallback); move the model to CUDA")
        return x.detach().to(dtype).contiguous()


# ------------------------------------------------------------------------------------------------------ GwcNet
class _GwcHourglass:
    def __init__(self, m):
        self.conv1, self.conv2 = _Packed(m.conv1[0][0], m.conv1[0][1]), _Packed(m.conv2[0][0], m.conv2[0][1])
        self.conv3, self.conv4 = _Packed(m.conv3[0][0], m.conv3[0][1]), _Packed(m.conv4[0][0], m.conv4[0][1])
        self.conv5, self.conv6 = _Packed(m.conv5[0], m.conv5[1]), _Packed(m.conv6[0], m.conv6[1])
        self.redir1, self.redir2 = _Packed(m.redir1[0], m.redir1[1]), _Packed(m.redir2[0], m.redir2[1])

    def __call__(self, x):
        c1 = _conv_auto(self.conv1, x, ACT_RELU)
        c2 = _conv_auto(self.conv2, c1, ACT_RELU)
        c3 = _conv_auto(self.conv3, c2, ACT_RELU)
        c4 = _conv_auto(self.conv4, c3, ACT_RELU)
        c5 = _deconv(self.conv5, c4, ACT_RELU, residual=_conv(self.redir2, c2))
        return _deconv(self.conv6, c5, ACT_RELU, residual=_conv(self.redir1, x))


def _hg_channels_last_ok(hg, x_shape_ndhwc):
    """True when every layer of a GwcNet hourglass has a tensor-core / channels-last kernel for this input."""
    if not USE_TENSOR_CORES:
        return False
    b, d, h, w, c = x_shape_ndhwc
    if d % 4 or h % 4 or w % 4:
        return False
    return (ops.conv3d_s2_tc_supported(hg.conv1.cin, hg.conv1.cout, d, h, w) and _tc_ok(hg.conv2, w // 2)
            and ops.conv3d_s2_tc_supported(hg.conv3.cin, hg.conv3.cout, d // 2, h // 2, w // 2) and _tc_ok(hg.conv4, w // 4)
            and ops.deconv3d_tc_supported(hg.conv5.cin, hg.conv5.cout, w // 4)
            and ops.deconv3d_tc_supported(hg.conv6.cin, hg.conv6.cout, w // 2)
            and (hg.redir1.cin, hg.redir1.cout) in ((32, 32), (64, 64)) and (hg.redir2.cin, hg.redir2.cout) in ((32, 32), (64, 64)))


def _s2_weight(layer):
    if "s2" not in layer._tc:
        layer._tc["s2"] = ops.pack_tc_weight(layer._w5, 16, kw_order=(1, 0, 2))
    return layer._tc["s2"]


def _dc_weight(layer):
    if "dc" not in layer._tc:
        layer._tc["dc"] = ops.pack_tc_deconv_weight(layer._w5)
    return layer._tc["dc"]


def _gwc_hourglass_channels_last(hg, x):
    """GwcNet hourglass (gwcnet/hourglass.py:46-56) with every tensor channels-last: no layout conversion between layers."""
    c1 = ops.conv3d_k3_s2_tc(x, _s2_weight(hg.conv1), hg.conv1.scale, hg.conv1.shift, None, ACT_RELU, out_ndhwc=True)
    c2 = _conv_tc(hg.conv2, c1, ACT_RELU)
    c3 = ops.conv3d_k3_s2_tc(c2, _s2_weight(hg.conv3), hg.conv3.scale, hg.conv3.shift, None, ACT_RELU, out_ndhwc=True)
    c4 = _conv_tc(hg.conv4, c3, ACT_RELU)
    r2 = ops.conv1x1_ndhwc(c2, hg.redir2.w, hg.redir2.scale, hg.redir2.shift)
    c5 = ops.deconv3d_k3_tc(c4, _dc_weight(hg.conv5), hg.conv5.scale, hg.conv5.shift, r2, ACT_RELU, out_ndhwc=True, res_ndhwc=True)
    r1 = ops.conv1x1_ndhwc(x, hg.redir1.w, hg.redir1.scale, hg.redir1.shift)
    return ops.deconv3d_k3_tc(c5, _dc_weight(hg.conv6), hg.conv6.scale, hg.conv6.shift, r1, ACT_RELU, out_ndhwc=True, res_ndhwc=True)


class GwcAggregation(_Engine):
    """Eval branch of GwcDispProcessor: volume (B,64,D',H',W') -> disparity (B,H,W)."""

    def _pack(self):
        m = self.module
        self.dres0 = [_Packed(m.dres0[0][0], m.dres0[0][1]), _Packed(m.dres0[2][0], m.dres0[2][1])]
        self.dres1 = [_Packed(m.dres1[0][0], m.dres1[0][1]), _Packed(m.dres1[2][0], m.dres1[2][1])]
        self.hg = [_GwcHourglass(m.dres2), _GwcHourglass(m.dres3), _GwcHourglass(m.dres4)]
        self.classif3 = [_Packed(m.classif3[0][0], m.classif3[0][1]), _Packed(m.classif3[2])]

    def logits(self, volume):
        volume = self._check(volume)
        self._ensure(volume.device)
        width = volume.shape[-1]
        stem_tc = all(_tc_ok(l, width) for l in (self.dres0[0], self.dres0[1], self.dres1[0], self.dres1[1]))
        b, _, dd, hh, ww = volume.shape
        if stem_tc and _tc_ok(self.classif3[0], width) and all(_hg_channels_last_ok(hg, (b, dd, hh, ww, 32)) for hg in self.hg):
            # everything from the volume to the classifier runs channels-last on the tensor cores: ONE layout conversion
            c = _conv_tc(self.dres0[1], _stem_in(self.dres0[0], volume, ACT_RELU), ACT_RELU)
            out = _conv_tc(self.dres1[1], _conv_tc(self.dres1[0], c, ACT_RELU), ACT_NONE, residual=c)
            for hg in self.hg:
                out = _gwc_hourglass_channels_last(hg, out)
            cls = self.classif3[1]
            if _tc_ok(cls, width):                                         # 32 -> 1 head on the narrow (Cout <= 16) tensor-core variant
                return _conv_tc(cls, _conv_tc(self.classif3[0], out, ACT_RELU), ACT_NONE, out_ndhwc=False, res_ndhwc=False)
            if cls.cin == 32 and cls.cout == 1 and cls._w5 is not None and cls.stride == 1:
                if "c1" not in cls._tc:
                    cls._tc["c1"] = ops.pack_c1_weight(cls._w5)
                head = _conv_tc(self.classif3[0], out, ACT_RELU)           # stays channels-last for the 1-channel head
                return ops.conv3d_k3_c1_ndhwc(head, cls._tc["c1"], cls.scale, cls.shift)
            head = _conv_tc(self.classif3[0], out, ACT_RELU, out_ndhwc=False)
            return _conv(cls, head)
        if stem_tc:
            # full-resolution stem on the tensor cores: channels-last inside, NCDHW handed to the hourglasses
            c = _conv_tc(self.dres0[1], _stem_in(self.dres0[0], volume, ACT_RELU), ACT_RELU)
            cost0 = _conv_tc(self.dres1[1], _conv_tc(self.dres1[0], c, ACT_RELU), ACT_NONE, residual=c, out_ndhwc=False)
        else:
            c = _conv(self.dres0[1], _conv(self.dres0[0], volume, ACT_RELU), ACT_RELU)
            cost0 = _conv(self.dres1[1], _conv(self.dres1[0], c, ACT_RELU), ACT_NONE, residual=c)
        out = cost0
        for hg in self.hg:
            out = hg(out)
        if _tc_ok(self.classif3[0], width):
            head = _conv_tc(self.classif3[0], ops.to_ndhwc(out), ACT_RELU, out_ndhwc=False)
        else:
            head = _conv(self.classif3[0], out, ACT_RELU)
        return _conv(self.classif3[1], head)

    def __call__(self, volume, h, w):
        mon = self._watch(volume.device)
        out = ops.upsample_softargmin(self.logits(volume), self.module.maxdisp, h, w, align_corners=False)
        if mon is not None:
            mon.poll()
        return out


# ------------------------------------------------------------------------------------------------------ PSMNet
class _PSMHourglass:
    def __init__(self, m):
        self.conv1, self.conv2 = _Packed(m.conv1[0], m.conv1[1]), _Packed(m.conv2[0], m.conv2[1])
        self.conv3, self.conv4 = _Packed(m.conv3[0], m.conv3[1]), _Packed(m.conv4[0], m.conv4[1])
        self.conv5, self.conv6 = _Packed(m.conv5[0], m.conv5[1]), _Packed(m.conv6[0], m.conv6[1])

    def __call__(self, x, presqu, postsqu, skip):
        out = _conv_auto(self.conv1, x, ACT_RELU)
        pre = _conv_auto(self.conv2, out, ACT_RELU, residual=postsqu)
        out = _conv_auto(self.conv4, _conv_auto(self.conv3, pre, ACT_RELU), ACT_RELU)
        post = _deconv(self.conv5, out, ACT_RELU, residual=presqu if presqu is not None else pre)
        # `out_i = hourglass(...) + cost0` (psmnet_cost_processor.py:188-194) rides on conv6's epilogue
        return _deconv(self.conv6, post, ACT_NONE, residual=skip), pre, post


def _psm_hg_channels_last_ok(hg, shape_ndhwc):
    """True when every layer of a PSMNet hourglass has a tensor-core kernel for this channels-last input."""
    if not USE_TENSOR_CORES:
        return False
    b, d, h, w, c = shape_ndhwc
    if d % 4 or h % 4 or w % 4 or any(l._w5 is None for l in (hg.conv1, hg.conv2, hg.conv3, hg.conv4, hg.conv5, hg.conv6)):
        return False
    return (ops.conv3d_s2_tc_supported(hg.conv1.cin, hg.conv1.cout, d, h, w) and _tc_ok(hg.conv2, w // 2)
            and ops.conv3d_s2_tc_supported(hg.conv3.cin, hg.conv3.cout, d // 2, h // 2, w // 2) and _tc_ok(hg.conv4, w // 4)
            and hg.conv5.kernel == 3 and hg.conv6.kernel == 3
            and ops.deconv3d_tc_supported(hg.conv5.cin, hg.conv5.cout, w // 4)
            and ops.deconv3d_tc_supported(hg.conv6.cin, hg.conv6.cout, w // 2))


def _psm_hourglass_channels_last(hg, x, presqu, postsqu, skip):
    """PSMNet hourglass (psmnet_cost_processor.py:108-132) with every tensor channels-last: the NCDHW route converted the layout in
    front of every layer.  Returns (out + skip, pre, post) like _PSMHourglass.__call__, all NDHWC."""
    out = ops.conv3d_k3_s2_tc(x, _s2_weight(hg.conv1), hg.conv1.scale, hg.conv1.shift, None, ACT_RELU, out_ndhwc=True)
    pre = _conv_tc(hg.conv2, out, ACT_RELU, residual=postsqu)
    out = ops.conv3d_k3_s2_tc(pre, _s2_weight(hg.conv3), hg.conv3.scale, hg.conv3.shift, None, ACT_RELU, out_ndhwc=True)
    out = _conv_tc(hg.conv4, out, ACT_RELU)
    post = ops.deconv3d_k3_tc(out, _dc_weight(hg.conv5), hg.conv5.scale, hg.conv5.shift, presqu if presqu is not None else pre, ACT_RELU,
                              out_ndhwc=True, res_ndhwc=True)
    out = ops.deconv3d_k3_tc(post, _dc_weight(hg.conv6), hg.conv6.scale, hg.conv6.shift, skip, ACT_NONE, out_ndhwc=True, res_ndhwc=True)
    return out, pre, post


class PSMAggregation(_Engine):
    """PSMAggregator + FasterSoftArgmin: raw concat volume -> [disp1, disp2, disp3], each (B,H,W)."""

    def _pack(self):
        m = self.module
        self.dres0 = [_Packed(m.dres0[0][0], m.dres0[0][1]), _Packed(m.dres0[1][0], m.dres0[1][1])]
        self.dres1 = [_Packed(m.dres1[0][0], m.dres1[0][1]), _Packed(m.dres1[1][0], m.dres1[1][1])]
        self.hg = [_PSMHourglass(m.dres2), _PSMHourglass(m.dres3), _PSMHourglass(m.dres4)]
        self.heads = [[_Packed(c[0][0], c[0][1]), _Packed(c[1])] for c in (m.classif1, m.classif2, m.classif3)]

    def logits(self, raw_cost):
        raw_cost = self._check(raw_cost)
        self._ensure(raw_cost.device)
        width = raw_cost.shape[-1]
        stem_tc = all(_tc_ok(l, width) for l in (self.dres0[0], self.dres0[1], self.dres1[0], self.dres1[1]))
        b, _, dd, hh, ww = raw_cost.shape
        if (stem_tc and all(_psm_hg_channels_last_ok(hg, (b, dd, hh, ww, 32)) for hg in self.hg)
                and all(_tc_ok(a, width) and _tc_ok(bb, width) for a, bb in self.heads)):
            # everything channels-last on the tensor cores: the stacked-hourglass skips (pre / post / cost0) never change layout
            c = _conv_tc(self.dres0[1], _stem_in(self.dres0[0], raw_cost, ACT_RELU), ACT_RELU)
            cost0 = _conv_tc(self.dres1[1], _conv_tc(self.dres1[0], c, ACT_RELU), ACT_NONE, residual=c)
            out1, pre1, post1 = _psm_hourglass_channels_last(self.hg[0], cost0, None, None, cost0)
            out2, pre2, post2 = _psm_hourglass_channels_last(self.hg[1], out1, pre1, post1, cost0)
            out3, _, _ = _psm_hourglass_channels_last(self.hg[2], out2, pre2, post2, cost0)
            costs, prev = [], None
            for (a, bb), x in zip(self.heads, (out1, out2, out3)):
                prev = _conv_tc(bb, _conv_tc(a, x, ACT_RELU), ACT_NONE, residual=prev, out_ndhwc=False, res_ndhwc=False)
                costs.append(prev)
            return costs
        if stem_tc:
            c = _conv_tc(self.dres0[1], _stem_in(self.dres0[0], raw_cost, ACT_RELU), ACT_RELU)
            cost0 = _conv_tc(self.dres1[1], _conv_tc(self.dres1[0], c, ACT_RELU), ACT_NONE, residual=c, out_ndhwc=False)
        else:
            c = _conv(self.dres0[1], _conv(self.dres0[0], raw_cost, ACT_RELU), ACT_RELU)
            cost0 = _conv(self.dres1[1], _conv(self.dres1[0], c, ACT_RELU), ACT_NONE, residual=c)
        out1, pre1, post1 = self.hg[0](cost0, None, None, cost0)
        out2, pre2, post2 = self.hg[1](out1, pre1, post1, cost0)
        out3, pre3, post3 = self.hg[2](out2, pre2, post2, cost0)

        def head(i, x, prev):
            a, b = self.heads[i]
            if _tc_ok(a, width) and _tc_ok(b, width):                   # both convs on tensor cores, channels-last in between
                return _conv_tc(b, _conv_tc(a, ops.to_ndhwc(x), ACT_RELU), ACT_NONE, residual=prev, out_ndhwc=False, res_ndhwc=False)
            if _tc_ok(a, width):
                return _conv(b, _conv_tc(a, ops.to_ndhwc(x), ACT_RELU, out_ndhwc=False), residual=prev)
            return _conv(b, _conv(a, x, ACT_RELU), residual=prev)

        cost1 = head(0, out1, None)
        cost2 = head(1, out2, cost1)
        cost3 = head(2, out3, cost2)
        return [cost1, cost2, cost3]

    def __call__(self, raw_cost):
        b, c, d, h, w = raw_cost.shape
        max_disp = self.module.max_disp
        mon = self._watch(raw_cost.device)
        out = [ops.upsample_softargmin(cost, max_disp, 4 * h, 4 * w, align_corners=True)
               for cost in self.logits(raw_cost)]
        if mon is not None:
            mon.poll()
        return out


# -------------------------------------------------------------------------------------------------- StereoBase
class _FeatureAtt:
    def __init__(self, m):
        blk = m.feat_att[0].block
        self.a = _Packed(blk[0], blk[1])
        self.b = _Packed(m.feat_att[1])
        self.act = ACT_LEAKY if any(isinstance(l, torch.nn.LeakyReLU) for l in blk) else ACT_NONE

    def __call__(self, feat):
        hidden = ops.conv3d_1x1(feat, self.a.w, self.a.scale, self.a.shift, act=ACT_LEAKY)
        return ops.conv3d_1x1(hidden, self.b.w, self.b.scale, self.b.shift, sigmoid_out=True)   # (B, cv_chan, H, W)


def _block(m):
    layers = list(m.block)
    bn = layers[1] if len(layers) > 1 and isinstance(layers[1], torch.nn.BatchNorm3d) else None
    act = ACT_LEAKY if any(isinstance(l, torch.nn.LeakyReLU) for l in layers) else ACT_NONE
    return _Packed(layers[0], bn), act


class StereoBaseAggregation(_Engine):
    """Hourglass(volume_channel, backbone_channels) with FeatureAtt gates: (B,C,D',H',W') + 2D features -> same shape.

    precision="fp32" (default): every input is computed with fp32-accurate products (3xFP16 split) and the result is fp32.
    precision="fp16": a float16 volume (the model runs under torch.autocast(float16)) whose shape has the whole tensor-core route
    (_h16_route_ok) stays fp16 end to end -- fp16 activations, one fp16 MMA per product, fp32 accumulation, BN / activation / gate
    in fp32, fp16 stores that saturate at +-65504 and make the next call raise (ops.TcOverflowMonitor) -- and the result is fp16.
    Any other input (fp32, bf16, other shapes) takes the fp32 path, as with precision="fp32"."""

    def __init__(self, module, precision="fp32"):
        if precision not in ("fp32", "fp16"):
            raise ValueError("precision must be 'fp32' or 'fp16', got %r" % (precision,))
        super().__init__(module)
        self.precision = precision

    def _pack(self):
        m = self.module
        self.conv = {name: [_block(b) for b in getattr(m, name)] for name in ("conv1", "conv2", "conv3", "agg_0", "agg_1")}
        self.up = {name: _block(getattr(m, name)) for name in ("conv3_up", "conv2_up", "conv1_up")}
        self.att = {name: _FeatureAtt(getattr(m, "feature_att_" + name)) for name in ("8", "16", "32", "up_16", "up_8")}

    def _pair(self, name, x, gate):
        (l0, a0), (l1, a1) = self.conv[name]
        return _conv(l1, _conv(l0, x, a0), a1, gate=gate)

    def _agg(self, name, up, skip, gate):
        (l0, a0), (l1, a1), (l2, a2) = self.conv[name]
        # torch.cat((up, skip), 1) -> 1x1 conv, without materialising the concat (hourglass.py:91-92,96-97)
        x = ops.conv3d_1x1(up, l0.w, l0.scale, l0.shift, act=a0, x1=skip)
        return _conv(l2, _conv(l1, x, a1), a2, gate=gate)

    # ---- tensor-core route: channels-last, channel plan zero-padded to multiples of 32 (24 -> 32, 48 -> 64, 96) -------------------
    @staticmethod
    def _pad32(c):
        return (c + 31) // 32 * 32

    def tc_route_ok(self, shape):
        """True when the 1/8 and 1/16 levels and the two upper transposed convs of this hourglass have tcgen05 variants for an
        input volume of `shape` (B, C, D', H', W'); the 1/32 level (6 % of the MACs at config 3) stays on the CUDA-core kernels."""
        if not USE_TENSOR_CORES:
            return False
        b, c, d, h, w = shape
        if d % 8 or h % 8 or w % 8:
            return False
        (l10, _), (l11, _) = self.conv["conv1"]
        (l20, _), (l21, _) = self.conv["conv2"]
        if (l10.cin, l10.cout, l20.cout) != (c, 2 * c, 4 * c) or any(l._w5 is None for l in (l10, l11, l20, l21)):
            return False
        pc, p2, p4 = self._pad32(c), self._pad32(2 * c), self._pad32(4 * c)
        return bool(ops.conv3d_s2_tc_supported(pc, p2, d, h, w) and ops.conv3d_tc_kc(p2, p2, w // 2) == 16
                    and ops.conv3d_s2_tc_supported(p2, p4, d // 2, h // 2, w // 2) and ops.conv3d_tc_kc(p4, p4, w // 4) == 16
                    and ops.deconv3d_k4_tc_supported(p4, p2, w // 4) and ops.deconv3d_k4_tc_supported(p2, pc, w // 2)
                    and (2 * p4, p4) in ((192, 96), (128, 64)) and (2 * p2, p2) in ((192, 96), (128, 64))
                    and self.up["conv2_up"][0].kernel == 4 and self.up["conv1_up"][0].kernel == 4)

    def _tc_pack(self, h16=False):
        """Zero-padded tensor-core packs of the layers on the 1/8 and 1/16 levels (built once per _ensure stamp); h16=True: the
        hi-only packs of the fp16 route, cached beside the split ones."""
        if getattr(self, "_tcp_stamp", None) != self._stamp:
            self._tcp, self._tcp_stamp = {}, self._stamp
        if h16 not in self._tcp:
            self._tcp[h16] = self._build_tc_pack(h16)
        return self._tcp[h16]

    def _build_tc_pack(self, h16):
        P = self._pad32

        def vec(v, n, fill):
            if v is None:
                return None
            out = v.new_full((n,), fill)
            out[:v.numel()] = v
            return out

        def conv(layer, kw_order=(0, 1, 2)):
            w = layer._w5
            wp = w.new_zeros((P(w.shape[0]), P(w.shape[1])) + tuple(w.shape[2:]))
            wp[:w.shape[0], :w.shape[1]] = w
            return (ops.pack_tc_weight(wp, 16, kw_order=kw_order, h16=h16), vec(layer.scale, wp.shape[0], 1.0),
                    vec(layer.shift, wp.shape[0], 0.0))

        def deconv(layer):
            w = layer._w5                                                   # (Cin, Cout, 4, 4, 4)
            wp = w.new_zeros((P(w.shape[0]), P(w.shape[1])) + tuple(w.shape[2:]))
            wp[:w.shape[0], :w.shape[1]] = w
            return (ops.pack_tc_deconv_weight(wp, h16=h16), vec(layer.scale, wp.shape[1], 1.0), vec(layer.shift, wp.shape[1], 0.0))

        def cat1x1(layer):
            w = layer.w                                                     # (C0 + C1, Cout), both slabs Cout channels wide
            cout = w.shape[1]
            wp = w.new_zeros((2 * P(cout), P(cout)))
            wp[:cout, :cout] = w[:cout]
            wp[P(cout):P(cout) + cout, :cout] = w[cout:]
            return (wp.contiguous(), vec(layer.scale, P(cout), 1.0), vec(layer.shift, P(cout), 0.0))

        t = {}
        for name in ("conv1", "conv2"):
            (l0, _), (l1, _) = self.conv[name]
            t[name] = (conv(l0, (1, 0, 2)), conv(l1))
        for name in ("agg_0", "agg_1"):
            (l0, _), (l1, _), (l2, _) = self.conv[name]
            t[name] = (cat1x1(l0), conv(l1), conv(l2))
        for name in ("conv2_up", "conv1_up"):
            t[name] = deconv(self.up[name][0])
        # 1/32 level: 6c = 144 runs as 160 = 96 + 64 output-channel slices (N = 3 * 160 exceeds one CTA's weight buffers), the
        # transposed conv back to 4c = 96 as 64 + 32 (N = 4 * 96 exceeds the UMMA N limit): separately packed weight slices
        (l0, _), (l1, _) = self.conv["conv3"]
        lu = self.up["conv3_up"][0]
        if P(l0.cout) == 160 and P(l0.cin) == 96 and lu.kernel == 4 and all(l._w5 is not None for l in (l0, l1, lu)):
            def slices(layer, bounds, transposed=False, kw_order=(0, 1, 2)):
                w = layer._w5
                if transposed:                                              # (Cin, Cout, 4, 4, 4): pad Cin, slice Cout
                    wp = w.new_zeros((P(w.shape[0]), P(w.shape[1])) + tuple(w.shape[2:]))
                    wp[:w.shape[0], :w.shape[1]] = w
                    n = wp.shape[1]
                else:
                    wp = w.new_zeros((P(w.shape[0]), P(w.shape[1])) + tuple(w.shape[2:]))
                    wp[:w.shape[0], :w.shape[1]] = w
                    n = wp.shape[0]
                sc, sh = vec(layer.scale, n, 1.0), vec(layer.shift, n, 0.0)
                out = []
                for lo, hi in bounds:
                    wt = (ops.pack_tc_deconv_weight(wp[:, lo:hi].contiguous(), h16=h16) if transposed
                          else ops.pack_tc_weight(wp[lo:hi].contiguous(), 16, kw_order=kw_order, h16=h16))
                    out.append((lo, wt, None if sc is None else sc[lo:hi].contiguous(), None if sh is None else sh[lo:hi].contiguous()))
                return out
            t["conv3"] = (slices(l0, ((0, 96), (96, 160)), kw_order=(1, 0, 2)), slices(l1, ((0, 96), (96, 160))))
            t["conv3_up"] = slices(lu, ((0, 64), (64, 96)), transposed=True)
        return t

    def _level32_tc_ok(self, shape):
        b, c, d, h, w = shape
        return bool(w // 8 == 16 and self._pad32(6 * c) == 160 and self._pad32(4 * c) == 96
                    and ops.conv3d_s2_tc_supported(96, 96, d // 4, h // 4, w // 4) and ops.conv3d_s2_tc_supported(96, 64, d // 4, h // 4, w // 4)
                    and ops.conv3d_tc_kc(160, 96, 16) == 16 and ops.conv3d_tc_kc(160, 64, 16) == 16
                    and ops.deconv3d_k4_tc_supported(160, 64, 16) and ops.deconv3d_k4_tc_supported(160, 32, 16))

    def _h16_route_ok(self, shape):
        """True when every layer of _call_tc has an fp16-activation kernel for an input volume of `shape` (the 1/32 level included)."""
        b, c, d, h, w = shape
        if not (self.tc_route_ok(shape) and self._level32_tc_ok(shape) and "conv3" in self._tc_pack()):
            return False
        pc, p2, p4 = self._pad32(c), self._pad32(2 * c), self._pad32(4 * c)
        return (ops.conv3d_s2_tc_h16_supported(pc, p2, d, h, w) and ops.conv3d_tc_h16_supported(p2, p2, w // 2)
                and ops.conv3d_s2_tc_h16_supported(p2, p4, d // 2, h // 2, w // 2) and ops.conv3d_tc_h16_supported(p4, p4, w // 4)
                and ops.conv3d_s2_tc_h16_supported(p4, 96, d // 4, h // 4, w // 4) and ops.conv3d_tc_h16_supported(160, 96, w // 8))

    def _gate_nhwc(self, name, feat, channels):
        fa = self.att[name]                                                 # one launch: (B, H, W, C padded), padded channels 0
        if fa.a.w.shape[1] % 4 == 0 and fa.b.w.shape[1] % 4 == 0:
            return ops.feature_att_gate(feat, fa.a.w, fa.a.scale, fa.a.shift, fa.b.w, fa.b.scale, fa.b.shift, pad_to=channels,
                                        act1=fa.act)
        return ops.to_ndhwc(fa(feat).unsqueeze(2), pad_to=channels).squeeze(1)

    def _call_tc(self, x, feats):
        """The tensor-core route; x fp32 (3xFP16 split kernels) or fp16 (H16 kernels: the ops dispatch on the activation dtype, every
        intermediate stays fp16, the gates stay fp32)."""
        t = self._tc_pack(x.dtype == torch.float16)
        c = x.shape[1]
        pc, p2, p4 = self._pad32(c), self._pad32(2 * c), self._pad32(4 * c)
        act = lambda name, i: self.conv[name][i][1]                         # noqa: E731
        xc = ops.to_ndhwc(x, pad_to=pc)
        (w0, sc0, sh0), (w1, sc1, sh1) = t["conv1"]
        c1 = ops.conv3d_k3_s2_tc(xc, w0, sc0, sh0, None, act("conv1", 0), out_ndhwc=True)
        conv1 = ops.conv3d_k3_tc(c1, w1, sc1, sh1, None, act("conv1", 1), gate=self._gate_nhwc("8", feats[1], p2))
        (w0, sc0, sh0), (w1, sc1, sh1) = t["conv2"]
        c2 = ops.conv3d_k3_s2_tc(conv1, w0, sc0, sh0, None, act("conv2", 0), out_ndhwc=True)
        conv2 = ops.conv3d_k3_tc(c2, w1, sc1, sh1, None, act("conv2", 1), gate=self._gate_nhwc("16", feats[2], p4))
        if "conv3" in t and self._level32_tc_ok(x.shape):
            # 1/32 level (768 voxels per pair at config 3: one 8 x 16 plane = one M tile) as output-channel slices
            b, d4, h4, w4, _ = conv2.shape
            s0, s1 = t["conv3"]
            y = conv2.new_empty((b, d4 // 2, h4 // 2, w4 // 2, 160))
            for lo, wt, sc, sh in s0:
                ops.tc_slice("s2", conv2, wt, sc, sh, y, lo, act("conv3", 0))
            g32 = self._gate_nhwc("32", feats[3], 160)
            conv3 = torch.empty_like(y)
            for lo, wt, sc, sh in s1:
                ops.tc_slice("s1", y, wt, sc, sh, conv3, lo, act("conv3", 1), gate=g32)
            up3 = conv2.new_empty((b, d4, h4, w4, p4))
            for lo, wt, sc, sh in t["conv3_up"]:
                ops.tc_slice("dc4", conv3, wt, sc, sh, up3, lo, self.up["conv3_up"][1])
        else:
            # 1/32 level on the fp32 CUDA-core kernels (NCDHW): 6 % of the MACs
            conv2_ncdhw = conv2[..., :4 * c].permute(0, 4, 1, 2, 3).contiguous()
            conv3 = self._pair("conv3", conv2_ncdhw, self.att["32"](feats[3]))
            l, a = self.up["conv3_up"]
            up3 = ops.to_ndhwc(_deconv(l, conv3, a), pad_to=p4)
        (wc, scc, shc), (w1, sc1, sh1), (w2, sc2, sh2) = t["agg_0"]
        y = ops.conv1x1_ndhwc_cat(up3, conv2, wc, scc, shc, act("agg_0", 0))
        y = ops.conv3d_k3_tc(y, w1, sc1, sh1, None, act("agg_0", 1))
        conv2 = ops.conv3d_k3_tc(y, w2, sc2, sh2, None, act("agg_0", 2), gate=self._gate_nhwc("up_16", feats[2], p4))
        wu, scu, shu = t["conv2_up"]
        up2 = ops.deconv3d_k4_tc(conv2, wu, scu, shu, None, self.up["conv2_up"][1])
        (wc, scc, shc), (w1, sc1, sh1), (w2, sc2, sh2) = t["agg_1"]
        y = ops.conv1x1_ndhwc_cat(up2, conv1, wc, scc, shc, act("agg_1", 0))
        y = ops.conv3d_k3_tc(y, w1, sc1, sh1, None, act("agg_1", 1))
        conv1 = ops.conv3d_k3_tc(y, w2, sc2, sh2, None, act("agg_1", 2), gate=self._gate_nhwc("up_8", feats[1], p2))
        wu, scu, shu = t["conv1_up"]
        return ops.deconv3d_k4_tc(conv1, wu, scu, shu, None, self.up["conv1_up"][1], out_ndhwc=False, cout_real=c)

    def __call__(self, x, features):
        h16 = self.precision == "fp16" and x.dtype == torch.float16
        x = self._check(x, torch.float16 if h16 else torch.float32)
        self._ensure(x.device)
        feats = [self._check(f) for f in features]
        if h16 and not self._h16_route_ok(x.shape):
            x = x.float()
        if self.tc_route_ok(x.shape):
            mon = self._watch(x.device)
            out = self._call_tc(x, feats)
            if mon is not None:
                mon.poll()
            return out
        g8, g16, g32 = self.att["8"](feats[1]), self.att["16"](feats[2]), self.att["32"](feats[3])
        conv1 = self._pair("conv1", x, g8)
        conv2 = self._pair("conv2", conv1, g16)
        conv3 = self._pair("conv3", conv2, g32)
        l, a = self.up["conv3_up"]
        conv2 = self._agg("agg_0", _deconv(l, conv3, a), conv2, self.att["up_16"](feats[2]))
        l, a = self.up["conv2_up"]
        conv1 = self._agg("agg_1", _deconv(l, conv2, a), conv1, self.att["up_8"](feats[1]))
        l, a = self.up["conv1_up"]
        return _deconv(l, conv1, a)


class StereoBaseCostHead(_Engine):
    """classifier Conv3d(C,1,3) -> softmax -> disparity_regression (stereobase_gru.py:101,163-164).
    ``module`` is the nn.Conv3d classifier."""

    def _pack(self):
        self.layer = _Packed(self.module)

    def __call__(self, geo, maxdisp_lowres):
        geo = self._check(geo)
        self._ensure(geo.device)
        lay = self.layer
        cp = (lay.cin + 31) // 32 * 32
        if (USE_TENSOR_CORES and lay.cout == 1 and lay._w5 is not None and lay.kernel == 3 and lay.stride == 1
                and ops.conv3d_tc_kc(cp, 1, geo.shape[-1]) == 32):
            # 24 -> 1 head on the narrow tensor-core variant: channels zero-padded to 32 while the layout changes (one pass), the
            # generic CUDA-core conv took 0.71 ms at config 3 (profiles/r2_c3_launches.csv)
            if "head" not in lay._tc:
                w = lay._w5.new_zeros((1, cp) + tuple(lay._w5.shape[2:]))
                w[:, :lay.cin] = lay._w5
                lay._tc["head"] = ops.pack_tc_weight(w, 32, pad_cout_to=16)
            mon = self._watch(geo.device)
            logits = ops.conv3d_k3_tc(ops.to_ndhwc(geo, pad_to=cp), lay._tc["head"], lay.scale, lay.shift, None, ACT_NONE,
                                      out_ndhwc=False, res_ndhwc=False)
            if mon is not None:
                mon.poll()
        else:
            logits = _conv(lay, geo)                            # (B,1,D',H',W')
        return ops.softargmin(logits.squeeze(1), maxdisp_lowres, keepdim=True)


# -------------------------------------------------------------------------------------------------- LightStereo
class _PW:
    """1x1 Conv2d (+BN or bias) packed for osb_conv3d_1x1_bn_act_fwd: weight (Cin, Cout)."""
    __slots__ = ("w", "scale", "shift")

    def __init__(self, conv, bn=None):
        self.w = conv.weight.detach().float().reshape(conv.out_channels, conv.in_channels).t().contiguous()
        self.scale, self.shift = ops.fold_bn(bn) if bn is not None else (None, None)
        if conv.bias is not None:
            bias = conv.bias.detach().float()
            self.shift = bias.contiguous() if self.shift is None else (self.shift + bias * self.scale).contiguous()


class _DW:
    """Depthwise Conv2d (+BN or bias)."""
    __slots__ = ("w", "scale", "shift", "stride")

    def __init__(self, conv, bn=None):
        assert conv.groups == conv.in_channels == conv.out_channels and conv.dilation == (1, 1)
        assert conv.padding == (conv.kernel_size[0] // 2, conv.kernel_size[1] // 2) and conv.stride[0] == conv.stride[1]
        self.w = conv.weight.detach().float().reshape(conv.out_channels, *conv.kernel_size).contiguous()
        self.stride = int(conv.stride[0])
        self.scale, self.shift = ops.fold_bn(bn) if bn is not None else (None, None)
        if conv.bias is not None:
            bias = conv.bias.detach().float()
            self.shift = bias.contiguous() if self.shift is None else (self.shift + bias * self.scale).contiguous()


class _InvertedResidual:
    """MobileV2Residual (lightstereo/aggregation.py:63-101): pw+BN+ReLU6 -> dw3x3+BN+ReLU6 -> pw+BN (+ identity)."""

    def __init__(self, m):
        self.pw = _PW(m.pwconv[0], m.pwconv[1])
        self.dw = _DW(m.dwconv[0], m.dwconv[1])
        self.pl = _PW(m.pwliner[0], m.pwliner[1])
        self.res = bool(m.use_res_connect)

    def __call__(self, x):
        h = ops.conv3d_1x1(x, self.pw.w, self.pw.scale, self.pw.shift, act=ACT_RELU6)
        h = ops.dwconv2d(h, self.dw.w, self.dw.scale, self.dw.shift, stride=self.dw.stride, act=ACT_RELU6)
        return ops.conv3d_1x1(h, self.pl.w, self.pl.scale, self.pl.shift, residual=x if self.res else None)


class _StripAttention:
    """AttentionModule (lightstereo/aggregation.py:104-134): cost * conv3(a + sum_k conv_k_2(conv_k_1(a))), a = conv0(feat)."""

    def __init__(self, m):
        self.conv0, self.conv3 = _PW(m.conv0), _PW(m.conv3)
        self.pairs = [(_DW(getattr(m, "conv%d_1" % i)), _DW(getattr(m, "conv%d_2" % i))) for i in range(3)]

    def __call__(self, cost, feat):
        a = ops.conv3d_1x1(feat, self.conv0.w, None, self.conv0.shift)
        acc = a
        for first, second in self.pairs:                        # acc = a + b0 + b1 + b2, accumulated by the second strip conv
            t = ops.dwconv2d(a, first.w, None, first.shift)
            acc = ops.dwconv2d(t, second.w, None, second.shift, residual=acc)
        return ops.conv3d_1x1(acc, self.conv3.w, None, self.conv3.shift, gate=cost)


class LightStereoAggregation(_Engine):
    """Aggregation.forward (lightstereo/aggregation.py:42-60): correlation volume (B, D/4, H/4, W/4) + left features at 1/4, 1/8,
    1/16 -> [(B, D/4, H/4, W/4)].  53 launches for LightStereo-S; no elementwise pass of its own (BN, ReLU6, shortcuts, the
    attention product and the final ReLUs all ride on the producing kernels)."""

    def _pack(self):
        m = self.module
        seq = lambda s: [_InvertedResidual(b) for b in s]
        self.conv0, self.conv2, self.conv4 = seq(m.conv0), seq(m.conv2), seq(m.conv4)
        self.conv1, self.conv3 = _InvertedResidual(m.conv1), _InvertedResidual(m.conv3)
        self.redir1, self.redir2 = _InvertedResidual(m.redir1), _InvertedResidual(m.redir2)
        self.up = []
        for blk in (m.conv5, m.conv6):
            sc, sh = ops.fold_bn(blk[1])
            self.up.append((ops.pack_deconv2d_weight(blk[0].weight), sc, sh))
        self.att = [_StripAttention(a) for a in (m.att0, m.att2, m.att4)] if m.left_att else None

    def __call__(self, x, features_left):
        x = self._check(x)
        self._ensure(x.device)
        feats = [self._check(f) for f in features_left]
        for blk in self.conv0:
            x = blk(x)
        if self.att:
            x = self.att[0](x, feats[0])
        half = self.conv1(x)
        for blk in self.conv2:
            half = blk(half)
        if self.att:
            half = self.att[1](half, feats[1])
        quarter = self.conv3(half)
        for blk in self.conv4:
            quarter = blk(quarter)
        if self.att:
            quarter = self.att[2](quarter, feats[2])
        w5, s5, b5 = self.up[0]
        up = ops.deconv2d_k3s2(quarter, w5, s5, b5, residual=self.redir2(half), act=ACT_RELU)
        w6, s6, b6 = self.up[1]
        return [ops.deconv2d_k3s2(up, w6, s6, b6, residual=self.redir1(x), act=ACT_RELU)]
