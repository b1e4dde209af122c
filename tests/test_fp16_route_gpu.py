"""GPU: the opt-in fp16 route of StereoBase's hourglass (precision="fp16"): the _h16 entry points against an fp64 convolution of the
same fp16 activations with the fp32 epilogue, next to cuDNN fp16 on the same operands; the engine against the CPU oracle and against
the oracle module under autocast; fp16 saturation and the monitor; the default precision unchanged under autocast."""
import pytest
import torch
import torch.nn.functional as F

from oracle import _reference_shim as shim
from oracle import aggregation as oagg
from oracle import seeded_init as si

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def osb():
    import __graft_entry__
    __graft_entry__.build()
    from openstereo_b200 import aggregation, ops
    torch.backends.cudnn.allow_tf32 = False
    return aggregation, ops


def rnd(seed, *shape, scale=1.0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed)) * scale


def _bn(cout, seed):
    return torch.rand(cout, generator=torch.Generator().manual_seed(seed)) + 0.5, rnd(seed + 1, cout, scale=0.1)


def _epilogue(y, sc, sh, gate=None):
    """fp32 epilogue (folded BN, LeakyReLU, gate) on an (B,C,D,H,W) conv result, in float64."""
    y = F.leaky_relu(y * sc.double().view(1, -1, 1, 1, 1) + sh.double().view(1, -1, 1, 1, 1))
    return y if gate is None else y * gate.double().unsqueeze(2)


def _check(got_ncdhw, want, cudnn, what):
    """max abs error <= 2e-3 of the output scale; mean abs error <= 1.25x that of cuDNN fp16 on the same operands."""
    got = got_ncdhw.detach().double().cpu()
    assert got.shape == want.shape, (what, got.shape, want.shape)
    scale = want.abs().max().item()
    err = (got - want).abs()
    ref_mean = (cudnn.double().cpu() - want).abs().mean().item()
    print("%s: max %.2e of scale, mean %.2e vs cuDNN fp16 %.2e" % (what, err.max().item() / scale, err.mean().item(), ref_mean))
    assert err.max().item() <= 2e-3 * scale, what
    assert err.mean().item() <= 1.25 * ref_mean, what


def _half_in(seed, *shape):
    return rnd(seed, *shape).half()                  # the fp16 activations both sides consume


@pytest.mark.parametrize("cin,cout,d,h,w,gated", [(64, 64, 2, 6, 64, True), (64, 64, 3, 4, 64, False),
                                                   (96, 96, 2, 8, 32, True), (96, 96, 1, 5, 32, False)])
def test_conv3d_k3_tc_h16(osb, cin, cout, d, h, w, gated):
    _, ops = osb
    x, wt = _half_in(500, 1, cin, d, h, w), rnd(501, cout, cin, 3, 3, 3, scale=0.1)
    sc, sh = _bn(cout, 502)
    gate = torch.sigmoid(rnd(504, 1, cout, h, w)) if gated else None
    want = _epilogue(F.conv3d(x.double(), wt.double(), padding=1), sc, sh, gate)
    cud = F.conv3d(x.cuda(), wt.half().cuda(), padding=1).float()
    cud = _epilogue(cud.double(), sc.cuda(), sh.cuda(), None if gate is None else gate.cuda()).half()
    wp = ops.pack_tc_weight(wt.cuda(), 16, h16=True)
    g = None if gate is None else gate.permute(0, 2, 3, 1).contiguous().cuda()
    got = ops.conv3d_k3_tc(ops.to_ndhwc(x.cuda()), wp, sc.cuda(), sh.cuda(), None, ops.ACT_LEAKY, gate=g)
    assert got.dtype == torch.float16
    _check(got.permute(0, 4, 1, 2, 3), want, cud, "k3 s1 h16 %d->%d W=%d gate=%s" % (cin, cout, w, gated))


def test_conv3d_k3_tc_h16_padded_channels_are_zero(osb):
    """48 -> 48 zero-padded to 64 -> 64 with the gate, as the 1/8 level runs it: padded channels exactly 0."""
    _, ops = osb
    b, c, cp, d, h, w = 1, 48, 64, 2, 6, 64
    x, wt = _half_in(510, b, c, d, h, w), rnd(511, c, c, 3, 3, 3, scale=0.1)
    sc, sh = _bn(c, 512)
    gate = torch.sigmoid(rnd(514, b, c, h, w))
    wpad = torch.zeros(cp, cp, 3, 3, 3)
    wpad[:c, :c] = wt
    scp, shp = torch.ones(cp), torch.zeros(cp)
    scp[:c], shp[:c] = sc, sh
    gp = torch.zeros(b, h, w, cp)
    gp[..., :c] = gate.permute(0, 2, 3, 1)
    xc = ops.to_ndhwc(x.cuda(), pad_to=cp)
    assert xc.dtype == torch.float16 and (xc[..., c:] == 0).all() and torch.equal(xc[..., :c], x.cuda().permute(0, 2, 3, 4, 1))
    got = ops.conv3d_k3_tc(xc, ops.pack_tc_weight(wpad.cuda(), 16, h16=True), scp.cuda(), shp.cuda(), None, ops.ACT_LEAKY, gate=gp.cuda())
    assert (got[..., c:] == 0).all()
    want = _epilogue(F.conv3d(x.double(), wt.double(), padding=1), sc, sh, gate)
    cud = _epilogue(F.conv3d(x.cuda(), wt.half().cuda(), padding=1).double(), sc.cuda(), sh.cuda(), gate.cuda()).half()
    _check(got[..., :c].permute(0, 4, 1, 2, 3), want, cud, "k3 h16 48 padded to 64")


@pytest.mark.parametrize("cin,cout,d,h,w", [(32, 64, 4, 8, 128), (64, 96, 4, 8, 64)])
def test_conv3d_k3_s2_tc_h16(osb, cin, cout, d, h, w):
    _, ops = osb
    assert ops.conv3d_s2_tc_h16_supported(cin, cout, d, h, w)
    x, wt = _half_in(520, 1, cin, d, h, w), rnd(521, cout, cin, 3, 3, 3, scale=0.1)
    sc, sh = _bn(cout, 522)
    want = _epilogue(F.conv3d(x.double(), wt.double(), stride=2, padding=1), sc, sh)
    cud = _epilogue(F.conv3d(x.cuda(), wt.half().cuda(), stride=2, padding=1).double(), sc.cuda(), sh.cuda()).half()
    got = ops.conv3d_k3_s2_tc(ops.to_ndhwc(x.cuda()), ops.pack_tc_weight(wt.cuda(), 16, kw_order=(1, 0, 2), h16=True), sc.cuda(),
                              sh.cuda(), None, ops.ACT_LEAKY, out_ndhwc=True)
    _check(got.permute(0, 4, 1, 2, 3), want, cud, "k3 s2 h16 %d->%d W=%d" % (cin, cout, w))


@pytest.mark.parametrize("cin,cout,d,h,w,ndhwc", [(96, 64, 3, 8, 32, True), (64, 32, 2, 10, 64, True), (64, 32, 2, 8, 64, False)])
def test_deconv3d_k4_tc_h16(osb, cin, cout, d, h, w, ndhwc):
    _, ops = osb
    x, wt = _half_in(530, 1, cin, d, h, w), rnd(531, cin, cout, 4, 4, 4, scale=0.1)
    sc, sh = _bn(cout, 532)
    want = _epilogue(F.conv_transpose3d(x.double(), wt.double(), stride=2, padding=1), sc, sh)
    cud = _epilogue(F.conv_transpose3d(x.cuda(), wt.half().cuda(), stride=2, padding=1).double(), sc.cuda(), sh.cuda()).half()
    wp = ops.pack_tc_deconv_weight(wt.cuda(), h16=True)
    if ndhwc:
        got = ops.deconv3d_k4_tc(ops.to_ndhwc(x.cuda()), wp, sc.cuda(), sh.cuda(), None, ops.ACT_LEAKY).permute(0, 4, 1, 2, 3)
        _check(got, want, cud, "k4 deconv h16 %d->%d W=%d" % (cin, cout, w))
    else:                                                        # the hourglass's last layer: NCDHW fp16, only the real channels
        creal = cout - 8
        got = ops.deconv3d_k4_tc(ops.to_ndhwc(x.cuda()), wp, sc.cuda(), sh.cuda(), None, ops.ACT_LEAKY, out_ndhwc=False, cout_real=creal)
        assert got.dtype == torch.float16 and got.shape == (1, creal, 2 * d, 2 * h, 2 * w)
        _check(got, want[:, :creal], cud[:, :creal], "k4 deconv h16 ncdhw real channels")


def test_channel_slices_h16_at_width_16(osb):
    """The 1/32 level: 96 -> 160 (96 + 64 slices) stride 2, 160 -> 160 stride 1 with gate, 160 -> 96 (64 + 32) k4 transposed conv."""
    _, ops = osb
    b, d, h, cin, ctot, w = 1, 2, 8, 96, 160, 16
    x, wt = _half_in(540, b, cin, 2 * d, 2 * h, 2 * w), rnd(541, ctot, cin, 3, 3, 3, scale=0.1)
    sc, sh = _bn(ctot, 542)
    want = _epilogue(F.conv3d(x.double(), wt.double(), stride=2, padding=1), sc, sh)
    cud = _epilogue(F.conv3d(x.cuda(), wt.half().cuda(), stride=2, padding=1).double(), sc.cuda(), sh.cuda()).half()
    y = torch.full((b, d, h, w, ctot), float("nan"), device="cuda", dtype=torch.float16)
    xc = ops.to_ndhwc(x.cuda())
    for lo, hi in ((0, 96), (96, 160)):
        ops.tc_slice("s2", xc, ops.pack_tc_weight(wt[lo:hi].cuda(), 16, kw_order=(1, 0, 2), h16=True), sc[lo:hi].contiguous().cuda(),
                     sh[lo:hi].contiguous().cuda(), y, lo, ops.ACT_LEAKY)
    _check(y.permute(0, 4, 1, 2, 3), want, cud, "s2 slices h16 @16")
    x1, wt1 = y.permute(0, 4, 1, 2, 3).contiguous(), rnd(543, ctot, ctot, 3, 3, 3, scale=0.05)
    gate = torch.sigmoid(rnd(544, b, ctot, h, w))
    want1 = _epilogue(F.conv3d(x1.cpu().double(), wt1.double(), padding=1), sc, sh, gate)
    cud1 = _epilogue(F.conv3d(x1, wt1.half().cuda(), padding=1).double(), sc.cuda(), sh.cuda(), gate.cuda()).half()
    y1 = torch.full_like(y, float("nan"))
    for lo, hi in ((0, 96), (96, 160)):
        ops.tc_slice("s1", y, ops.pack_tc_weight(wt1[lo:hi].cuda(), 16, h16=True), sc[lo:hi].contiguous().cuda(),
                     sh[lo:hi].contiguous().cuda(), y1, lo, ops.ACT_LEAKY, gate=gate.permute(0, 2, 3, 1).contiguous().cuda())
    _check(y1.permute(0, 4, 1, 2, 3), want1, cud1, "s1 slices + gate h16 @16")
    wt2 = rnd(545, ctot, 96, 4, 4, 4, scale=0.05)
    sc2, sh2 = _bn(96, 546)
    x2 = y1.permute(0, 4, 1, 2, 3).contiguous()
    want2 = _epilogue(F.conv_transpose3d(x2.cpu().double(), wt2.double(), stride=2, padding=1), sc2, sh2)
    cud2 = _epilogue(F.conv_transpose3d(x2, wt2.half().cuda(), stride=2, padding=1).double(), sc2.cuda(), sh2.cuda()).half()
    y2 = torch.full((b, 2 * d, 2 * h, 2 * w, 96), float("nan"), device="cuda", dtype=torch.float16)
    for lo, hi in ((0, 64), (64, 96)):
        ops.tc_slice("dc4", y1, ops.pack_tc_deconv_weight(wt2[:, lo:hi].contiguous().cuda(), h16=True), sc2[lo:hi].contiguous().cuda(),
                     sh2[lo:hi].contiguous().cuda(), y2, lo, ops.ACT_LEAKY)
    _check(y2.permute(0, 4, 1, 2, 3), want2, cud2, "k4 deconv slices h16 @16")


def test_conv1x1_ndhwc_cat_h16(osb):
    _, ops = osb
    for (c, v) in ((96, 1000), (64, 777)):
        x0, x1 = rnd(550, v, c).half(), rnd(551, v, c).half()
        wt = rnd(552, 2 * c, c, scale=0.1)
        sc, sh = _bn(c, 553)
        want = F.leaky_relu((torch.cat((x0, x1), 1).double() @ wt.double()) * sc.double() + sh.double())
        got = ops.conv1x1_ndhwc_cat(x0.cuda(), x1.cuda(), wt.cuda(), sc.cuda(), sh.cuda(), ops.ACT_LEAKY)
        assert got.dtype == torch.float16
        err = (got.cpu().double() - want).abs() / want.abs().max()
        assert err.max().item() <= 2e-3                        # fp32 arithmetic, one fp16 rounding of the result
        with pytest.raises(ValueError):
            ops.conv1x1_ndhwc_cat(x0.cuda(), x1.float().cuda(), wt.cuda(), sc.cuda(), sh.cuda(), ops.ACT_LEAKY)


def test_h16_saturation_is_counted(osb):
    """An output beyond 65504 is stored as +-65504 (finite) and bumps the sticky fp16-range counter."""
    _, ops = osb
    ops.tc_overflow_count(reset=True)
    x, wt = _half_in(560, 1, 64, 2, 4, 64), rnd(561, 64, 64, 3, 3, 3, scale=0.1)
    wp = ops.pack_tc_weight(wt.cuda(), 16, h16=True)
    got = ops.conv3d_k3_tc(ops.to_ndhwc(x.cuda()), wp, torch.full((64,), 1e5).cuda(), None, None, ops.ACT_NONE)
    assert torch.isfinite(got).all() and got.abs().max().item() == 65504.0
    assert ops.tc_overflow_count(reset=True) >= 1 and ops.tc_overflow_count() == 0
    got = ops.conv3d_k3_tc(ops.to_ndhwc(x.cuda()), wp, None, None, None, ops.ACT_NONE)
    assert ops.tc_overflow_count() == 0
    with pytest.raises(ValueError, match="h16=True"):
        ops.conv3d_k3_tc(ops.to_ndhwc(x.cuda()), ops.pack_tc_weight(wt.cuda(), 16), None, None, None, ops.ACT_NONE)
    with pytest.raises(ValueError, match="h16=False"):
        ops.conv3d_k3_tc(ops.to_ndhwc(x.float().cuda()), wp, None, None, None, ops.ACT_NONE)


def _stereobase_case(b, dq, hq, wq, seed):
    m = oagg.StereoBaseCostHead(24, [96, 64, 192, 160], max_disp=4 * dq).eval()
    m.load_state_dict(si.seeded_state_dict(m.state_dict(), seed=seed, scale={"classifier.weight": 150.0}))
    vol = rnd(seed + 1, b, 24, dq, hq, wq).half()
    feats = [rnd(seed + 2, b, 96, hq, wq), rnd(seed + 3, b, 64, hq // 2, wq // 2), rnd(seed + 4, b, 192, hq // 4, wq // 4),
             rnd(seed + 5, b, 160, hq // 8, wq // 8)]
    return m, vol, [f.half() for f in feats]


@pytest.mark.parametrize("dq,hq", [(8, 16), (48, 64)])
def test_stereobase_hourglass_fp16_route(osb, dq, hq):
    """Hourglass(24, [96, 64, 192, 160]) with precision="fp16" vs the CPU oracle in fp32 on the same fp16-valued inputs, next to the
    oracle module run on the GPU under autocast (cuDNN fp16)."""
    agg, ops = osb
    m, vol, feats = _stereobase_case(1, dq, hq, 128, 570)
    with torch.no_grad():
        want = m.cost_agg(vol.float(), [f.float() for f in feats]).double()
        m.cuda()
        fg = [f.cuda() for f in feats]
        with torch.autocast("cuda", torch.float16):
            amp = m.cost_agg(vol.cuda(), fg).double().cpu()
        eng = agg.StereoBaseAggregation(m.cost_agg, precision="fp16")
        ops.profile_start()
        got = eng(vol.cuda(), fg)
        names = ops.profile_stop()
    assert got.dtype == torch.float16 and got.shape == vol.shape
    assert {"osb_conv3d_k3_tc_gate_h16_fwd", "osb_conv3d_k3_s2_tc_h16_fwd", "osb_deconv3d_k4_tc_h16_fwd", "osb_conv3d_k3_tc_cs_h16_fwd",
            "osb_conv3d_k3_s2_tc_cs_h16_fwd", "osb_deconv3d_k4_tc_cs_h16_fwd", "osb_conv1x1_ndhwc_cat_h16_fwd",
            "osb_ncdhw_to_ndhwc_pad_h16"} <= set(names)
    assert not any(n.startswith("osb_conv3d_k3_tc_gate_fwd") or n == "osb_conv3d_k3_s2_tc_fwd" for n in names)
    err = (got.double().cpu() - want).abs()
    e_amp = (amp - want).abs().mean().item()
    rel = err.max().item() / want.abs().max().item()
    print("fp16 hourglass D'=%d H'=%d: mean %.3e (autocast oracle %.3e), max rel %.2e" % (dq, hq, err.mean().item(), e_amp, rel))
    assert err.mean().item() <= 1.25 * e_amp
    assert rel <= 1e-2
    assert ops.tc_overflow_count() == 0


def test_stereobase_default_precision_unchanged_under_autocast(osb):
    """precision="fp32" (patch()'s default) given fp16 tensors: no _h16 entry point runs and the result is exactly the fp32 route's,
    cast to fp16 the way patch() casts it."""
    agg, ops = osb
    m, vol, feats = _stereobase_case(1, 8, 16, 128, 580)
    m.cuda()
    fg = [f.cuda() for f in feats]
    eng = agg.StereoBaseAggregation(m.cost_agg)
    with torch.no_grad(), torch.autocast("cuda", torch.float16):
        ops.profile_start()
        got = eng(vol.cuda(), fg).to(torch.float16)
        names = ops.profile_stop()
        want = eng(vol.cuda().float(), [f.float() for f in fg]).half()
    assert not any("h16" in n for n in names)
    assert torch.equal(got, want)
    # precision="fp16" with fp32 or bf16 input keeps the fp32 route too
    eng16 = agg.StereoBaseAggregation(m.cost_agg, precision="fp16")
    with torch.no_grad():
        assert torch.equal(eng16(vol.cuda().float(), fg), eng(vol.cuda().float(), fg))
        ops.profile_start()
        eng16(vol.cuda().bfloat16(), fg)
        assert not any("h16" in n for n in ops.profile_stop())


def test_stereobase_fp16_saturation_raises_on_next_call(osb):
    agg, ops = osb
    m, vol, feats = _stereobase_case(1, 8, 16, 128, 590)
    with torch.no_grad():
        m.cost_agg.conv1[0].block[0].weight.mul_(1e6)             # the first layer's outputs leave the fp16 range
    m.cuda()
    fg = [f.cuda() for f in feats]
    ops.tc_overflow_count(reset=True)
    eng = agg.StereoBaseAggregation(m.cost_agg, precision="fp16")
    with torch.no_grad():
        eng(vol.cuda(), fg)
        torch.cuda.synchronize()
        with pytest.raises(RuntimeError, match="fp16 range"):
            eng(vol.cuda(), fg)
    assert ops.tc_overflow_count(reset=True) == 0


@pytest.mark.skipif(not shim.available(), reason="reference tree (oracle/_ref) not staged")
def test_patch_stereobase_reference_class_fp16(osb):
    """The reference's own StereoBase from the unchanged stereobase_sceneflow.yaml (AMP: true) evaluated under autocast at 256x512:
    patch(m, precision="fp16") runs the _h16 entry points, and its init_disp stays within 1.25x (+ 1e-3 px) of the unpatched
    model's own autocast error against the fp32 CPU reference."""
    _, ops = osb
    from openstereo_b200.patch import patch
    shim.install_timm_stub()
    cfg = shim.load_cfg("cfgs/stereobase/stereobase_sceneflow.yaml").MODEL
    m = shim.load("stereo.modeling.models.stereobase.stereobase_gru").StereoBase(cfg).eval()
    m.load_state_dict(si.seeded_state_dict(m.state_dict(), seed=3, scale={"classifier.weight": 8.0}))
    g = torch.Generator().manual_seed(20)
    x = {"left": torch.randn(1, 3, 256, 512, generator=g), "right": torch.randn(1, 3, 256, 512, generator=g)}
    with torch.no_grad():
        want_cpu = m(dict(x))["init_disp"]
        m.cuda()
        xg = {k: v.cuda() for k, v in x.items()}
        with torch.autocast("cuda", torch.float16):
            amp = m(dict(xg))["init_disp"].float().cpu()
            patch(m, precision="fp16")
            ops.profile_start()
            got = m(dict(xg))["init_disp"].float().cpu()
            names = ops.profile_stop()
    e_amp, e_got = (amp - want_cpu).abs().mean().item(), (got - want_cpu).abs().mean().item()
    print("patch(StereoBase, precision='fp16') init_disp EPE %.3e vs CPU fp32 (unpatched autocast %.3e)" % (e_got, e_amp))
    assert "osb_conv3d_k3_tc_gate_h16_fwd" in names and "osb_deconv3d_k4_tc_h16_fwd" in names
    assert e_got <= 1.25 * e_amp + 1e-3
