"""GPU: op-level parity of the CUDA kernels (through the C ABI) against the CPU oracle and the committed golden
vectors.  Tolerances: volumes <= 1e-6 abs (products / means of <= 24 fp32 terms; zeros of the w<d triangle are exact);
soft-argmin <= 1e-4 px on small ranges and, for 192-bin expectations whose value is ~100 px (fp32 ulp 7.6e-6, the
reference's own softmax->mul->sum chain carries the same noise: FasterSoftArgmin vs disparity_regression differ by
4.6e-5, SURVEY.md section 4.3), max <= 5e-4 px with mean <= 5e-5 px -- both far inside the 1e-3 px EPE bar;
conv primitives <= 1e-5 relative to the output scale (fp32 accumulation order differs)."""
import pytest
import torch

from conftest import load_golden

pytestmark = pytest.mark.gpu

from oracle import cost_volume as ocv      # noqa: E402
from oracle import regression as oreg      # noqa: E402


@pytest.fixture(scope="module")
def ops():
    import __graft_entry__
    __graft_entry__.build()
    from openstereo_b200 import ops as _ops
    return _ops


def dev(t):
    return t.cuda()


def rnd(seed, *shape, scale=1.0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed)) * scale


def assert_close(got, want, atol, what=""):
    got = got.detach().cpu()
    assert got.shape == want.shape, (what, got.shape, want.shape)
    err = (got - want).abs().max().item() if want.numel() else 0.0
    assert err <= atol, "%s: max abs err %g > %g" % (what, err, atol)


def assert_zero_triangle(vol, d_axis):
    """Columns w < d must be exactly zero (the reference never writes them after new_zeros)."""
    v = vol.detach().cpu().movedim(d_axis, 0)
    for d in range(v.shape[0]):
        assert (v[d][..., :min(d, v.shape[-1])] == 0).all()


# ------------------------------------------------------------------------------------------------ volumes
@pytest.mark.parametrize("name", ["gwc_small", "gwc_d_gt_w", "gwc_k12", "gwc_k8_w128"])
def test_gwc_volume_golden(ops, name):
    g = load_golden(name)
    out = ops.build_gwc_volume(dev(g["left"]), dev(g["right"]), g["maxdisp"], g["groups"])
    assert out.is_contiguous() and out.dtype == torch.float32
    assert_close(out, g["out"], 1e-6, name)
    assert_zero_triangle(out, 2)


@pytest.mark.parametrize("name", ["concat_small", "concat_d_gt_w", "concat_c12_w128"])
def test_concat_volume_golden(ops, name):
    g = load_golden(name)
    out = ops.build_concat_volume(dev(g["left"]), dev(g["right"]), g["maxdisp"])
    assert torch.equal(out.cpu(), g["out"])                       # pure copy: bit exact
    assert torch.equal(ops.cat_fms(dev(g["left"]), dev(g["right"]), max_disp=g["maxdisp"]).cpu(), g["out"])
    out = ops.build_concat_volume(dev(g["left"]), dev(g["right"]), g["maxdisp"], mask_left=False)
    assert torch.equal(out.cpu(), g["out_unmasked"])


def test_corr_and_fused_golden(ops):
    g = load_golden("corr_small")
    assert_close(ops.correlation_volume(dev(g["left"]), dev(g["right"]), g["maxdisp"]), g["out"], 1e-6, "corr")
    g = load_golden("gwc_concat_fused")
    out = ops.gwc_concat_volume(dev(g["lg"]), dev(g["rg"]), dev(g["lc"]), dev(g["rc"]), g["maxdisp"], g["groups"])
    assert_close(out, g["out"], 1e-6, "fused")
    assert torch.equal(out[:, g["groups"]:].cpu(), g["out"][:, g["groups"]:])   # concat half is a bit-exact copy


@pytest.mark.parametrize("b,c,h,w,d,g", [
    (2, 320, 3, 128, 48, 40),     # GwcNet shape (config 2), few rows
    (1, 96, 2, 160, 48, 8),       # IGEV / StereoBase K=12, two column tiles
    (1, 16, 2, 130, 70, 4),       # W % 4 != 0 (no TMA), two disparity chunks
    (1, 24, 3, 184, 48, 1),       # LightStereo correlation (G=1, K=24)
    (1, 8, 1, 5, 3, 8),           # K = 1
    (3, 12, 2, 36, 9, 3),
])
def test_gwc_volume_vs_oracle(ops, b, c, h, w, d, g):
    l, r = rnd(1, b, c, h, w), rnd(2, b, c, h, w)
    out = ops.build_gwc_volume(dev(l), dev(r), d, g)
    assert_close(out, ocv.build_gwc_volume(l, r, d, g), 1e-6, "gwc %s" % ((b, c, h, w, d, g),))
    assert_zero_triangle(out, 2)


@pytest.mark.parametrize("b,c,h,w,d", [(2, 12, 3, 128, 48), (1, 32, 2, 128, 48), (1, 5, 2, 37, 70), (1, 3, 1, 260, 9)])
def test_concat_volume_vs_oracle(ops, b, c, h, w, d):
    l, r = rnd(3, b, c, h, w), rnd(4, b, c, h, w)
    assert torch.equal(ops.build_concat_volume(dev(l), dev(r), d).cpu(), ocv.build_concat_volume(l, r, d))


def test_fused_volume_gwcnet_shape(ops):
    lg, rg, lc, rc = rnd(5, 1, 320, 2, 128), rnd(6, 1, 320, 2, 128), rnd(7, 1, 12, 2, 128), rnd(8, 1, 12, 2, 128)
    out = ops.gwc_concat_volume(dev(lg), dev(rg), dev(lc), dev(rc), 48, 40)
    assert out.shape == (1, 64, 48, 2, 128)
    assert_close(out, ocv.gwc_concat_volume(lg, rg, lc, rc, 48, 40), 1e-6, "fused gwcnet")


def test_volume_properties_full_size(ops):
    """Config-2 size (B=8, C=320, G=40, 64x128, D'=48): size-independent properties instead of a CPU oracle run.
    (1) linearity in the left feature; (2) the d=0 slice equals the plain group mean of l*r; (3) zero triangle;
    (4) shifting the right image by s columns shifts the disparity axis by s."""
    torch.manual_seed(0)
    l = torch.randn(8, 320, 64, 128, device="cuda")
    r = torch.randn(8, 320, 64, 128, device="cuda")
    v1 = ops.build_gwc_volume(l, r, 48, 40)
    v2 = ops.build_gwc_volume(2.0 * l, r, 48, 40)
    assert torch.equal(v2, 2.0 * v1)                              # scaling by 2 is exact in fp32
    d0 = (l * r).view(8, 40, 8, 64, 128).mean(2)
    assert (v1[:, :, 0] - d0).abs().max().item() <= 1e-6
    assert_zero_triangle(v1[:1], 2)
    s = 5
    r_shift = torch.zeros_like(r)
    r_shift[..., s:] = r[..., :-s]                                # r_shift[w] = r[w-s]
    v3 = ops.build_gwc_volume(l, r_shift, 48, 40)                 # v3[d] pairs l[w] with r[w-d-s] = v1[d+s] where defined
    assert (v3[:, :, :48 - s, :, 48:] - v1[:, :, s:, :, 48:]).abs().max().item() <= 1e-6


def test_half_inputs_roundtrip(ops):
    """Under autocast StereoBase feeds fp16 features (stereobase_sceneflow.yaml:50); output dtype = input dtype."""
    l, r = rnd(9, 1, 16, 2, 32).half(), rnd(10, 1, 16, 2, 32).half()
    out = ops.build_gwc_volume(dev(l), dev(r), 8, 4)
    assert out.dtype == torch.float16
    ref = ocv.build_gwc_volume(l.float(), r.float(), 8, 4)
    assert (out.float().cpu() - ref).abs().max().item() <= 2e-3


def test_reference_assertions(ops):
    x = torch.randn(1, 10, 2, 8, device="cuda")
    with pytest.raises(AssertionError):
        ops.build_gwc_volume(x, x, 4, 3)                          # cost_volume.py:61: C % num_groups
    with pytest.raises(AssertionError):
        ops.disparity_regression(torch.randn(1, 4, 4, device="cuda"), 4)   # disp_regression.py:9


# ------------------------------------------------------------------------------------------------ soft-argmin
def test_softargmin_golden(ops):
    g = load_golden("softargmin_small")
    assert_close(ops.softargmin(dev(g["cost"]), g["maxdisp"]), g["out_keepdim"], 1e-4, "softargmin")
    assert_close(ops.disparity_regression(dev(g["prob"]), g["maxdisp"]), g["out_keepdim"], 1e-4, "regression keepdim")
    assert_close(ops.disparity_regression(dev(g["prob"]), g["maxdisp"], keepdim=False), g["out_flat"], 1e-4, "regression")
    g = load_golden("faster_softargmin")
    assert_close(ops.faster_soft_argmin(dev(g["cost"]), g["maxdisp"]), g["out"], 1e-4, "faster")


def test_upsample_softargmin_golden(ops):
    g = load_golden("upsample_softargmin")
    got = ops.upsample_softargmin(dev(g["cost"]), g["maxdisp"], g["out_h"], g["out_w"], align_corners=False)
    assert_close(got, g["out_gwc"], 1e-4, "gwc tail")
    got = ops.upsample_softargmin(dev(g["cost"]), g["maxdisp"], g["out_h"], g["out_w"], align_corners=True)
    assert_close(got, g["out_psm"], 1e-4, "psm tail")


@pytest.mark.parametrize("align", [False, True])
def test_upsample_softargmin_vs_oracle(ops, align):
    cost = rnd(11, 2, 1, 48, 16, 32, scale=4.0)
    got = ops.upsample_softargmin(dev(cost), 192, 64, 128, align_corners=align)
    want = oreg.upsample_softargmin(cost, 192, 64, 128, align_corners=align, psm_tail=align)
    assert_close(got, want, 5e-4, "upsample align=%s" % align)
    assert (got.cpu() - want).abs().mean().item() <= 5e-5
    assert want.std() > 5.0


def test_softargmin_shapes(ops):
    for shape, scale in [((2, 48, 16, 32), 3.0), ((1, 192, 8, 40), 6.0), ((1, 5, 3, 7), 30.0)]:
        cost = rnd(12, *shape, scale=scale)
        assert_close(ops.softargmin(dev(cost), shape[1]), oreg.softargmin(cost, shape[1]), 5e-4 if shape[1] > 100 else 1e-4, str(shape))
    cost = rnd(13, 1, 24, 4, 9)
    got = ops.faster_soft_argmin(dev(cost), 24, alpha=2.5)
    assert_close(got, oreg.faster_soft_argmin(cost, 24, alpha=2.5), 1e-4, "alpha")


def test_softargmin_properties_full_size(ops):
    """Config-2 size: a one-hot-like cost volume regresses to the argmax; a constant shift of the logits changes nothing."""
    b, d, h, w = 2, 192, 256, 512
    idx = torch.randint(0, d, (b, 1, h, w), device="cuda")
    cost = torch.full((b, d, h, w), -40.0, device="cuda").scatter_(1, idx, 40.0)
    out = ops.softargmin(cost, d, keepdim=False)
    assert (out - idx[:, 0].float()).abs().max().item() <= 1e-4
    out2 = ops.softargmin(cost + 7.0, d, keepdim=False)
    assert (out - out2).abs().max().item() <= 1e-4


def test_epe_partial(ops):
    g = load_golden("epe_per_image")
    got = ops.epe_per_image(dev(g["pred"]), dev(g["gt"]), 192)
    assert_close(got, g["out"], 1e-4, "epe")
    assert got[2].item() == 0.0                                   # image without valid pixels


# ------------------------------------------------------------------------------------------------ conv primitives
def rel_close(got, want, rtol, what):
    got = got.detach().cpu()
    assert got.shape == want.shape, (what, got.shape, want.shape)
    scale = want.abs().max().item() + 1e-12
    err = (got - want).abs().max().item() / scale
    assert err <= rtol, "%s: rel err %g > %g" % (what, err, rtol)


@pytest.mark.parametrize("cin,cout,d,h,w,stride", [
    (8, 32, 8, 8, 32, 1), (32, 32, 5, 7, 19, 1), (12, 24, 6, 6, 40, 1), (16, 1, 4, 9, 33, 1),
    (8, 64, 8, 8, 32, 2), (16, 48, 7, 9, 21, 2), (32, 1, 6, 6, 16, 2), (20, 40, 3, 4, 12, 1),
])
def test_conv3d_k3(ops, cin, cout, d, h, w, stride):
    import torch.nn.functional as F
    x, wt = rnd(20, 2, cin, d, h, w), rnd(21, cout, cin, 3, 3, 3, scale=0.2)
    sc, sh = torch.rand(cout, generator=torch.Generator().manual_seed(22)) + 0.5, rnd(23, cout, scale=0.1)
    want = F.conv3d(x, wt, stride=stride, padding=1)
    res = rnd(24, *want.shape)
    got = ops.conv3d_k3(dev(x), ops.pack_conv_weight(dev(wt)), stride=stride)
    rel_close(got, want, 1e-5, "plain")
    got = ops.conv3d_k3(dev(x), ops.pack_conv_weight(dev(wt)), dev(sc), dev(sh), dev(res), None, stride, ops.ACT_RELU)
    want2 = F.relu(want * sc.view(1, -1, 1, 1, 1) + sh.view(1, -1, 1, 1, 1) + res)
    rel_close(got, want2, 1e-5, "bn+res+relu")
    gate = torch.sigmoid(rnd(25, 2, cout, want.shape[3], want.shape[4]))
    got = ops.conv3d_k3(dev(x), ops.pack_conv_weight(dev(wt)), dev(sc), dev(sh), None, dev(gate), stride, ops.ACT_LEAKY)
    want3 = F.leaky_relu(want * sc.view(1, -1, 1, 1, 1) + sh.view(1, -1, 1, 1, 1)) * gate.unsqueeze(2)
    rel_close(got, want3, 1e-5, "bn+leaky+gate")


@pytest.mark.parametrize("cin,cout,d,h,w,k", [(16, 16, 4, 4, 32, 3), (24, 8, 3, 5, 9, 3), (12, 24, 2, 3, 40, 4),
                                              (8, 16, 4, 4, 32, 4), (128, 64, 3, 4, 8, 3)])
def test_deconv3d(ops, cin, cout, d, h, w, k):
    import torch.nn.functional as F
    x, wt = rnd(30, 2, cin, d, h, w), rnd(31, cin, cout, k, k, k, scale=0.2)
    want = F.conv_transpose3d(x, wt, stride=2, padding=1, output_padding=1 if k == 3 else 0)
    assert want.shape[2:] == (2 * d, 2 * h, 2 * w)
    got = ops.deconv3d(dev(x), ops.pack_deconv_weight(dev(wt)), kernel=k)
    rel_close(got, want, 1e-5, "deconv k%d" % k)
    sc, sh, res = torch.rand(cout) + 0.5, rnd(33, cout, scale=0.1), rnd(34, *want.shape)
    got = ops.deconv3d(dev(x), ops.pack_deconv_weight(dev(wt)), dev(sc), dev(sh), dev(res), k, ops.ACT_RELU)
    rel_close(got, F.relu(want * sc.view(1, -1, 1, 1, 1) + sh.view(1, -1, 1, 1, 1) + res), 1e-5, "deconv fused")


def test_conv3d_1x1(ops):
    import torch.nn.functional as F
    x0, x1 = rnd(40, 2, 24, 3, 5, 16), rnd(41, 2, 40, 3, 5, 16)
    wt = rnd(42, 48, 64, 1, 1, 1, scale=0.2)
    want = F.conv3d(torch.cat((x0, x1), 1), wt)
    got = ops.conv3d_1x1(dev(x0), dev(wt.view(48, 64).t().contiguous()), x1=dev(x1))
    rel_close(got, want, 1e-5, "1x1 two slabs")
    x = rnd(43, 1, 200, 2, 3, 7)                                   # Cin > one weight slab, W % 4 != 0
    wt = rnd(44, 20, 200, 1, 1, 1, scale=0.1)
    sh = rnd(45, 20)
    got = ops.conv3d_1x1(dev(x), dev(wt.view(20, 200).t().contiguous()), None, dev(sh), sigmoid_out=True)
    rel_close(got, torch.sigmoid(F.conv3d(x, wt, bias=sh)), 1e-5, "1x1 sigmoid")
    f = rnd(46, 2, 16, 6, 10)                                      # 2-D feature map (FeatureAtt)
    wt = rnd(47, 8, 16, 1, 1, scale=0.3)
    got = ops.conv3d_1x1(dev(f), dev(wt.view(8, 16).t().contiguous()), act=ops.ACT_LEAKY)
    rel_close(got, F.leaky_relu(F.conv2d(f, wt)), 1e-5, "1x1 2d")


def test_conv1x1_channels_last(ops):
    import torch.nn.functional as F
    for k, (c, v) in enumerate(((32, (2, 3, 5, 37)), (64, (1, 4, 3, 130)))):            # voxel counts not multiples of 256
        x = rnd(48 + k, v[0], c, *v[1:])
        wt = rnd(148 + k, c, c, 1, 1, 1, scale=0.2)
        sc, sh = rnd(150 + k, c).abs() + 0.5, rnd(152 + k, c)
        want = F.relu(F.conv3d(x, wt) * sc.view(1, -1, 1, 1, 1) + sh.view(1, -1, 1, 1, 1)).permute(0, 2, 3, 4, 1)
        got = ops.conv1x1_ndhwc(dev(x.permute(0, 2, 3, 4, 1).contiguous()), dev(wt.view(c, c).t().contiguous()), dev(sc), dev(sh),
                                ops.ACT_RELU)
        rel_close(got, want.contiguous(), 1e-5, "1x1 channels-last C=%d" % c)
    with pytest.raises(RuntimeError):
        ops.conv1x1_ndhwc(dev(rnd(1, 4, 16)), dev(rnd(2, 16, 16)))


def test_conv3d_head_channels_last(ops):
    """Conv3d(32, 1, 3, 1, 1) classifier head on a channels-last input, ragged sizes (partial tiles in D, H and W)."""
    import torch.nn.functional as F
    for k, shape in enumerate(((2, 32, 5, 7, 45), (1, 32, 2, 4, 32), (1, 32, 3, 9, 130))):
        x = rnd(160 + k, *shape)
        wt = rnd(170 + k, 1, 32, 3, 3, 3, scale=0.1)
        want = F.conv3d(x, wt, padding=1)
        got = ops.conv3d_k3_c1_ndhwc(dev(x.permute(0, 2, 3, 4, 1).contiguous()), dev(ops.pack_c1_weight(wt)))
        rel_close(got, want, 1e-5, "head conv %s" % (shape,))
    sc, sh = torch.tensor([1.7]), torch.tensor([-0.3])
    got = ops.conv3d_k3_c1_ndhwc(dev(x.permute(0, 2, 3, 4, 1).contiguous()), dev(ops.pack_c1_weight(wt)), dev(sc), dev(sh))
    rel_close(got, want * 1.7 - 0.3, 1e-5, "head conv scale/shift")
    with pytest.raises(RuntimeError):
        ops.conv3d_k3_c1_ndhwc(dev(rnd(1, 1, 2, 2, 4, 16)), dev(rnd(2, 27, 16)))


# ------------------------------------------------------------------------------------------------ tensor-core conv (3xTF32)
def test_to_ndhwc(ops):
    x = rnd(50, 2, 40, 3, 5, 16)
    assert torch.equal(ops.to_ndhwc(dev(x)).cpu(), x.permute(0, 2, 3, 4, 1).contiguous())


@pytest.mark.parametrize("b,cin,d,h", [(1, 32, 1, 5), (1, 32, 3, 7), (2, 64, 4, 11), (1, 32, 2, 64), (1, 96, 2, 3)])
def test_conv3d_tc_matches_fp32(ops, b, cin, d, h):
    """3xFP16-split tensor-core conv vs the fp32 reference conv: same 1e-5 bar as the CUDA-core kernel."""
    import torch.nn.functional as F
    w, cout = 128, 32
    assert ops.conv3d_tc_supported(cin, cout, w)
    x, wt = rnd(60, b, cin, d, h, w), rnd(61, cout, cin, 3, 3, 3, scale=0.2)
    sc, sh = torch.rand(cout, generator=torch.Generator().manual_seed(62)) + 0.5, rnd(63, cout, scale=0.1)
    want = F.conv3d(x.double(), wt.double(), padding=1).float()
    xc = ops.to_ndhwc(dev(x))
    wp = ops.pack_tc_weight(dev(wt))
    got = ops.conv3d_k3_tc(xc, wp, out_ndhwc=False)
    rel_close(got, want, 1e-5, "tc plain ncdhw-out")
    got = ops.conv3d_k3_tc(xc, wp, out_ndhwc=True)
    rel_close(got.permute(0, 4, 1, 2, 3), want, 1e-5, "tc plain ndhwc-out")
    res = rnd(64, *want.shape)
    want2 = F.relu(want * sc.view(1, -1, 1, 1, 1) + sh.view(1, -1, 1, 1, 1) + res)
    got = ops.conv3d_k3_tc(xc, wp, dev(sc), dev(sh), dev(res), ops.ACT_RELU, out_ndhwc=False, res_ndhwc=False)
    rel_close(got, want2, 1e-5, "tc bn+res+relu ncdhw")
    got = ops.conv3d_k3_tc(xc, wp, dev(sc), dev(sh), dev(res.permute(0, 2, 3, 4, 1).contiguous()), ops.ACT_RELU,
                           out_ndhwc=True, res_ndhwc=True)
    rel_close(got.permute(0, 4, 1, 2, 3), want2, 1e-5, "tc bn+res+relu ndhwc")
    # NCDHW input (the cost volume as the volume kernel wrote it): same numbers, no layout-conversion pass
    got = ops.conv3d_k3_tc(dev(x), wp, dev(sc), dev(sh), dev(res), ops.ACT_RELU, out_ndhwc=False, res_ndhwc=False, in_ncdhw=True)
    rel_close(got, want2, 1e-5, "tc ncdhw-in")
    assert ops.tc_overflow_count() == 0


@pytest.mark.parametrize("cout", [1, 3, 16])
def test_conv3d_tc_narrow_head(ops, cout):
    """Classifier heads (32 -> 1, gwcnet_disp_processor.py:60-70) on the COUT = 16 instantiation: weights zero-padded to 16 rows,
    only the real channels are written; NCDHW residual = PSMNet's cost_{i-1} (psmnet_cost_processor.py:196-198)."""
    import torch.nn.functional as F
    x, wt = rnd(65, 2, 32, 3, 7, 128), rnd(66, cout, 32, 3, 3, 3, scale=0.2)
    want = F.conv3d(x.double(), wt.double(), padding=1).float()
    wp = ops.pack_tc_weight(dev(wt), 32, pad_cout_to=16)
    got = ops.conv3d_k3_tc(ops.to_ndhwc(dev(x)), wp, out_ndhwc=False, res_ndhwc=False)
    assert got.shape == want.shape
    rel_close(got, want, 1e-5, "narrow head")
    res, sh = rnd(67, *want.shape), rnd(68, cout, scale=0.1)
    got = ops.conv3d_k3_tc(ops.to_ndhwc(dev(x)), wp, None, dev(sh), dev(res), out_ndhwc=False, res_ndhwc=False)
    rel_close(got, want + sh.view(1, -1, 1, 1, 1) + res, 1e-5, "narrow head + bias + residual")


def test_tc_fp16_range_guard(ops):
    """Activations beyond +-4094 do not fit the fp16 operand split: conversions saturate (finite output) and the sticky counter
    reports it; in-range inputs with a huge dynamic range (1e-6 .. 1e3) keep fp32-level accuracy."""
    import torch.nn.functional as F
    ops.tc_overflow_count(reset=True)
    wt = rnd(81, 32, 32, 3, 3, 3, scale=0.1)
    wp = ops.pack_tc_weight(dev(wt))
    x = rnd(80, 1, 32, 2, 5, 128) * torch.logspace(-6, 3, 128).view(1, 1, 1, 1, 128)
    got = ops.conv3d_k3_tc(ops.to_ndhwc(dev(x)), wp, out_ndhwc=False)
    want = F.conv3d(x.double(), wt.double(), padding=1).float()
    assert ops.tc_overflow_count() == 0
    err = (got.cpu() - want).abs()
    col_scale = want.abs().amax(dim=(0, 1, 2, 3)).clamp(min=1e-7)                # per-column magnitude spans 9 decades
    assert (err.amax(dim=(0, 1, 2, 3)) <= 2e-5 * col_scale + 1e-8).all()
    x[0, 0, 0, 0, 5] = 1e4
    got = ops.conv3d_k3_tc(ops.to_ndhwc(dev(x)), wp, out_ndhwc=False)
    assert torch.isfinite(got).all() and ops.tc_overflow_count(reset=True) >= 1 and ops.tc_overflow_count() == 0


@pytest.mark.parametrize("b,cin,cout,d,h,w", [
    (1, 64, 64, 3, 8, 64),      # GwcNet/PSMNet conv2 @ 1/8 (two image rows per M tile)
    (2, 16, 64, 2, 5, 64),      # ragged H (5 rows, blocks of 4)
    (1, 128, 128, 3, 8, 32),    # GwcNet conv4 @ 1/16 (four rows per tile, N = 3 x 128)
    (1, 64, 64, 2, 16, 32),     # PSMNet conv4
    (1, 32, 128, 1, 3, 32),     # ragged H, single plane
    (2, 64, 64, 1, 7, 128),     # 2D backbone layer2 as a one-plane volume: full-width rows, two tiles per item, ragged H
    (1, 128, 128, 1, 5, 128),   # 2D backbone layer3: N = 3 x 128 at full width
    (1, 64, 64, 2, 4, 128),     # the same kernel on a real volume (kd taps live)
])
def test_conv3d_tc_generic_tiles(ops, b, cin, cout, d, h, w):
    """Multi-row-tile tensor-core conv (conv3d_tcg.cu) vs the fp64 reference conv."""
    import torch.nn.functional as F
    assert ops.conv3d_tc_supported(cin, cout, w) and ops.conv3d_tc_kc(cin, cout, w) == 16
    x, wt = rnd(70, b, cin, d, h, w), rnd(71, cout, cin, 3, 3, 3, scale=0.2)
    sc, sh = torch.rand(cout, generator=torch.Generator().manual_seed(72)) + 0.5, rnd(73, cout, scale=0.1)
    want = F.conv3d(x.double(), wt.double(), padding=1).float()
    xc = ops.to_ndhwc(dev(x))
    wp = ops.pack_tc_weight(dev(wt), 16)
    got = ops.conv3d_k3_tc(xc, wp, out_ndhwc=False)
    rel_close(got, want, 1e-5, "tcg plain ncdhw-out")
    res = rnd(74, *want.shape)
    want2 = F.relu(want * sc.view(1, -1, 1, 1, 1) + sh.view(1, -1, 1, 1, 1) + res)
    got = ops.conv3d_k3_tc(xc, wp, dev(sc), dev(sh), dev(res), ops.ACT_RELU, out_ndhwc=False, res_ndhwc=False)
    rel_close(got, want2, 1e-5, "tcg bn+res+relu ncdhw")
    got = ops.conv3d_k3_tc(xc, wp, dev(sc), dev(sh), dev(res.permute(0, 2, 3, 4, 1).contiguous()), ops.ACT_RELU,
                           out_ndhwc=True, res_ndhwc=True)
    rel_close(got.permute(0, 4, 1, 2, 3), want2, 1e-5, "tcg bn+res+relu ndhwc")


@pytest.mark.parametrize("dil,b,c,h", [(2, 2, 128, 9), (1, 1, 64, 6), (2, 1, 128, 2)])
def test_conv2d_tc_dilated(ops, dil, b, c, h):
    """3x3 Conv2d (dilation 1 / 2, padding = dilation) of the backbone's residual blocks on the tensor cores, full-width rows."""
    import torch.nn.functional as F
    w = 128
    assert ops.conv2d_tc_kc(c, c, w, dil) == 16 and ops.conv2d_tc_kc(64, 64, w, 2) == 0
    x, wt = rnd(180, b, c, h, w), rnd(181, c, c, 3, 3, scale=0.1)
    bias, res = rnd(182, c, scale=0.1), rnd(183, b, c, h, w)
    want = F.relu(F.conv2d(x.double(), wt.double(), bias.double(), padding=dil, dilation=dil).float() + res)
    w5 = torch.zeros(c, c, 3, 3, 3)
    w5[:, :, 1] = wt
    wp = ops.pack_tc_weight(dev(w5), 16)
    xc = dev(x.permute(0, 2, 3, 1).contiguous())
    got = ops.conv2d_k3_tc(xc, wp, None, dev(bias), dev(res.permute(0, 2, 3, 1).contiguous()), ops.ACT_RELU, dil)
    rel_close(got.permute(0, 3, 1, 2), want, 1e-5, "conv2d tc nhwc dil=%d" % dil)
    got = ops.conv2d_k3_tc(xc, wp, None, dev(bias), dev(res), ops.ACT_RELU, dil, out_nhwc=False, res_nhwc=False)
    rel_close(got, want, 1e-5, "conv2d tc nchw dil=%d" % dil)


@pytest.mark.parametrize("b,cin,cout,d,h,w", [
    (1, 32, 64, 4, 8, 128),     # GwcNet/PSMNet conv1: 1/4 -> 1/8 res
    (2, 16, 64, 2, 6, 128),     # ragged output rows (3 rows, blocks of 4)
    (1, 64, 128, 4, 8, 64),     # GwcNet conv3: 1/8 -> 1/16 res (N = 128 + 256)
    (1, 64, 64, 2, 16, 64),     # PSMNet conv3
])
def test_conv3d_s2_tc(ops, b, cin, cout, d, h, w):
    """Stride-2 tensor-core conv (conv3d_tcs2.cu) vs the fp64 reference conv."""
    import torch.nn.functional as F
    assert ops.conv3d_s2_tc_supported(cin, cout, d, h, w)
    x, wt = rnd(80, b, cin, d, h, w), rnd(81, cout, cin, 3, 3, 3, scale=0.2)
    sc, sh = torch.rand(cout, generator=torch.Generator().manual_seed(82)) + 0.5, rnd(83, cout, scale=0.1)
    want = F.conv3d(x.double(), wt.double(), stride=2, padding=1).float()
    xc = ops.to_ndhwc(dev(x))
    wp = ops.pack_tc_weight(dev(wt), 16, kw_order=(1, 0, 2))
    got = ops.conv3d_k3_s2_tc(xc, wp)
    rel_close(got, want, 1e-5, "s2 tc plain")
    res = rnd(84, *want.shape)
    want2 = F.relu(want * sc.view(1, -1, 1, 1, 1) + sh.view(1, -1, 1, 1, 1) + res)
    got = ops.conv3d_k3_s2_tc(xc, wp, dev(sc), dev(sh), dev(res), ops.ACT_RELU)
    rel_close(got, want2, 1e-5, "s2 tc bn+res+relu")
    got = ops.conv3d_k3_s2_tc(xc, wp, dev(sc), dev(sh), None, ops.ACT_RELU, out_ndhwc=True)
    rel_close(got.permute(0, 4, 1, 2, 3), F.relu(want * sc.view(1, -1, 1, 1, 1) + sh.view(1, -1, 1, 1, 1)), 1e-5, "s2 tc ndhwc out")


@pytest.mark.parametrize("b,cin,cout,d,h,w", [
    (1, 128, 64, 3, 8, 32),     # GwcNet conv5: 1/16 -> 1/8 res
    (2, 64, 64, 2, 5, 32),      # PSMNet conv5, ragged rows
    (1, 64, 32, 3, 10, 64),     # conv6: 1/8 -> 1/4 res (five 2-row tiles per item)
    (2, 16, 32, 1, 3, 64),      # ragged, single input plane
    (1, 32, 32, 4, 9, 64),      # conv6 shape class on the parity-quad kernel (channels-last calls): odd row count, 4 planes
    (1, 64, 32, 2, 1, 64),      # one input row
])
def test_deconv3d_tc(ops, b, cin, cout, d, h, w):
    """Transposed conv on the tensor cores (conv3d_tcdc.cu) vs the fp64 reference."""
    import torch.nn.functional as F
    assert ops.deconv3d_tc_supported(cin, cout, w)
    x, wt = rnd(90, b, cin, d, h, w), rnd(91, cin, cout, 3, 3, 3, scale=0.2)
    sc, sh = torch.rand(cout, generator=torch.Generator().manual_seed(92)) + 0.5, rnd(93, cout, scale=0.1)
    want = F.conv_transpose3d(x.double(), wt.double(), stride=2, padding=1, output_padding=1).float()
    xc = ops.to_ndhwc(dev(x))
    wp = ops.pack_tc_deconv_weight(dev(wt))
    got = ops.deconv3d_k3_tc(xc, wp)
    rel_close(got, want, 1e-5, "deconv tc plain")
    res = rnd(94, *want.shape)
    want2 = F.relu(want * sc.view(1, -1, 1, 1, 1) + sh.view(1, -1, 1, 1, 1) + res)
    got = ops.deconv3d_k3_tc(xc, wp, dev(sc), dev(sh), dev(res), ops.ACT_RELU)
    rel_close(got, want2, 1e-5, "deconv tc bn+res+relu")
    got = ops.deconv3d_k3_tc(xc, wp, dev(sc), dev(sh), dev(res.permute(0, 2, 3, 4, 1).contiguous()), ops.ACT_RELU,
                             out_ndhwc=True, res_ndhwc=True)
    rel_close(got.permute(0, 4, 1, 2, 3), want2, 1e-5, "deconv tc ndhwc")


@pytest.mark.timeout(120)
def test_tc_kernels_partial_blocks_many_items(ops):
    """Regression for the accumulator hand-off: work items whose row block is partial leave accumulator tiles unused; with
    several such items per persistent CTA and a slow epilogue (residual reads) the unused tiles' barriers used to complete
    twice and alias in parity (deadlock).  Shapes: H=32 with 10-row blocks (deconv, 5 tiles) and H=68 with 5-row blocks."""
    x = torch.randn(4, 64, 12, 32, 64, device="cuda")
    wt = torch.randn(64, 32, 3, 3, 3, device="cuda") * 0.1
    sc, sh = torch.rand(32, device="cuda") + 0.5, torch.randn(32, device="cuda") * 0.1
    res = torch.randn(4, 32, 24, 64, 128, device="cuda")
    ref = ops.deconv3d(x, ops.pack_deconv_weight(wt), sc, sh, res, 3, ops.ACT_RELU)
    for _ in range(3):
        got = ops.deconv3d_k3_tc(ops.to_ndhwc(x), ops.pack_tc_deconv_weight(wt), sc, sh, res, ops.ACT_RELU)
    torch.cuda.synchronize()
    assert ((got - ref).abs().max() / ref.abs().max()).item() <= 1e-5
    x = torch.randn(2, 32, 6, 68, 128, device="cuda")            # 68 rows = 13 full blocks of 5 + one of 3
    wt = torch.randn(32, 32, 3, 3, 3, device="cuda") * 0.1
    res = torch.randn(2, 32, 6, 68, 128, device="cuda")
    ref = ops.conv3d_k3(x, ops.pack_conv_weight(wt), sc, sh, res, None, 1, ops.ACT_RELU)
    for _ in range(3):
        got = ops.conv3d_k3_tc(ops.to_ndhwc(x), ops.pack_tc_weight(wt), sc, sh, res, ops.ACT_RELU, out_ndhwc=False, res_ndhwc=False)
    torch.cuda.synchronize()
    assert ((got - ref).abs().max() / ref.abs().max()).item() <= 1e-5


# ------------------------------------------------------------------------------------------------ SURVEY 8(f) row 4 (first piece)
def test_disparity_regression_interval_golden(ops):
    """IGEV++'s strided expectation on the soft-argmin kernel (normalize off, step = interval) vs the reference output."""
    g = load_golden("regression_flavours")
    out = ops.disparity_regression_interval(dev(g["prob"]), g["maxdisp"], g["interval"])
    assert out.shape == g["out_interval"].shape
    assert_close(out, g["out_interval"], 1e-5 * g["maxdisp"], "interval regression")


def test_gwc_normalized_and_coex_golden(ops):
    """FoundationStereo's L2-normalised gwc volume and CoExCostVolume vs the outputs of the unmodified reference functions
    (tests/golden, tools/make_golden.py: flavours).  <= 2e-6 abs on values of magnitude <= 1 (normalised) / <= 1e-5 of the scale."""
    g = load_golden("gwc_normalized")
    out = ops.build_gwc_volume_normalized(dev(g["left"]), dev(g["right"]), g["maxdisp"], g["groups"])
    assert out.shape == g["out"].shape
    assert_close(out, g["out"], 2e-6, "normalised gwc volume")
    w = g["left"].shape[-1]
    for d in range(1, min(g["maxdisp"], w)):
        assert (out[:, :, d, :, :d] == 0).all()
    g = load_golden("coex_volume")
    out = ops.coex_cost_volume(dev(g["left"]), dev(g["right"]), g["maxdisp"], g["group"])
    assert out.shape == g["out"].shape
    assert_close(out, g["out"], 1e-5 * float(g["out"].abs().max()), "CoEx volume")


def test_sub_volume_vs_oracle_and_reference(ops):
    """build_sub_volume (cost_volume.py:108-117): CPU restatement, and the output of the reference's own function on the same
    inputs (tests/golden/sub_volume_reference.npz; whole, or a seeded sample of its elements)."""
    from oracle import cost_volume as ocv
    g = load_golden("sub_volume_reference")
    for shape, d in (((2, 12, 5, 37), 9), ((1, 96, 4, 128), 48), ((1, 3, 2, 6), 8)):
        l, r = rnd(70, *shape), rnd(71, *shape)
        got = ops.build_sub_volume(dev(l), dev(r), d)
        want = ocv.build_sub_volume(l, r, d)
        assert got.shape == want.shape
        tol = 1e-5 * float(want.abs().max())
        assert_close(got, want, tol, "sub volume vs oracle")
        key = "sub_%s_%d" % ("_".join(map(str, shape)), d)
        if key in g:
            assert_close(got, g[key], tol, "sub volume vs the reference")
        else:
            assert_close(got.cpu().reshape(-1)[g[key + "__idx"].long()], g[key + "__val"], tol, "sub volume vs the reference")


def test_disparity_regression_values_golden(ops):
    g = load_golden("regression_flavours")
    out = ops.disparity_regression_values(dev(g["prob"]), dev(g["values"]))
    assert out.shape == g["out_values"].shape
    assert_close(out, g["out_values"], 1e-5 * float(g["out_values"].abs().max()), "explicit-hypothesis regression")
