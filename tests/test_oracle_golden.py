"""CPU: the oracle restatement reproduces the reference's own outputs (tests/golden/*.npz,
written by tools/make_golden.py from the unmodified reference) BIT-EXACTLY.

Exception: outputs of CPU kernels whose summation order depends on the host CPU -- 3D/2D convolutions, the geometry
lookup's batched matmul, trilinear interpolation, the per-image EPE mean -- agree with vectors stored on another host to
within fp32 reordering, REORDER of the output's largest magnitude (assert_reordered); on the host that wrote them they
are bit-equal."""
import pytest
import torch

from oracle import aggregation as oagg
from oracle import cost_volume as ocv
from oracle import geo_lookup as ogeo
from oracle import models as omodels
from oracle import regression as oreg
from oracle import seeded_init as si

from conftest import load_golden


REORDER = 1e-5


def assert_reordered(got, want):
    assert got.shape == want.shape
    assert (got - want).abs().max().item() <= REORDER * want.abs().max().item()


def checksum(sd):
    return float(sum(v.double().abs().sum() for v in sd.values()))


@pytest.mark.parametrize("name", ["gwc_small", "gwc_d_gt_w", "gwc_k12", "gwc_k8_w128"])
def test_gwc_volume(name):
    g = load_golden(name)
    assert torch.equal(ocv.build_gwc_volume(g["left"], g["right"], g["maxdisp"], g["groups"]), g["out"])


@pytest.mark.parametrize("name", ["concat_small", "concat_d_gt_w", "concat_c12_w128"])
def test_concat_volume(name):
    g = load_golden(name)
    assert torch.equal(ocv.build_concat_volume(g["left"], g["right"], g["maxdisp"]), g["out"])
    assert torch.equal(ocv.cat_fms(g["left"], g["right"], max_disp=g["maxdisp"]), g["out"])
    assert torch.equal(ocv.build_concat_volume(g["left"], g["right"], g["maxdisp"], mask_left=False), g["out_unmasked"])


@pytest.mark.parametrize("name", ["cat_fms_neg", "cat_fms_dil"])
def test_cat_fms_variants(name):
    g = load_golden(name)
    out = ocv.cat_fms(g["left"], g["right"], max_disp=g["max_disp"], start_disp=g["start_disp"], dilation=g["dilation"])
    assert torch.equal(out, g["out"])


def test_corr_and_fused():
    g = load_golden("corr_small")
    assert torch.equal(ocv.correlation_volume(g["left"], g["right"], g["maxdisp"]), g["out"])
    g = load_golden("gwc_concat_fused")
    assert torch.equal(ocv.gwc_concat_volume(g["lg"], g["rg"], g["lc"], g["rc"], g["maxdisp"], g["groups"]), g["out"])


def test_regression_tails():
    g = load_golden("softargmin_small")
    assert torch.equal(oreg.disparity_regression(g["prob"], g["maxdisp"], keepdim=True), g["out_keepdim"])
    assert torch.equal(oreg.disparity_regression(g["prob"], g["maxdisp"], keepdim=False), g["out_flat"])
    assert torch.equal(oreg.softargmin(g["cost"], g["maxdisp"]), g["out_keepdim"])
    g = load_golden("faster_softargmin")
    assert torch.equal(oreg.faster_soft_argmin(g["cost"], g["maxdisp"]), g["out"])
    with pytest.raises(ValueError):
        oreg.faster_soft_argmin(g["cost"][0], g["maxdisp"])
    g = load_golden("upsample_softargmin")
    assert_reordered(oreg.upsample_softargmin(g["cost"], g["maxdisp"], g["out_h"], g["out_w"]), g["out_gwc"])
    assert_reordered(oreg.upsample_softargmin(g["cost"], g["maxdisp"], g["out_h"], g["out_w"], align_corners=True,
                                              psm_tail=True), g["out_psm"])
    g = load_golden("epe_per_image")
    mask = (g["gt"] < 192) & (g["gt"] > 0)
    assert_reordered(oreg.epe_per_image(g["pred"], g["gt"], mask), g["out"])


def test_modules():
    with torch.no_grad():
        g = load_golden("gwc_hourglass_c8")
        m = oagg.GwcHourglass(8).eval()
        sd = si.seeded_state_dict(m.state_dict(), seed=g["seed"])
        assert checksum(sd) == pytest.approx(g["sd_checksum"], rel=1e-12)
        m.load_state_dict(sd)
        assert_reordered(m(g["x"]), g["out"])

        g = load_golden("gwc_disp_processor")
        m = oagg.GwcDispProcessor(maxdisp=32, downsample=4, num_groups=4, use_concat_volume=True, concat_channels=2).eval()
        m.load_state_dict(si.seeded_state_dict(m.state_dict(), seed=g["seed"], scale={"classif3.2.weight": 60.0}))
        assert_reordered(m(g["volume"], 32, 64), g["out"])

        g = load_golden("psm_aggregator")
        m = oagg.PSMAggregator(32, 8).eval()
        m.load_state_dict(si.seeded_state_dict(m.state_dict(), seed=g["seed"], scale={
            "classif1.1.weight": 20.0, "classif2.1.weight": 20.0, "classif3.1.weight": 20.0}))
        low = m.aggregate(g["raw"])
        assert_reordered(low[2], g["cost3_low"])
        assert_reordered(low[0], g["cost1_low"])

        g = load_golden("stereobase_head")
        m = oagg.StereoBaseCostHead(8, [16, 16, 24, 20], max_disp=64).eval()
        sd = si.seeded_state_dict(m.state_dict(), seed=g["seed_head"], scale={"classifier.weight": 30.0})
        sd_h = si.seeded_state_dict(m.cost_agg.state_dict(), seed=g["seed_hourglass"])
        sd.update({"cost_agg." + k: v for k, v in sd_h.items()})
        m.load_state_dict(sd)
        geo, init_disp = m(g["volume"], [g["f0"], g["f1"], g["f2"], g["f3"]])
        assert_reordered(geo, g["geo"])
        assert_reordered(init_disp, g["init_disp"])


def test_gwcnet_model():
    g = load_golden("gwcnet_64x128")
    m = omodels.GwcNet().eval()
    sd = si.seeded_state_dict(m.state_dict(), seed=g["seed"], scale=si.GWCNET_SCALE)
    assert checksum(sd) == pytest.approx(g["sd_checksum"], rel=1e-12)
    m.load_state_dict(sd)
    with torch.no_grad():
        out = m({"left": g["left"], "right": g["right"]})["disp_pred"]
    assert_reordered(out, g["out"])
    assert out.std() > 10.0          # the seeded init is not the degenerate constant-95.5 case


def test_psmnet_model():
    g = load_golden("psmnet_256x256")
    m = omodels.PSMNet().eval()
    m.load_state_dict(si.seeded_state_dict(m.state_dict(), seed=g["seed"], scale=si.PSMNET_SCALE, keep=si.PSMNET_KEEP))
    with torch.no_grad():
        out = m({"left": g["left"], "right": g["right"]})["disp_pred"]
    assert_reordered(out, g["out"])


@pytest.mark.parametrize("name", ["geo_lookup_small", "geo_lookup_3lvl"])
def test_geo_lookup(name):
    """SURVEY.md section 8(f) row 1: the oracle reproduces the reference's lookup output and pyramids."""
    g = load_golden(name)
    vol = ogeo.GeoEncodingVolume(g["fmap1"], g["fmap2"], g["volume"], num_levels=g["levels"], radius=g["radius"])
    assert_reordered(vol(g["disp"], g["coords"]), g["out"])
    assert torch.equal(vol.geo_pyramid[-1], g["geo_last"])                        # pooling only: bit for bit
    assert_reordered(vol.corr_pyramid[-1], g["corr_last"])
    assert g["out"].shape[1] == g["levels"] * (g["volume"].shape[1] + 1) * (2 * g["radius"] + 1)


def test_context_upsample():
    g = load_golden("context_upsample")
    assert_reordered(ogeo.context_upsample(g["disp_low"], g["up_weights"], g["scale"]), g["out"])


def test_row4_volume_and_regression_flavours():
    """SURVEY.md section 8(f) row 4: oracle restatements pinned against the reference ahead of their kernels."""
    g = load_golden("gwc_normalized")
    out = ocv.build_gwc_volume_normalized(g["left"], g["right"], g["maxdisp"], g["groups"])
    assert torch.equal(out, g["out"]) and out.abs().max() <= 1.0 + 1e-6          # cosine similarities
    g = load_golden("coex_volume")
    assert torch.equal(ocv.coex_cost_volume(g["left"], g["right"], g["maxdisp"], g["group"]), g["out"])
    assert g["out"].shape[2] == g["maxdisp"] + 1
    g = load_golden("corr_volume_quirk")
    out = ocv.build_corr_volume(g["left"], g["right"], g["maxdisp"])
    assert torch.equal(out, g["out"])
    w = g["left"].shape[-1]
    assert torch.equal(out[:, w], out[:, 0])                                     # hypotheses d >= W correlate the unshifted images
    g = load_golden("regression_flavours")
    assert torch.equal(oreg.disparity_regression_interval(g["prob"], g["maxdisp"], g["interval"]), g["out_interval"])
    assert torch.equal(oreg.disparity_regression_values(g["prob"], g["values"]), g["out_values"])


def test_lightstereo_aggregation():
    """SURVEY.md section 8(f) row 2: the restated MobileNetV2-block hourglass + strip attention reproduces the reference output."""
    from oracle import lightstereo as olight
    g = load_golden("lightstereo_aggregation")
    m = olight.Aggregation(in_channels=12, left_att=True, blocks=[1, 2, 2], expanse_ratio=4, backbone_channels=[10, 14, 18]).eval()
    sd = si.seeded_state_dict(m.state_dict(), seed=g["seed"])
    assert abs(checksum(sd) - g["sd_checksum"]) <= 1e-6 * g["sd_checksum"]
    m.load_state_dict(sd)
    with torch.no_grad():
        out = m(g["x"], [g["f0"], g["f1"], g["f2"]])[0]
    assert_reordered(out, g["out"])
    assert out.std() > 1e-3
