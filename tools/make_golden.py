#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the UNMODIFIED reference (authoring container only).

    python tools/make_golden.py [group ...]     # needs the reference tree (oracle/_reference_shim.py); groups: GROUPS below

For every case: seeded inputs -> the reference's own function/module (imported through
oracle/_reference_shim.py) -> outputs saved next to the inputs.  While generating, the script also
asserts that the oracle restatement is BIT-EQUAL to the reference on the same inputs; that is what
"the oracle is pinned against outputs of the reference itself" means (oracle/__init__.py).

Module weights are not stored (GwcNet is 27 MB): they are regenerated from
``oracle.seeded_init.seeded_state_dict(seed)``, and a checksum of the generated state_dict is stored
so a drift of torch's CPU RNG would be detected instead of silently changing the test.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import _reference_shim as shim                      # noqa: E402
from oracle import aggregation as oagg                          # noqa: E402
from oracle import cost_volume as ocv                           # noqa: E402
from oracle import geo_lookup as ogeo                           # noqa: E402
from oracle import lightstereo as olight                        # noqa: E402
from oracle import models as omodels                            # noqa: E402
from oracle import regression as oreg                           # noqa: E402
from oracle import seeded_init as si                            # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def rnd(seed, *shape, scale=1.0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed)) * scale


def checksum(sd):
    return float(sum(v.double().abs().sum() for v in sd.values()))


def save(name, **arrays):
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **{k: (v.detach().numpy() if torch.is_tensor(v) else np.asarray(v))
                                 for k, v in arrays.items()})
    print("%-34s %8.1f KB" % (name, os.path.getsize(path) / 1024))


def must_equal(a, b, what):
    if not torch.equal(a, b):
        raise SystemExit("oracle != reference for %s (max diff %g)" % (what, (a - b).abs().max()))


def volumes():
    rcv = shim.load("stereo.modeling.cost_volume.cost_volume")
    rgw = shim.load("stereo.modeling.models.gwcnet.gwcnet_cost_processor")
    rpsm = shim.load("stereo.modeling.models.psmnet.psmnet_cost_processor")
    rigev = shim.load("stereo.modeling.models.igev.submodule")
    # (name, B, C, H, W, D, G)
    for name, b, c, h, w, d, g in [("gwc_small", 2, 24, 5, 20, 6, 4), ("gwc_d_gt_w", 1, 16, 3, 7, 10, 2),
                                   ("gwc_k12", 1, 96, 4, 33, 12, 8), ("gwc_k8_w128", 1, 64, 2, 128, 48, 8)]:
        l, r = rnd(1, b, c, h, w), rnd(2, b, c, h, w)
        ref = rcv.build_gwc_volume(l, r, d, g)
        must_equal(ref, ocv.build_gwc_volume(l, r, d, g), name)
        # the GwcNet method copy is the same function (gwcnet_cost_processor.py:22-39)
        proc = rgw.GwcVolumeCostProcessor(maxdisp=d * 4, downsample=4, num_groups=g)
        must_equal(ref, proc.build_gwc_volume(l, r), name + "/method")
        save(name, left=l, right=r, maxdisp=d, groups=g, out=ref)
    for name, b, c, h, w, d in [("concat_small", 2, 6, 5, 20, 6), ("concat_d_gt_w", 1, 4, 3, 7, 10),
                                ("concat_c12_w128", 1, 12, 2, 128, 48)]:
        l, r = rnd(3, b, c, h, w), rnd(4, b, c, h, w)
        ref = rcv.build_concat_volume(l, r, d)
        must_equal(ref, ocv.build_concat_volume(l, r, d), name)
        must_equal(ref, rpsm.cat_fms(l, r, max_disp=d), name + "/cat_fms")
        must_equal(ref, ocv.cat_fms(l, r, max_disp=d), name + "/cat_fms oracle")
        unmasked = rigev.build_concat_volume(l, r, d)
        must_equal(unmasked, ocv.build_concat_volume(l, r, d, mask_left=False), name + "/unmasked")
        save(name, left=l, right=r, maxdisp=d, out=ref, out_unmasked=unmasked)
    l, r = rnd(5, 2, 24, 6, 23), rnd(6, 2, 24, 6, 23)
    ref = rcv.correlation_volume(l, r, 9)
    must_equal(ref, ocv.correlation_volume(l, r, 9), "corr")
    save("corr_small", left=l, right=r, maxdisp=9, out=ref)
    # fused gwc+concat as GwcVolumeCostProcessor.forward returns it
    lg, rg, lc, rc = rnd(7, 1, 32, 4, 40), rnd(8, 1, 32, 4, 40), rnd(9, 1, 3, 4, 40), rnd(10, 1, 3, 4, 40)
    proc = rgw.GwcVolumeCostProcessor(maxdisp=64, downsample=4, num_groups=4, use_concat_volume=True)
    ref = proc({"ref_feature": {"gwc_feature": lg, "concat_feature": lc},
                "tgt_feature": {"gwc_feature": rg, "concat_feature": rc}})["cost_volume"]
    must_equal(ref, ocv.gwc_concat_volume(lg, rg, lc, rc, 16, 4), "fused")
    save("gwc_concat_fused", lg=lg, rg=rg, lc=lc, rc=rc, maxdisp=16, groups=4, out=ref)
    # cat_fms with start_disp / dilation (only the oracle restates these; PSMNet never uses them)
    l, r = rnd(11, 1, 4, 3, 17), rnd(12, 1, 4, 3, 17)
    for tag, kw in [("neg", dict(max_disp=8, start_disp=-3, dilation=1)), ("dil", dict(max_disp=9, start_disp=0, dilation=2))]:
        ref = rpsm.cat_fms(l, r, **kw)
        must_equal(ref, ocv.cat_fms(l, r, **kw), "cat_fms " + tag)
        save("cat_fms_" + tag, left=l, right=r, out=ref, **kw)


def regression():
    rreg = shim.load("stereo.modeling.disp_pred.disp_regression")
    rgdp = shim.load("stereo.modeling.models.gwcnet.gwcnet_disp_processor")
    rpdp = shim.load("stereo.modeling.models.psmnet.psmnet_disp_processor")
    rmet = shim.load("stereo.evaluation.metric_per_image") if os.path.exists(
        os.path.join(shim.REFERENCE_ROOT, "stereo/evaluation/metric_per_image.py")) else None
    import torch.nn.functional as F
    cost = rnd(20, 2, 12, 4, 9, scale=3.0)
    prob = F.softmax(cost, dim=1)
    ref_keep = rreg.disparity_regression(prob, 12)
    ref_flat = rgdp.disparity_regression(prob, 12)
    must_equal(ref_keep, oreg.disparity_regression(prob, 12, keepdim=True), "regression keepdim")
    must_equal(ref_flat, oreg.disparity_regression(prob, 12, keepdim=False), "regression flat")
    must_equal(ref_keep, oreg.softargmin(cost, 12), "softargmin")
    save("softargmin_small", cost=cost, prob=prob, maxdisp=12, out_keepdim=ref_keep, out_flat=ref_flat)
    fsa = rpdp.FasterSoftArgmin(max_disp=16)
    cost = rnd(21, 2, 16, 3, 5, scale=2.0)
    ref = fsa(cost)
    must_equal(ref, oreg.faster_soft_argmin(cost, 16), "faster soft argmin")
    save("faster_softargmin", cost=cost, maxdisp=16, out=ref)
    # fused tails: trilinear x4 -> softmax -> regression
    low = rnd(22, 2, 1, 6, 5, 7, scale=3.0)
    up = F.interpolate(low, [24, 20, 28], mode="trilinear")
    ref_gwc = rgdp.disparity_regression(F.softmax(torch.squeeze(up, 1), dim=1), 24)
    must_equal(ref_gwc, oreg.upsample_softargmin(low, 24, 20, 28, align_corners=False), "gwc tail")
    up = F.interpolate(low, [24, 20, 28], mode="trilinear", align_corners=True)
    ref_psm = rpdp.FasterSoftArgmin(max_disp=24)(torch.squeeze(up, 1))
    must_equal(ref_psm, oreg.upsample_softargmin(low, 24, 20, 28, align_corners=True, psm_tail=True), "psm tail")
    save("upsample_softargmin", cost=low, maxdisp=24, out_h=20, out_w=28, out_gwc=ref_gwc, out_psm=ref_psm)
    if rmet is not None:
        pred, gt = rnd(23, 3, 6, 8).abs() * 40, rnd(24, 3, 6, 8).abs() * 60
        gt[2] = 500.0                                  # an image with no valid pixel
        mask = (gt < 192) & (gt > 0)
        ref = rmet.epe_metric(pred, gt, mask)
        must_equal(ref, oreg.epe_per_image(pred, gt, mask), "epe")
        save("epe_per_image", pred=pred, gt=gt, out=ref)


def modules():
    rgh = shim.load("stereo.modeling.models.gwcnet.hourglass")
    rgdp = shim.load("stereo.modeling.models.gwcnet.gwcnet_disp_processor")
    rpcp = shim.load("stereo.modeling.models.psmnet.psmnet_cost_processor")
    rsbh = shim.load("stereo.modeling.models.stereobase.hourglass")
    with torch.no_grad():
        # GwcNet hourglass, 8 channels
        ref, mine = rgh.Hourglass(8).eval(), oagg.GwcHourglass(8).eval()
        sd = si.seeded_state_dict(ref.state_dict(), seed=31)
        ref.load_state_dict(sd), mine.load_state_dict(sd)
        x = rnd(32, 1, 8, 8, 8, 12)
        y = ref(x)
        must_equal(y, mine(x), "gwc hourglass")
        save("gwc_hourglass_c8", x=x, out=y, seed=31, sd_checksum=checksum(sd))
        # GwcDispProcessor eval branch
        kw = dict(maxdisp=32, downsample=4, num_groups=4, use_concat_volume=True, concat_channels=2)
        ref, mine = rgdp.GwcDispProcessor(**kw).eval(), oagg.GwcDispProcessor(**kw).eval()
        sd = si.seeded_state_dict(ref.state_dict(), seed=33, scale={"classif3.2.weight": 60.0})
        ref.load_state_dict(sd), mine.load_state_dict(sd)
        vol = rnd(34, 1, 8, 8, 8, 16)
        left = torch.zeros(1, 3, 32, 64)
        y = ref({"cost_volume": vol, "left": left})["inference_disp"]["disp_est"]
        must_equal(y, mine(vol, 32, 64), "gwc disp processor")
        save("gwc_disp_processor", volume=vol, out=y, logits=mine.aggregate(vol), seed=33, sd_checksum=checksum(sd))
        # PSMAggregator
        ref, mine = rpcp.PSMAggregator(max_disp=32, in_planes=8).eval(), oagg.PSMAggregator(32, 8).eval()
        sd = si.seeded_state_dict(ref.state_dict(), seed=35,
                                  scale={"classif1.1.weight": 20.0, "classif2.1.weight": 20.0, "classif3.1.weight": 20.0})
        ref.load_state_dict(sd), mine.load_state_dict(sd)
        raw = rnd(36, 1, 8, 8, 8, 16)
        ys, ms = ref(raw), mine(raw)
        for a, b in zip(ys, ms):
            must_equal(a, b, "psm aggregator")
        low = mine.aggregate(raw)
        save("psm_aggregator", raw=raw, cost3_low=low[2], cost2_low=low[1], cost1_low=low[0], seed=35,
             sd_checksum=checksum(sd))
        # StereoBase hourglass + classifier + softargmin
        bc = [16, 16, 24, 20]
        ref = rsbh.Hourglass(8, bc).eval()
        mine = oagg.StereoBaseCostHead(8, bc, max_disp=64).eval()
        sd_h = si.seeded_state_dict(ref.state_dict(), seed=37)
        ref.load_state_dict(sd_h)
        sd = si.seeded_state_dict(mine.state_dict(), seed=38, scale={"classifier.weight": 30.0})
        sd.update({"cost_agg." + k: v for k, v in sd_h.items()})
        mine.load_state_dict(sd)
        vol = rnd(39, 1, 8, 16, 16, 32)
        feats = [rnd(40, 1, 16, 16, 32), rnd(41, 1, 16, 8, 16), rnd(42, 1, 24, 4, 8), rnd(43, 1, 20, 2, 4)]
        geo = ref(vol, feats)
        geo2, init_disp = mine(vol, feats)
        must_equal(geo, geo2, "stereobase hourglass")
        save("stereobase_head", volume=vol, f0=feats[0], f1=feats[1], f2=feats[2], f3=feats[3], geo=geo,
             init_disp=init_disp, seed_hourglass=37, seed_head=38, sd_checksum=checksum(sd))


def models():
    with torch.no_grad():
        cfg = shim.load_cfg("cfgs/gwcnet/gwcnet_sceneflow.yaml").MODEL
        ref = shim.load("stereo.modeling.models.gwcnet.gwcnet").GwcNet(cfg).eval()
        mine = omodels.GwcNet(cfg.MAX_DISP, cfg.USE_CONCAT_VOLUME, cfg.CONCAT_CHANNELS, cfg.DOWNSAMPLE,
                              cfg.NUM_GROUPS).eval()
        assert list(ref.state_dict().keys()) == list(mine.state_dict().keys())
        sd = si.seeded_state_dict(ref.state_dict(), seed=1, scale=si.GWCNET_SCALE)
        ref.load_state_dict(sd), mine.load_state_dict(sd)
        x = {"left": rnd(50, 1, 3, 64, 128), "right": rnd(51, 1, 3, 64, 128)}
        y = ref(dict(x))["disp_pred"]
        must_equal(y, mine(dict(x))["disp_pred"], "GwcNet")
        save("gwcnet_64x128", left=x["left"], right=x["right"], out=y, seed=1, sd_checksum=checksum(sd))

        cfg = shim.load_cfg("cfgs/psmnet/psmnet_sceneflow.yaml").MODEL
        ref = shim.load("stereo.modeling.models.psmnet.psmnet").PSMNet(cfg).eval()
        mine = omodels.PSMNet(cfg.MAX_DISP).eval()
        assert list(ref.state_dict().keys()) == list(mine.state_dict().keys())
        sd = si.seeded_state_dict(ref.state_dict(), seed=1, scale=si.PSMNET_SCALE, keep=si.PSMNET_KEEP)
        ref.load_state_dict(sd), mine.load_state_dict(sd)
        # inputs are rounded to fp16-representable values so they can be stored compactly and exactly
        x = {"left": rnd(52, 1, 3, 256, 256).half().float(), "right": rnd(53, 1, 3, 256, 256).half().float()}
        y = ref(dict(x))
        m = mine(dict(x))
        for a, b in zip(y["train_preds"], m["train_preds"]):
            must_equal(a, b, "PSMNet")
        save("psmnet_256x256", left=x["left"].half(), right=x["right"].half(), out=y["disp_pred"], seed=1,
             sd_checksum=checksum(sd))


def lookups():
    """SURVEY.md section 8(f) rows 1 and 3: geometry-encoding volume lookup and context up-sampling."""
    rgeo = shim.load("stereo.modeling.models.igev.geometry")
    rsb = shim.load("stereo.modeling.models.stereobase.gru_blocks")
    rblk = shim.load("stereo.modeling.models.stereobase.igev_blocks")
    # (name, B, C_feat, C_geo, D, H, W, levels, radius)
    for name, b, cf, cg, d, h, w, levels, radius in (("geo_lookup_small", 2, 6, 8, 12, 3, 10, 2, 4),
                                                     ("geo_lookup_3lvl", 1, 4, 3, 17, 2, 21, 3, 2)):
        f1, f2 = rnd(60, b, cf, h, w), rnd(61, b, cf, h, w)
        vol = rnd(62, b, cg, d, h, w)
        # disparities inside, at the borders of and beyond the volume; two iterations like the GRU loop
        disp = torch.rand(b, 1, h, w, generator=torch.Generator().manual_seed(63)) * (d + 6) - 3
        disp[0, 0, 0, :3] = torch.tensor([0.0, d - 1.0, 2.5])
        coords = torch.arange(w).float().reshape(1, 1, w, 1).repeat(b, h, 1, 1)
        ref = rgeo.Combined_Geo_Encoding_Volume(f1, f2, vol, num_levels=levels, radius=radius)
        ref2 = rsb.CombinedGeoEncodingVolume(f1, f2, vol, num_levels=levels, radius=radius)
        mine = ogeo.GeoEncodingVolume(f1, f2, vol, num_levels=levels, radius=radius)
        out = ref(disp, coords)
        must_equal(out, ref2(disp, coords), name + " igev vs stereobase class")
        must_equal(out, mine(disp, coords), name)
        must_equal(ref.init_corr_pyramid[-1], mine.corr_pyramid[-1], name + " corr pyramid")
        must_equal(ref.geo_volume_pyramid[-1], mine.geo_pyramid[-1], name + " geo pyramid")
        save(name, fmap1=f1, fmap2=f2, volume=vol, disp=disp, coords=coords, levels=levels, radius=radius, out=out,
             geo_last=ref.geo_volume_pyramid[-1], corr_last=ref.init_corr_pyramid[-1])
    low = rnd(64, 2, 1, 5, 7).abs() * 20
    wts = torch.softmax(rnd(65, 2, 9, 20, 28), dim=1)
    ref = rblk.context_upsample(low, wts)
    must_equal(ref, ogeo.context_upsample(low, wts), "context_upsample")
    save("context_upsample", disp_low=low, up_weights=wts, scale=4, out=ref)


def lightstereo():
    """SURVEY.md section 8(f) row 2: LightStereo's 2D aggregation (cfgs/lightstereo: in_channels 48, blocks [4, 8, 14], expanse 4
    in LightStereo-M; a reduced [1, 2, 2] stack with every block kind keeps the fixture small)."""
    ragg = shim.load("stereo.modeling.models.lightstereo.aggregation")
    with torch.no_grad():
        args = dict(in_channels=12, left_att=True, blocks=[1, 2, 2], expanse_ratio=4, backbone_channels=[10, 14, 18])
        ref, mine = ragg.Aggregation(**args).eval(), olight.Aggregation(**args).eval()
        assert list(ref.state_dict().keys()) == list(mine.state_dict().keys())
        sd = si.seeded_state_dict(ref.state_dict(), seed=5)
        ref.load_state_dict(sd), mine.load_state_dict(sd)
        x = rnd(86, 2, 12, 8, 20)
        feats = [rnd(87, 2, 10, 8, 20), rnd(88, 2, 14, 4, 10), rnd(89, 2, 18, 2, 5)]
        y = ref(x, feats)[0]
        must_equal(y, mine(x, feats)[0], "LightStereo aggregation")
        if not y.std() > 1e-3:
            raise SystemExit("degenerate LightStereo fixture (std %g)" % y.std())
        save("lightstereo_aggregation", x=x, f0=feats[0], f1=feats[1], f2=feats[2], out=y, seed=5, sd_checksum=checksum(sd))


def flavours():
    """SURVEY.md section 8(f) row 4: the remaining volume / regression flavours (oracle pinned ahead of the kernels)."""
    import torch.nn.functional as F
    rcv = shim.load("stereo.modeling.cost_volume.cost_volume")
    import types
    for missing in ("trimesh", "imageio", "open3d", "transformations"):     # imported at module level by foundationstereo/Utils.py,
        if missing not in sys.modules:                                      # never dereferenced by the two functions used here
            try:
                __import__(missing)
            except Exception:
                sys.modules[missing] = types.ModuleType(missing)
    rfs = shim.load("stereo.modeling.models.foundationstereo.core.submodule")
    rpp = shim.load("stereo.modeling.models.igevpp.submodule")
    rcas = shim.load("stereo.modeling.models.casnet.submodule")
    l, r = rnd(80, 2, 24, 3, 17), rnd(81, 2, 24, 3, 17)
    ref = rfs.build_gwc_volume(l, r, 9, 4)
    must_equal(ref, ocv.build_gwc_volume_normalized(l, r, 9, 4), "normalised gwc volume")
    save("gwc_normalized", left=l, right=r, maxdisp=9, groups=4, out=ref)
    ref = rcv.CoExCostVolume(6, group=3)(l, r)
    must_equal(ref, ocv.coex_cost_volume(l, r, 6, 3), "CoEx volume")
    save("coex_volume", left=l, right=r, maxdisp=6, group=3, out=ref)
    ls, rs = rnd(82, 1, 5, 2, 6), rnd(83, 1, 5, 2, 6)
    ref = rcv.build_corr_volume(ls, rs, 9)                          # 9 > W = 6: exercises the unshifted else-branch
    must_equal(ref, ocv.build_corr_volume(ls, rs, 9), "corr volume (d >= W quirk)")
    save("corr_volume_quirk", left=ls, right=rs, maxdisp=9, out=ref)
    prob = F.softmax(rnd(84, 2, 12, 3, 5, scale=2.0), dim=1)
    ref = rpp.disparity_regression(prob, 48, 4)
    must_equal(ref, oreg.disparity_regression_interval(prob, 48, 4), "interval regression")
    vals = rnd(85, 2, 12, 3, 5).abs() * 30
    ref2 = rcas.disparity_regression(prob, vals)
    must_equal(ref2, oreg.disparity_regression_values(prob, vals), "explicit-hypothesis regression")
    save("regression_flavours", prob=prob, maxdisp=48, interval=4, out_interval=ref, values=vals, out_values=ref2)


def pinned(out, key, t, full_max=4096, n_sample=2048):
    """Store a reference output under `key`: whole when it has at most `full_max` elements, otherwise a seeded sample of
    `n_sample` elements (flat indices + values) with the shape and the float64 sum and absolute sum of the whole tensor."""
    t = t.detach().contiguous()
    if t.numel() <= full_max:
        out[key] = t
        return
    idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(7))[:n_sample].sort().values
    out[key + "__idx"], out[key + "__val"] = idx.int(), t.reshape(-1)[idx]
    out[key + "__shape"] = torch.tensor(t.shape, dtype=torch.int64)
    out[key + "__sum"], out[key + "__abssum"] = t.double().sum(), t.double().abs().sum()


def pins():
    """The reference outputs that tests/test_oracle_pins_reference.py, tests/test_patch_cpu.py and
    tests/test_ops_gpu.py::test_sub_volume_vs_oracle_and_reference compare against, on the seeded inputs those tests
    regenerate (same seeds, same shapes)."""
    rcv = shim.load("stereo.modeling.cost_volume.cost_volume")
    rpsm = shim.load("stereo.modeling.models.psmnet.psmnet_cost_processor")
    rreg = shim.load("stereo.modeling.disp_pred.disp_regression")
    rpdp = shim.load("stereo.modeling.models.psmnet.psmnet_disp_processor")
    rgh = shim.load("stereo.modeling.models.gwcnet.hourglass")
    rgeo = shim.load("stereo.modeling.models.igev.geometry")
    rsb = shim.load("stereo.modeling.models.stereobase.gru_blocks")
    rblk = shim.load("stereo.modeling.models.stereobase.igev_blocks")
    out = {}
    for b, c, h, w, d, g in [(2, 24, 4, 19, 7, 3), (1, 40, 3, 33, 40, 5), (1, 8, 2, 6, 9, 8)]:
        tag = "%d_%d_%d_%d_%d_%d" % (b, c, h, w, d, g)
        l, r = rnd(1, b, c, h, w), rnd(2, b, c, h, w)
        pinned(out, "gwc_" + tag, rcv.build_gwc_volume(l, r, d, g))
        concat = rcv.build_concat_volume(l, r, d)
        must_equal(concat, rpsm.cat_fms(l, r, max_disp=d), "concat volume vs cat_fms " + tag)     # one array serves both
        pinned(out, "concat_" + tag, concat)
        pinned(out, "corr_" + tag, rcv.correlation_volume(l, r, d))
    p = torch.softmax(rnd(3, 2, 20, 5, 6) * 3, 1)
    out["regression"] = rreg.disparity_regression(p, 20)
    out["faster_softargmin"] = rpdp.FasterSoftArgmin(max_disp=20, alpha=2.0)(rnd(4, 2, 20, 5, 6))
    with torch.no_grad():
        ref = rgh.Hourglass(8).eval()
        ref.load_state_dict(si.seeded_state_dict(ref.state_dict(), seed=5))
        x = rnd(6, 1, 8, 4, 8, 8)
        out["gwc_hourglass"] = ref(x)
        ref = rpsm.Hourglass(8).eval()
        ref.load_state_dict(si.seeded_state_dict(ref.state_dict(), seed=7))
        for i, t in enumerate(ref(x, rnd(8, 1, 16, 2, 4, 4), rnd(9, 1, 16, 2, 4, 4))):
            out["psm_hourglass_%d" % i] = t
    for b, cf, cg, d, h, w, levels, radius in [(1, 5, 8, 24, 4, 30, 2, 4), (2, 3, 2, 9, 2, 11, 1, 3)]:
        f1, f2, vol = rnd(70, b, cf, h, w), rnd(71, b, cf, h, w), rnd(72, b, cg, d, h, w)
        disp = torch.rand(b, 1, h, w, generator=torch.Generator().manual_seed(73)) * (d + 4) - 2
        coords = torch.arange(w).float().reshape(1, 1, w, 1).repeat(b, h, 1, 1)
        a = rgeo.Combined_Geo_Encoding_Volume(f1, f2, vol, num_levels=levels, radius=radius)(disp, coords)
        must_equal(a, rsb.CombinedGeoEncodingVolume(f1, f2, vol, num_levels=levels, radius=radius)(disp, coords),
                   "geo lookup: igev vs stereobase class")
        pinned(out, "geo_%d_%d_%d_%d_%d_%d_%d_%d" % (b, cf, cg, d, h, w, levels, radius), a)
    low, wts = rnd(74, 2, 1, 6, 9).abs() * 30, torch.softmax(rnd(75, 2, 9, 24, 36), dim=1)
    out["context_upsample"] = rblk.context_upsample(low, wts)
    save("pins_reference", **out)

    # build_sub_volume allocates its output with device='cuda'; its arithmetic (an L1 norm over channels) is run here on
    # the host by allocating that output on the inputs' device instead
    zeros = torch.zeros
    rcv.torch.zeros = lambda *a, device=None, **k: zeros(*a, **k)
    try:
        sub = {}
        for shape, d in (((2, 12, 5, 37), 9), ((1, 96, 4, 128), 48), ((1, 3, 2, 6), 8)):
            pinned(sub, "sub_%s_%d" % ("_".join(map(str, shape)), d), rcv.build_sub_volume(rnd(70, *shape), rnd(71, *shape), d))
    finally:
        rcv.torch.zeros = zeros
    save("sub_volume_reference", **sub)

    # the module globals StereoBase's forward and upsample_disp reach by name: what per-instance rebinding has to override
    sbm = shim.load("stereo.modeling.models.stereobase.stereobase_gru")
    names = (set(sbm.StereoBase.forward.__code__.co_names) | set(sbm.StereoBase.upsample_disp.__code__.co_names)) & set(vars(sbm))
    save("stereobase_globals", names=np.array(sorted(names)))


GROUPS = {"volumes": volumes, "regression": regression, "modules": modules, "models": models, "lookups": lookups,
          "flavours": flavours, "lightstereo": lightstereo, "pins": pins}


if __name__ == "__main__":
    if not shim.available():
        raise SystemExit("reference tree not found; golden vectors can only be generated where it is present")
    torch.set_num_threads(os.cpu_count() or 1)
    for name in sys.argv[1:] or GROUPS:
        GROUPS[name]()
    print("all oracle restatements bit-equal to the reference; golden vectors written to", OUT)
