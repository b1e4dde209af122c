"""patch(model): make an UNMODIFIED OpenStereo model instance (GwcNet / PSMNet / StereoBase / LightStereo / IGEVStereo, built by the
reference's own classes from an unchanged cfg YAML) run its cost-volume hot path on the sm_100a kernels.

The reference has no operator registry; names are bound three different ways (SURVEY.md section 8b), and each
needs its own rebinding:

* GwcNet      bound methods on ``CostProcessor`` (gwcnet_cost_processor.py:58-64) and the ``DispProcessor``
              forward (gwcnet_disp_processor.py:83-140)                    -> per-instance ``forward`` override
* PSMNet      ``cat_fms`` captured by functools.partial at construction (psmnet_cost_processor.py:227-232),
              aggregator + FasterSoftArgmin modules                          -> ``CostProcessor.forward`` / ``FasterSoftArgmin.forward``
* LightStereo / IGEVStereo  like StereoBase: names imported into lightstereo.py:4-6 / igev_stereo.py:1-3 (``from .submodule import *``)
* StereoBase  functions imported INTO the module namespace (stereobase_gru.py:5-6,10-11) and the ``cost_agg``
              Hourglass                                                      -> per-INSTANCE copies of the methods that use those names,
                                                                                with a private globals dict (the module itself, and
                                                                                therefore every other StereoBase instance, is untouched)

Parameters stay where they are (the engines read them through the reference's attribute names), so
``state_dict()`` / ``load_state_dict()`` and checkpoints are untouched.

When is a call accelerated?  Only when it is a CUDA inference call: every tensor on a CUDA device, the module in eval
mode, and autograd not recording (``torch.no_grad()`` as in trainer_template.py:260-283, or no operand requires grad).
The kernels have no backward, so anything else must NOT reach them silently:
  strict=True  (default) such a call RAISES -- there is no CPU / autograd path in this package;
  strict=False           such a call runs the reference's own original Python code, gradients intact (tools/train.py).
"""
import types

import torch

from . import ops
from .aggregation import GwcAggregation, PSMAggregation, StereoBaseAggregation
from .geo import CombinedGeoEncodingVolume


def _tensors(args):
    for a in args:
        if isinstance(a, torch.Tensor):
            yield a
        elif isinstance(a, (list, tuple)):
            yield from _tensors(a)
        elif isinstance(a, dict):
            yield from _tensors(a.values())


def _recording(*args):
    """True when autograd would record an op on these operands (the kernels would silently cut the graph)."""
    return torch.is_grad_enabled() and any(t.requires_grad for t in _tensors(args))


def _accelerable(module, *args):
    ts = list(_tensors(args))
    return (module is None or not module.training) and bool(ts) and all(t.is_cuda for t in ts) and not _recording(*ts)


def _refuse(what):
    raise RuntimeError("openstereo_b200: %s is patched for CUDA inference only (model.eval() on a CUDA device, under "
                       "torch.no_grad() or with no operand requiring grad); use patch(model, strict=False) to delegate "
                       "training / CPU calls to the reference implementation" % what)


def _patch_backbone(bb, net, extract, split):
    """2D feature extractor (gwcnet_backbone.py:96-107 / psmnet_backbone.py:118-126; not a SURVEY section-8 row, but inside the
    measured forward): CUDA inference calls run a BN-folded twin of `net` whose identity-shortcut 3x3 residual blocks use the
    tcgen05 conv kernels where a variant serves the shape (host_models.gwc_extract / psm_extract; every other layer is the
    module's own cuDNN conv), left and right images in ONE batched pass (the weights are shared).  Parameters stay in `net`;
    the twin is rebuilt when they change.  Any other call (CPU, training, autograd recording) runs the reference's forward."""
    from . import host_models
    rt = host_models._FoldedRuntime(net)
    orig = bb.forward

    def forward(self, inputs):
        left, right = inputs["left"], inputs["right"]
        trainable = torch.is_grad_enabled() and any(q.requires_grad for q in net.parameters())   # the folded twin would cut them off
        if trainable or not (_accelerable(self, left, right) and left.dtype == torch.float32 and left.shape == right.shape):
            return orig(inputs)
        both = extract(rt.get(), torch.cat((left, right), 0))
        return split(both, left.shape[0])

    bb.forward = types.MethodType(forward, bb)


def _split_dict(both, b):
    return {"ref_feature": {k: v[:b] for k, v in both.items()}, "tgt_feature": {k: v[b:] for k, v in both.items()}}


def _split_tensor(both, b):
    return {"ref_feature": both[:b], "tgt_feature": both[b:]}


def _patch_gwcnet(model, strict, backbone=True):
    if backbone:
        from .host_models import gwc_extract
        _patch_backbone(model.Backbone, model.Backbone.feature_extraction, gwc_extract, _split_dict)
    cp, dp = model.CostProcessor, model.DispProcessor
    cp_orig, dp_orig = cp.forward, dp.forward                                 # the reference's bound methods
    gwc_orig, cat_orig = cp.build_gwc_volume, cp.build_concat_volume
    engine = GwcAggregation(dp)

    def cost_forward(self, inputs):
        lf, rf = inputs["ref_feature"], inputs["tgt_feature"]
        if not _accelerable(self, lf, rf):
            if strict:
                _refuse("GwcVolumeCostProcessor")
            saved = self.build_gwc_volume, self.build_concat_volume            # the reference's forward calls these two
            self.build_gwc_volume, self.build_concat_volume = gwc_orig, cat_orig
            try:
                return cp_orig(inputs)
            finally:
                self.build_gwc_volume, self.build_concat_volume = saved
        d = self.maxdisp // self.downsample
        if self.use_concat_volume:
            vol = ops.gwc_concat_volume(lf["gwc_feature"], rf["gwc_feature"], lf["concat_feature"],
                                        rf["concat_feature"], d, self.num_groups)
        else:
            vol = ops.build_gwc_volume(lf["gwc_feature"], rf["gwc_feature"], d, self.num_groups)
        return {"cost_volume": vol}

    def disp_forward(self, inputs):
        if not _accelerable(self, inputs["cost_volume"]):
            return dp_orig(inputs) if not strict else _refuse("GwcDispProcessor")
        h, w = inputs["left"].shape[2:]
        return {"inference_disp": {"disp_est": engine(inputs["cost_volume"], h, w)}}

    cp.forward = types.MethodType(cost_forward, cp)
    dp.forward = types.MethodType(disp_forward, dp)

    # the two volume builders stay callable on their own, with the reference's method signatures
    def build_gwc(ref, tgt):
        if _accelerable(None, ref, tgt):
            return ops.build_gwc_volume(ref, tgt, cp.maxdisp // cp.downsample, cp.num_groups)
        return gwc_orig(ref, tgt) if not strict else _refuse("build_gwc_volume")

    def build_concat(ref, tgt):
        if _accelerable(None, ref, tgt):
            return ops.build_concat_volume(ref, tgt, cp.maxdisp // cp.downsample)
        return cat_orig(ref, tgt) if not strict else _refuse("build_concat_volume")

    cp.build_gwc_volume, cp.build_concat_volume = build_gwc, build_concat
    return model


class FusedCost:
    """What the patched PSMCostProcessor hands to PSMDispProcessor in place of a (B, 192, H, W) cost tensor: the fused tail
    (trilinear x4 + softmax + expectation in one kernel) already produced the disparity and the full-resolution cost is never
    materialised.  The patched FasterSoftArgmin recognises it; any other consumer gets a loud AttributeError/TypeError
    instead of a silently wrong tensor."""
    __slots__ = ("disp",)

    def __init__(self, disp):
        self.disp = disp


def _patch_psmnet(model, strict, backbone=True):
    if backbone:
        from .host_models import psm_extract
        _patch_backbone(model.Backbone, model.Backbone, psm_extract, _split_tensor)
    cp, dp = model.CostProcessor, model.DispProcessor
    cp_orig = cp.forward
    engine = PSMAggregation(cp.aggregator)
    max_disp = cp.aggregator.max_disp
    cat_orig = cp.cat_func                                          # functools.partial(cat_fms, ...) of the reference

    def cost_forward(self, inputs):
        lf, rf = inputs["ref_feature"], inputs["tgt_feature"]
        if not _accelerable(self, lf, rf):
            if strict:
                _refuse("PSMCostProcessor")
            saved, self.cat_func = self.cat_func, cat_orig
            try:
                return cp_orig(inputs)
            finally:
                self.cat_func = saved
        raw = ops.cat_fms(lf, rf, max_disp=int(max_disp // 4), start_disp=0, dilation=1)
        d1, d2, d3 = engine(raw)
        return {"cost1": FusedCost(d1), "cost2": FusedCost(d2), "cost3": FusedCost(d3)}

    cp.forward = types.MethodType(cost_forward, cp)

    def cat_func(l, r):
        if _accelerable(None, l, r):
            return ops.cat_fms(l, r, max_disp=int(max_disp // 4), start_disp=0, dilation=1)
        return cat_orig(l, r) if not strict else _refuse("cat_fms")

    cp.cat_func = cat_func
    sa = dp.disp_processor                                          # FasterSoftArgmin: keep the frozen Conv3d parameter
    sa_orig = sa.forward

    def sa_forward(self, cost):
        if isinstance(cost, FusedCost):
            return cost.disp
        if _accelerable(None, cost):
            return ops.faster_soft_argmin(cost, self.max_disp, self.start_disp, self.dilation, self.alpha, self.normalize)
        return sa_orig(cost) if not strict else _refuse("FasterSoftArgmin")

    sa.forward = types.MethodType(sa_forward, sa)
    return model


def _rebind_methods(model, overrides):
    """Give `model` private copies of the methods of its class that use any name in `overrides` as a module global: same code
    object, closure and defaults, but a globals dict with the overrides applied.  The module namespace and the class are not
    modified, so other instances (patched or not) are unaffected."""
    for name, fn in vars(type(model)).items():
        if isinstance(fn, types.FunctionType) and set(fn.__code__.co_names) & set(overrides):
            g = dict(fn.__globals__)
            g.update(overrides)
            copy = types.FunctionType(fn.__code__, g, fn.__name__, fn.__defaults__, fn.__closure__)
            copy.__kwdefaults__ = fn.__kwdefaults__
            setattr(model, name, types.MethodType(copy, model))


def _patch_stereobase(model, strict, backbone=True, precision="fp32"):
    g = type(model).forward.__globals__                             # stereo.modeling.models.stereobase.stereobase_gru namespace
    hg = model.cost_agg
    hg_orig = hg.forward
    agg = StereoBaseAggregation(hg, precision=precision)
    orig = {n: g[n] for n in ("build_gwc_volume", "build_concat_volume", "disparity_regression", "CombinedGeoEncodingVolume",
                              "context_upsample")}

    def gwc(ref, tgt, maxdisp, groups):
        if _accelerable(model, ref, tgt):
            return ops.build_gwc_volume(ref, tgt, maxdisp, groups)
        return orig["build_gwc_volume"](ref, tgt, maxdisp, groups) if not strict else _refuse("build_gwc_volume")

    def concat(ref, tgt, maxdisp):
        if _accelerable(model, ref, tgt):
            return ops.build_concat_volume(ref, tgt, maxdisp)
        return orig["build_concat_volume"](ref, tgt, maxdisp) if not strict else _refuse("build_concat_volume")

    def regression(x, maxdisp):
        if _accelerable(model, x):
            return ops.disparity_regression(x, maxdisp)
        return orig["disparity_regression"](x, maxdisp) if not strict else _refuse("disparity_regression")

    # SURVEY.md section 8(f) rows 1 and 3: the per-GRU-iteration lookup and the convex up-sampling (stereobase_gru.py:172-209)
    def geo_factory(fmap1, fmap2, volume, num_levels=2, radius=4):
        fast = _accelerable(model, fmap1, fmap2, volume)
        if not fast and strict:
            _refuse("CombinedGeoEncodingVolume")
        cls = CombinedGeoEncodingVolume if fast else orig["CombinedGeoEncodingVolume"]
        return cls(fmap1, fmap2, volume, num_levels=num_levels, radius=radius)

    def upsample(disp_low, up_weights, scale_factor=4):
        if _accelerable(model, disp_low, up_weights):
            return ops.context_upsample(disp_low, up_weights, scale_factor).to(disp_low.dtype)
        return orig["context_upsample"](disp_low, up_weights, scale_factor) if not strict else _refuse("context_upsample")

    _rebind_methods(model, {"build_gwc_volume": gwc, "build_concat_volume": concat, "disparity_regression": regression,
                            "CombinedGeoEncodingVolume": geo_factory, "context_upsample": upsample})

    def hg_forward(self, x, features, return_multi=False):
        if return_multi or not _accelerable(self, x, features):
            return hg_orig(x, features, return_multi) if not strict else _refuse("StereoBase Hourglass")
        return agg(x, features).to(x.dtype)

    hg.forward = types.MethodType(hg_forward, hg)
    return model


def _volume_tail_overrides(model, strict, orig, with_corr):
    """Guarded replacements of the module-global hot-path functions LightStereo / IGEV import into their model module."""
    out = {}
    if with_corr:
        def corr(left, right, max_disp):
            if _accelerable(model, left, right):
                return ops.correlation_volume(left, right, max_disp)
            return orig["correlation_volume"](left, right, max_disp) if not strict else _refuse("correlation_volume")
        out["correlation_volume"] = corr
    else:
        def gwc(ref, tgt, maxdisp, groups):
            if _accelerable(model, ref, tgt):
                return ops.build_gwc_volume(ref, tgt, maxdisp, groups)
            return orig["build_gwc_volume"](ref, tgt, maxdisp, groups) if not strict else _refuse("build_gwc_volume")
        out["build_gwc_volume"] = gwc

    def regression(x, maxdisp):
        if _accelerable(model, x):
            return ops.disparity_regression(x, maxdisp)
        return orig["disparity_regression"](x, maxdisp) if not strict else _refuse("disparity_regression")

    def upsample(disp_low, up_weights, scale_factor=4):
        if scale_factor == 4 and _accelerable(model, disp_low, up_weights):
            return ops.context_upsample(disp_low, up_weights, 4).to(disp_low.dtype)
        if strict:
            _refuse("context_upsample")
        return orig["context_upsample"](disp_low, up_weights) if scale_factor == 4 else orig["context_upsample"](disp_low, up_weights, scale_factor)

    out["disparity_regression"], out["context_upsample"] = regression, upsample
    return out


def _patch_lightstereo(model, strict, backbone=True):
    """LightStereo (BASELINE config 4; lightstereo/lightstereo.py:44-70): correlation_volume, the 2D `Aggregation` hourglass
    (cost_agg), disparity_regression and context_upsample; backbone / refine heads stay the reference's cuDNN code."""
    from .aggregation import LightStereoAggregation
    g = type(model).forward.__globals__
    orig = {n: g[n] for n in ("correlation_volume", "disparity_regression", "context_upsample")}
    _rebind_methods(model, _volume_tail_overrides(model, strict, orig, with_corr=True))
    agg_mod = model.cost_agg
    agg_orig = agg_mod.forward
    engine = LightStereoAggregation(agg_mod)

    def agg_forward(self, x, features_left):
        if not _accelerable(self, x, features_left[:3]):
            return agg_orig(x, features_left) if not strict else _refuse("LightStereo Aggregation")
        return [t.to(x.dtype) for t in engine(x, features_left[:3])]

    agg_mod.forward = types.MethodType(agg_forward, agg_mod)
    return model


def _patch_igev(model, strict, backbone=True):
    """IGEV-Stereo (BASELINE config 5; igev/igev_stereo.py:136-213): the gwc volume, the soft-argmin regression of the initial
    disparity, the per-GRU-iteration lookup of the combined geometry-encoding volume and the convex up-sampling.  The hourglass(8),
    feature nets and ConvGRU update blocks stay the reference's cuDNN code."""
    g = type(model).forward.__globals__
    orig = {n: g[n] for n in ("build_gwc_volume", "disparity_regression", "context_upsample", "Combined_Geo_Encoding_Volume")}
    over = _volume_tail_overrides(model, strict, orig, with_corr=False)

    def geo_factory(fmap1, fmap2, volume, num_levels=2, radius=4):
        fast = _accelerable(model, fmap1, fmap2, volume)
        if not fast and strict:
            _refuse("Combined_Geo_Encoding_Volume")
        cls = CombinedGeoEncodingVolume if fast else orig["Combined_Geo_Encoding_Volume"]
        return cls(fmap1, fmap2, volume, num_levels=num_levels, radius=radius)

    over["Combined_Geo_Encoding_Volume"] = geo_factory
    _rebind_methods(model, over)
    return model


_PATCHERS = {"GwcNet": _patch_gwcnet, "PSMNet": _patch_psmnet, "StereoBase": _patch_stereobase, "LightStereo": _patch_lightstereo,
             "IGEVStereo": _patch_igev}


def patch(model, strict=True, backbone=True, precision="fp32"):
    """Rebind the hot path of a reference model instance in place and return it.  backbone=True (default) also routes the
    GwcNet / PSMNet 2D extractor's residual blocks to the tcgen05 conv kernels in CUDA inference calls (_patch_backbone);
    backbone=False leaves the extractor entirely to the reference's cuDNN code.

    precision="fp32" (default): every accelerated op computes fp32-accurate results, also under torch.autocast (fp16 / bf16
    tensors are up-converted and the results cast back).  precision="fp16" (StereoBase only): under torch.autocast(float16) the
    cost-aggregation hourglass runs with fp16 activations and one fp16 tensor-core product per multiply-add (fp32 accumulation,
    BN / activation / FeatureAtt gate in fp32) and returns fp16 -- an accuracy choice like allow_tf32, not a free speed-up.  Its
    envelope is fp16's: intermediate values are stored as fp16, so |values| above 65504 saturate; when that happens the next
    forward raises RuntimeError (the saturated result was already returned).  Volumes, classifier head and regression keep fp32
    arithmetic; fp32 and bf16 inputs and shapes without the fp16 kernels take the fp32 path (INTEGRATION.md section 1)."""
    if not isinstance(model, torch.nn.Module):
        raise TypeError("patch() expects an nn.Module")
    if precision not in ("fp32", "fp16"):
        raise ValueError("precision must be 'fp32' or 'fp16', got %r" % (precision,))
    name = type(model).__name__
    if precision == "fp16" and name != "StereoBase":
        raise ValueError("precision='fp16' is implemented for StereoBase only")
    if name not in _PATCHERS:
        raise NotImplementedError("patch(): no hot-path drop-in for %s (supported: %s)" % (name, sorted(_PATCHERS)))
    if getattr(model, "_osb_patched", False):
        return model
    if precision == "fp16":
        _PATCHERS[name](model, strict, backbone, precision=precision)
    else:
        _PATCHERS[name](model, strict, backbone)
    model._osb_patched = True
    return model
