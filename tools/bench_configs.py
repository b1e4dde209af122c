#!/usr/bin/env python
"""Hot-path timings at the OTHER BASELINE.json configurations (bench.py is the contract line for configs[1], GwcNet):

    python tools/bench_configs.py [--only c1,c3,c3h,c4,c5] [--iters 10]

  c1  PSMNet cfgs/psmnet, 1 pair 256x512 D=192: whole-model forward of the host mirror (pairs/s) + EPE vs the CPU oracle
  c3  StereoBase cfgs/stereobase, 4 pairs/GPU (batch 32 over 8 GPUs) @256x512: the hot sub-graph on synthetic features --
      gwc (C=96, G=8) + concat (C=8) volume -> Hourglass(24, [96,64,192,160]) with FeatureAtt gates -> classifier -> softmax ->
      regression (stereobase_gru.py:139-164)
  c3h the c3 sub-graph under torch.autocast("cuda", torch.float16), as StereoBase's own AMP configs evaluate it
      (stereobase_sceneflow.yaml AMP: true): three arms alternated in one process -- (a) the oracle modules on cuDNN fp16 (the
      reference's AMP behaviour), (b) this library with precision="fp32" (fp32-accurate hourglass), (c) precision="fp16" (fp16
      hourglass) -- with per-kernel times of (b) and (c) and the init-disparity EPE of (a) and (c) against (b)
  c4  LightStereo-S cfgs/lightstereo, batch 16 @320x736: correlation_volume (C=24... the 1/4 features) -> Aggregation(48, [1,2,4],
      expanse 4, left attention) -> softmax/regression -> context_upsample (lightstereo.py:51-62)
  c5  IGEV cfgs/igev, batch 8 @480x640: gwc volume (C=96, G=8, D'=48) + 16 GRU-iteration lookups of the combined geometry
      encoding volume (igev_stereo.py:158,181-193; geometry.py:32-57) + 16 context up-samplings
Each line: this library (CUDA events, L2 flushed between iterations by the working set itself: every config streams > 126 MB per
step) next to the SAME graph of the oracle modules (bit-equal restatements of the reference: identical aten calls) on this GPU with
cuDNN fp32 (TF32 off) -- SURVEY.md section 8d's GPU comparator -- and the max abs / EPE difference between the two.
Test / measurement infrastructure: imports oracle/ as the checker and comparator."""
import argparse
import json
import os
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import __graft_entry__                                  # noqa: E402
__graft_entry__.build()
from openstereo_b200 import aggregation as agg          # noqa: E402
from openstereo_b200 import geo, host_models, ops       # noqa: E402
from oracle import aggregation as oagg                  # noqa: E402
from oracle import cost_volume as ocv                   # noqa: E402
from oracle import geo_lookup as ogeo                   # noqa: E402
from oracle import lightstereo as olight                # noqa: E402
from oracle import models as omodels                    # noqa: E402
from oracle import regression as oreg                   # noqa: E402
from oracle import seeded_init as si                    # noqa: E402

torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False
# under torchrun (python -m torch.distributed.run --nproc-per-node N tools/bench_configs.py --only c3): one process per GPU, every
# rank times the same per-GPU workload (weak scaling: BASELINE config 3 is batch 32 over 8 GPUs = 4 pairs per GPU), the step time is
# the max over ranks, rank 0 prints the aggregate
WORLD = int(os.environ.get("WORLD_SIZE", "1"))
RANK = int(os.environ.get("RANK", "0"))
DEV = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
torch.cuda.set_device(DEV)
if WORLD > 1:
    import torch.distributed as dist
    dist.init_process_group("nccl", device_id=DEV)


def over_ranks(ms):
    """max over ranks of a per-rank time (ms)"""
    if WORLD == 1:
        return ms
    t = torch.tensor([ms], device=DEV, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def timeit(fn, iters, warm=3):
    for _ in range(warm):
        out = fn()
    torch.cuda.synchronize()
    if WORLD > 1:
        dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters, out


NO_REF = bool(os.environ.get("OSB_NO_REF"))         # launch lists under ncu: skip the cuDNN comparator


def rnd(gen, *shape, scale=1.0):
    return (torch.randn(*shape, generator=gen) * scale).to(DEV)


def emit(**kw):
    if RANK == 0:
        print(json.dumps(kw), flush=True)


def c1(iters):
    oracle = omodels.PSMNet(192).eval()
    sd = si.seeded_state_dict(oracle.state_dict(), seed=1, scale=si.PSMNET_SCALE, keep=si.PSMNET_KEEP)
    oracle.load_state_dict(sd)
    mine = host_models.PSMNet({"MAX_DISP": 192}).eval()
    mine.load_state_dict(sd)
    mine.to(DEV)
    g = torch.Generator().manual_seed(7)
    x = {"left": torch.randn(1, 3, 256, 512, generator=g), "right": torch.randn(1, 3, 256, 512, generator=g)}
    xg = {k: v.to(DEV) for k, v in x.items()}
    with torch.no_grad():
        want = oracle(dict(x))["disp_pred"]
        ms, got = timeit(lambda: mine(dict(xg))["disp_pred"], iters)
        oracle.to(DEV)
        ms_ref, ref_gpu = timeit(lambda: oracle(dict(xg))["disp_pred"], max(2, iters // 3), warm=1)
    emit(config="c1 PSMNet 1 pair 256x512 D=192", ms_per_step=round(ms, 3), pairs_per_s=round(1e3 / ms, 2),
         reference_cudnn_fp32_ms=round(ms_ref, 2), speedup_vs_reference_gpu=round(ms_ref / ms, 2),
         epe_vs_cpu_oracle_px=float("%.3e" % (got.cpu() - want).abs().mean().item()), overflow_count=ops.tc_overflow_count())


def c3(iters, B=4):
    gen = torch.Generator().manual_seed(7)
    ml, mr, cl, cr = rnd(gen, B, 96, 64, 128), rnd(gen, B, 96, 64, 128), rnd(gen, B, 8, 64, 128), rnd(gen, B, 8, 64, 128)
    feats = [rnd(gen, B, 96, 64, 128), rnd(gen, B, 64, 32, 64), rnd(gen, B, 192, 16, 32), rnd(gen, B, 160, 8, 16)]
    m = oagg.StereoBaseCostHead(24, [96, 64, 192, 160], max_disp=192).eval()
    m.load_state_dict(si.seeded_state_dict(m.state_dict(), seed=9, scale={"classifier.weight": 150.0}))
    m.to(DEV)
    hg, head = agg.StereoBaseAggregation(m.cost_agg), agg.StereoBaseCostHead(m.classifier)

    def ours():
        vol = ops.gwc_concat_volume(ml, mr, cl, cr, 48, 8)
        return head(hg(vol, feats), 48)

    def ref():
        vol = torch.cat((ocv.build_gwc_volume(ml, mr, 48, 8), ocv.build_concat_volume(cl, cr, 48)), 1)
        return m(vol, feats)[1]

    with torch.no_grad():
        ms, got = timeit(ours, iters, warm=1 if NO_REF else 3)
        ms = over_ranks(ms)
        ms_ref, want = (float("nan"), got) if NO_REF else timeit(ref, max(2, iters // 3), warm=1)
    emit(config="c3 StereoBase hot sub-graph, B=%d/GPU @256x512 (volume -> Hourglass(24)+FeatureAtt -> classifier -> soft-argmin)" % B,
         n_gpus=WORLD, ms_per_step=round(ms, 3), pairs_per_s=round(WORLD * B * 1e3 / ms, 2), reference_cudnn_fp32_ms=round(ms_ref, 2),
         speedup_vs_reference_gpu=round(ms_ref / ms, 2), init_disp_epe_vs_reference_gpu_px=float("%.3e" % (got - want).abs().mean().item()),
         gmac_per_pair=23.48)


def gpu_identity():
    """(name, power limit) of the GPU these numbers were measured on, read in the same process."""
    import subprocess
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(DEV.index), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        q = "unavailable (%s)" % exc
    return torch.cuda.get_device_name(DEV), q


def c3h(iters, B=4, rounds=5):
    gen = torch.Generator().manual_seed(7)
    ml, mr, cl, cr = (rnd(gen, B, 96, 64, 128).half(), rnd(gen, B, 96, 64, 128).half(), rnd(gen, B, 8, 64, 128).half(),
                      rnd(gen, B, 8, 64, 128).half())
    feats = [rnd(gen, B, 96, 64, 128).half(), rnd(gen, B, 64, 32, 64).half(), rnd(gen, B, 192, 16, 32).half(),
             rnd(gen, B, 160, 8, 16).half()]
    m = oagg.StereoBaseCostHead(24, [96, 64, 192, 160], max_disp=192).eval()
    m.load_state_dict(si.seeded_state_dict(m.state_dict(), seed=9, scale={"classifier.weight": 150.0}))
    m.to(DEV)
    head = agg.StereoBaseCostHead(m.classifier)
    engines = {"fp32": agg.StereoBaseAggregation(m.cost_agg), "fp16": agg.StereoBaseAggregation(m.cost_agg, precision="fp16")}

    def ours(precision):
        def step():   # patch.py's StereoBase route: fp16 volume in, the hourglass result cast back to the volume's dtype
            vol = ops.gwc_concat_volume(ml, mr, cl, cr, 48, 8)
            return head(engines[precision](vol, feats).to(vol.dtype), 48)
        return step

    def ref():
        vol = torch.cat((ocv.build_gwc_volume(ml, mr, 48, 8), ocv.build_concat_volume(cl, cr, 48)), 1)
        return m(vol, feats)[1]

    arms = {"a_reference_cudnn_fp16": ref, "b_ours_fp32": ours("fp32"), "c_ours_fp16": ours("fp16")}
    times = {k: [] for k in arms}
    outs = {}
    with torch.no_grad(), torch.autocast("cuda", torch.float16):
        for k, fn in arms.items():                                          # warm every arm (module loads, cuDNN algorithm choice)
            outs[k] = fn().float()
        for _ in range(rounds):                                             # alternate the arms: drift of the shared host hits all
            for k, fn in arms.items():
                ms, _ = timeit(fn, iters, warm=1)
                times[k].append(ms)
        kernels = {}
        for k in ("b_ours_fp32", "c_ours_fp16"):                            # per entry point, CUDA events (separate from the timing)
            arms[k]()
            torch.cuda.synchronize()
            ops.profile_start()
            for _ in range(iters):
                arms[k]()
            prof = ops.profile_stop()
            torch.cuda.synchronize()
            kernels[k] = {n: round(sum(a.elapsed_time(b) for a, b in ev) / iters, 4) for n, ev in sorted(prof.items())}
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    name, power = gpu_identity()
    base = outs["b_ours_fp32"]
    emit(config="c3h StereoBase hot sub-graph under autocast(fp16), B=%d @256x512" % B, gpu=name, power_limit_and_max_sm_clock=power,
         iters_per_round=iters, rounds=rounds, ms_per_step_median={k: round(v, 3) for k, v in med.items()},
         ms_per_step_all={k: [round(x, 3) for x in v] for k, v in times.items()},
         speedup_c_vs_b=round(med["b_ours_fp32"] / med["c_ours_fp16"], 3),
         speedup_c_vs_a=round(med["a_reference_cudnn_fp16"] / med["c_ours_fp16"], 3),
         init_disp_epe_vs_b_px={"a_reference_cudnn_fp16": float("%.3e" % (outs["a_reference_cudnn_fp16"] - base).abs().mean().item()),
                                "c_ours_fp16": float("%.3e" % (outs["c_ours_fp16"] - base).abs().mean().item())},
         per_entry_point_ms_per_step=kernels, overflow_count=ops.tc_overflow_count())


def c4(iters, B=16):
    gen = torch.Generator().manual_seed(11)
    h, w = 80, 184
    fl, fr = rnd(gen, B, 24, h, w), rnd(gen, B, 24, h, w)
    feats = [fl, rnd(gen, B, 32, h // 2, w // 2), rnd(gen, B, 96, h // 4, w // 4)]
    spx = torch.softmax(rnd(gen, B, 9, 4 * h, 4 * w), 1)
    m = olight.Aggregation(in_channels=48, left_att=True, blocks=[1, 2, 4], expanse_ratio=4, backbone_channels=[24, 32, 96]).eval()
    m.load_state_dict(si.seeded_state_dict(m.state_dict(), seed=6))
    m.to(DEV)
    eng = agg.LightStereoAggregation(m)

    def ours():
        vol = ops.correlation_volume(fl, fr, 48)
        enc = eng(vol, feats)[0]
        init = ops.softargmin(enc, 48, keepdim=True)
        return ops.context_upsample(init * 4.0, spx, 4)

    def ref():
        vol = ocv.correlation_volume(fl, fr, 48)
        enc = m(vol, feats)[0]
        init = oreg.disparity_regression(F.softmax(enc, 1), 48)
        return ogeo.context_upsample(init * 4.0, spx)

    with torch.no_grad():
        ms, got = timeit(ours, iters)
        ms_ref, want = timeit(ref, max(2, iters // 3), warm=1)
    emit(config="c4 LightStereo-S hot path, B=%d @320x736 (corr volume -> 2D aggregation -> soft-argmin -> context_upsample)" % B,
         ms_per_step=round(ms, 3), pairs_per_s=round(B * 1e3 / ms, 2), reference_cudnn_fp32_ms=round(ms_ref, 2),
         speedup_vs_reference_gpu=round(ms_ref / ms, 2), disp_epe_vs_reference_gpu_px=float("%.3e" % (got - want.reshape(got.shape)).abs().mean().item()),
         disparity_std_px=round(want.std().item(), 2))


def c5(iters, B=8, gru_iters=16):
    gen = torch.Generator().manual_seed(13)
    h, w, d = 120, 160, 48
    ml, mr = rnd(gen, B, 96, h, w), rnd(gen, B, 96, h, w)
    f1, f2 = rnd(gen, B, 96, h, w), rnd(gen, B, 96, h, w)
    cv = rnd(gen, B, 8, d, h, w)                                              # stands in for the hourglass(8) output
    disp = (torch.rand(B, 1, h, w, generator=gen) * (d - 1)).to(DEV)
    coords = torch.arange(w, device=DEV).float().reshape(1, 1, w, 1).repeat(B, h, 1, 1)
    spx = torch.softmax(rnd(gen, B, 9, 4 * h, 4 * w), 1)

    def ours():
        vol = ops.build_gwc_volume(ml, mr, d, 8)
        gv = geo.CombinedGeoEncodingVolume(f1, f2, cv, num_levels=2, radius=4)
        out = None
        for _ in range(gru_iters):
            feat = gv(disp, coords)
            out = ops.context_upsample(disp * 4.0, spx, 4)
        return vol, feat, out

    def ref():
        vol = ocv.build_gwc_volume(ml, mr, d, 8)
        gv = ogeo.GeoEncodingVolume(f1, f2, cv, num_levels=2, radius=4)
        out = None
        for _ in range(gru_iters):
            feat = gv(disp, coords)
            out = ogeo.context_upsample(disp * 4.0, spx)
        return vol, feat, out

    with torch.no_grad():
        ms, got = timeit(ours, iters)
        ms_ref, want = timeit(ref, max(2, iters // 3), warm=1)
    emit(config="c5 IGEV hot path, B=%d @480x640: gwc volume (C=96,G=8,D'=48) + %d x (geo-volume lookup + context_upsample)" % (B, gru_iters),
         ms_per_step=round(ms, 3), pairs_per_s=round(B * 1e3 / ms, 2), reference_cudnn_fp32_ms=round(ms_ref, 2),
         speedup_vs_reference_gpu=round(ms_ref / ms, 2),
         max_abs_diff={"volume": float("%.2e" % (got[0] - want[0]).abs().max().item()),
                       "lookup": float("%.2e" % (got[1] - want[1]).abs().max().item()),
                       "upsample": float("%.2e" % (got[2] - want[2].reshape(got[2].shape)).abs().max().item())})


def gw(iters):
    """GwcNet hot path (gwc+concat volume -> 3D aggregation -> fused tail) at widths the whole-row tensor-core kernels do not serve:
    the reference's own timing shape 1x3x544x960 (tools/measure.py:32, W' = 240) and a KITTI crop 384x1248 (W' = 312).  Three
    columns: column-tile tcgen05 kernels, the fp32 CUDA-core kernels of the same engine (what round 1 ran at these widths) and the
    oracle modules on cuDNN fp32."""
    for (h, w) in ((544, 960), (384, 1248)):
        gen = torch.Generator().manual_seed(17)
        hq, wq = h // 4, w // 4
        ml, mr = rnd(gen, 1, 320, hq, wq), rnd(gen, 1, 320, hq, wq)
        cl, cr = rnd(gen, 1, 12, hq, wq), rnd(gen, 1, 12, hq, wq)
        m = oagg.GwcDispProcessor(maxdisp=192, downsample=4, num_groups=40, use_concat_volume=True, concat_channels=12).eval()
        m.load_state_dict(si.seeded_state_dict(m.state_dict(), seed=41, scale={"classif3.2.weight": 60.0}))
        m.to(DEV)
        eng = agg.GwcAggregation(m)

        def ours():
            return eng(ops.gwc_concat_volume(ml, mr, cl, cr, 48, 40), h, w)

        def ref():
            vol = torch.cat((ocv.build_gwc_volume(ml, mr, 48, 40), ocv.build_concat_volume(cl, cr, 48)), 1)
            return m(vol, h, w)

        with torch.no_grad():
            ms, got = timeit(ours, iters)
            agg.USE_TENSOR_CORES = False
            try:
                ms_cc, got_cc = timeit(lambda: agg.GwcAggregation(m)(ops.gwc_concat_volume(ml, mr, cl, cr, 48, 40), h, w), max(2, iters // 3), warm=1)
            finally:
                agg.USE_TENSOR_CORES = True
            ms_ref, want = timeit(ref, max(2, iters // 3), warm=1)
        emit(config="gw GwcNet hot path, 1 pair @%dx%d D=192 (W' = %d: column-tile tcgen05 kernels)" % (h, w, wq),
             ms_per_step=round(ms, 3), pairs_per_s=round(1e3 / ms, 2), cuda_core_kernels_ms=round(ms_cc, 2),
             reference_cudnn_fp32_ms=round(ms_ref, 2), speedup_vs_cuda_core=round(ms_cc / ms, 2),
             speedup_vs_reference_gpu=round(ms_ref / ms, 2),
             epe_vs_reference_gpu_px=float("%.3e" % (got - want.reshape(got.shape)).abs().mean().item()),
             epe_vs_cuda_core_px=float("%.3e" % (got - got_cc).abs().mean().item()), disparity_std_px=round(want.std().item(), 2),
             overflow_count=ops.tc_overflow_count())


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="c1,c3,c3h,c4,c5,gw")
    ap.add_argument("--iters", type=int, default=10)
    a = ap.parse_args()
    for name in a.only.split(","):
        try:
            {"c1": c1, "c3": c3, "c3h": c3h, "c4": c4, "c5": c5, "gw": gw}[name](a.iters)
        except Exception as exc:                                               # one config must not hide the others
            emit(config=name, error=repr(exc)[:300])
    if WORLD > 1:
        dist.destroy_process_group()
