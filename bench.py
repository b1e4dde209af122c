#!/usr/bin/env python
"""bench.py -- stereo pairs/sec for GwcNet @256x512, D=192 (BASELINE.json metric), 1..8 x B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch 8] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one GwcNet inference forward (2D backbone -> cost volume -> 3D aggregation -> soft-argmin) over one batch
of B=8 synthetic SceneFlow-shaped pairs per GPU (BASELINE.json configs[1]); batches shard over the GPUs (weak scaling,
independent pairs) and ONE NCCL all_gather of the per-image EPE partial sums closes the timed region, as in the
reference's eval loop (stereo/modeling/trainer_template.py:313-329).

Reported in one JSON line (rank 0):
  value      pairs/s, inputs already resident in HBM, CUDA-event timed, max over ranks
  e2e        same metric through the public model call with PINNED HOST inputs: H2D copy of the images + ground truth
             and D2H read-back of the per-image EPE inside the timed region, every step
  roofline   the DOMINANT kernel family of the step (3x3x3 Conv3d / ConvTranspose3d on tcgen05, split-operand fp32-accurate
             MMAs; tensor-bound), timed live with CUDA events around every launch inside the timed steps
  roofline_volume  the cost-volume kernel the metric names (HBM-bound) against MEASURED_PEAKS.json hbm_gbs and the 8 TB/s nominal;
             roofline_cuda_core = the fp32 layers still on CUDA cores
  cpu_baseline  the UNMODIFIED reference GwcNet (oracle/_ref, staged by oracle/make_ref.py; kind "reference") on the host
             cores, bounded sample -- the oracle port (kind "port") only when the staged reference is absent
  parity_epe_px  mean |disparity - reference| of one pair of the timed batch: this library on the GPU vs that CPU forward
  dropin     the same step through the reference's OWN GwcNet class + openstereo_b200.patch.patch() (what a maintainer gets)
  comparators  the unmodified reference on the same B200 (cuDNN fp32, TF32 off) and its Triton gwc kernel
               (fast_foundationstereo/core/submodule.py:443-478) against this library's gwc volume kernel
--impl reference times the reference's own CPU implementation as the reference arm.
--dump-outputs DIR writes what the last timed step returned (rank 0) as float32 .npy files: disp_pred.npy, the (B, 256, 512)
disparities of that step's batch, and epe_partials.npy, the gathered (B * n_gpus, 2) per-image {sum |err|, #valid}
(--impl reference: disp_pred.npy of its 1-pair step).  Inputs and weights are seeded, so two builds run with the same
arguments can be compared output for output.  The EPE sums are float32 block partials added with atomics, so they vary
in the last bits from run to run; disp_pred does not.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "stereo_pairs_per_sec_gwcnet_256x512_d192"
# dram__bytes_read.sum + dram__bytes_write.sum per launch at B = 8 from `ncu --set full` captures of this command
# (profiles/README.md names the capture each figure comes from); None = not captured for the current kernel version
NCU_TRAFFIC = {"volume_kernel": 919946496, "conv3d_tc_kernel": 765931264}
CFG = {"MAX_DISP": 192, "USE_CONCAT_VOLUME": True, "CONCAT_CHANNELS": 12, "DOWNSAMPLE": 4, "NUM_GROUPS": 40}
H, W = 256, 512


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d.get("hbm_gbs", 6650.0)), "measured (MEASURED_PEAKS.json)", float(d.get("sm_max_mhz", 1965.0))
    return 6650.0, "fallback (B200_PROFILING.md)", 1965.0


def synthetic_weights(model, seed=1):
    """Architecture-shaped random weights (no checkpoints ship with the reference; no network).  Variance-preserving
    normal conv weights and randomised BN statistics, so activations stay O(1) -- default init collapses the logits."""
    gen = torch.Generator().manual_seed(seed)
    sd = model.state_dict()
    for key in sorted(sd):
        t = sd[key]
        if key.endswith("num_batches_tracked") or "disp_regression" in key:
            continue
        if key.endswith("running_var"):
            v = torch.rand(t.shape, generator=gen) + 0.5
        elif key.endswith("running_mean") or (t.dim() == 1 and not key.endswith("weight")):
            v = torch.randn(t.shape, generator=gen) * 0.1
        elif t.dim() == 1:
            v = torch.rand(t.shape, generator=gen) * 0.5 + 0.5
        else:
            fan_in = t[0].numel()
            v = torch.randn(t.shape, generator=gen) * (1.0 / fan_in) ** 0.5
        sd[key] = v.to(t.dtype)
    sd["DispProcessor.classif3.2.weight"] = sd["DispProcessor.classif3.2.weight"] * 145.0
    model.load_state_dict(sd)
    return model


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self):
        self.proc, self.path = None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.QUERY, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self, n_gpus):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        clocks, reasons, mx = [], set(), None
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 8 or not f[0].isdigit() or int(f[0]) >= n_gpus:
                    continue
                try:
                    power = float(f[3])
                    clk = float(f[1])
                except ValueError:
                    continue
                mx = float(f[2])
                if power > 250.0:                                  # sample taken under load
                    clocks.append(clk)
                for name, val in zip(names, f[4:8]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if clocks:
            out["sm_mhz"] = statistics.median(clocks)
        out["sm_max_mhz"] = mx
        out["reasons"] = sorted(reasons)
        out["samples_under_load"] = len(clocks)
        return out


def usable_cores():
    """Host threads this process may really use: min(affinity mask, cgroup CPU quota) -- os.cpu_count() alone
    oversubscribes a quota-limited container and makes the CPU arm look far slower than it is."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // per))
        except Exception:
            pass
    return max(1, n)


def dist_setup(n_gpus):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
    elif n_gpus > 1:
        raise SystemExit("--gpus %d needs torchrun (one process per GPU); WORLD_SIZE is 1" % n_gpus)
    return world, rank, local


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()


def reference_available():
    try:
        from oracle import _reference_shim as shim
        return shim.available()
    except Exception:
        return False


def reference_model():
    """-> (model, kind).  The UNMODIFIED reference GwcNet built by its own class from its own cfgs/gwcnet/gwcnet_sceneflow.yaml
    (oracle/_ref on the GPU box: byte copies staged by oracle/make_ref.py), kind "reference"; the oracle port (same aten calls,
    bit-equal: tests/test_oracle_pins_reference.py), kind "port", only when no reference tree is present.  Same synthetic weights
    as the timed model (identical state_dict keys).  Checker / baseline legs only."""
    if reference_available():
        from oracle import _reference_shim as shim
        cfg = shim.load_cfg("cfgs/gwcnet/gwcnet_sceneflow.yaml").MODEL
        assert (cfg.MAX_DISP, cfg.NUM_GROUPS, cfg.CONCAT_CHANNELS) == (CFG["MAX_DISP"], CFG["NUM_GROUPS"], CFG["CONCAT_CHANNELS"])
        m = shim.load("stereo.modeling.models.gwcnet.gwcnet").GwcNet(cfg).eval()
        return synthetic_weights(m), "reference"
    from oracle import models as omodels
    m = omodels.GwcNet(CFG["MAX_DISP"], CFG["USE_CONCAT_VOLUME"], CFG["CONCAT_CHANNELS"], CFG["DOWNSAMPLE"],
                       CFG["NUM_GROUPS"]).eval()
    return synthetic_weights(m), "port"


def time_cpu(model, pairs_per_step, steps, warmup, x=None):
    """-> (seconds for `steps` forwards, last output).  x defaults to seeded synthetic pairs."""
    if x is None:
        gen = torch.Generator().manual_seed(0)
        x = {"left": torch.randn(pairs_per_step, 3, H, W, generator=gen), "right": torch.randn(pairs_per_step, 3, H, W, generator=gen)}
    out = None
    with torch.no_grad():
        for _ in range(warmup):
            model(dict(x))
        t0 = time.perf_counter()
        for _ in range(steps):
            out = model(dict(x))["disp_pred"]
        dt = time.perf_counter() - t0
    return dt, out


def run_reference(args):
    """Reference arm: the reference's own CPU path (unmodified GwcNet from oracle/_ref) with every host thread, rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = usable_cores()
    torch.set_num_threads(cores)
    model, kind = reference_model()
    pairs = 1                                                       # bounded sample: one pair of the B=8 batch per step
    dt, out = time_cpu(model, pairs, args.steps, min(args.warmup, 2))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"disp_pred": out})
    value = pairs * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": min(args.warmup, 2), "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "GwcNet cfgs/gwcnet_sceneflow 256x512 D=192 (configs[1]); CPU step = 1 pair sample",
                   "global_batch": pairs, "parallelism": "cpu-threads"},
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": cores, "kind": kind,
                         "sample": "%d forward(s) of 1 pair; %s" % (args.steps, "unmodified reference GwcNet class (oracle/_ref)"
                                                                   if kind == "reference" else "oracle port of the reference")},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_ours(args):
    world, rank, local = dist_setup(args.gpus)
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    torch.backends.cudnn.allow_tf32 = False                         # fp32 end to end (cfg AMP: false; 1e-3 px EPE bar)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.benchmark = True
    from openstereo_b200 import _lib, host_models, ops

    B = args.batch
    model = synthetic_weights(host_models.GwcNet(CFG)).eval().to(dev)
    gen = torch.Generator().manual_seed(1234 + rank)
    rot = args.rotate                                               # distinct input batches: rot * 12.6 MB > L2 (126 MB)
    host_left = [torch.randn(B, 3, H, W, generator=gen).pin_memory() for _ in range(rot)]
    host_right = [torch.randn(B, 3, H, W, generator=gen).pin_memory() for _ in range(rot)]
    host_gt = [(torch.rand(B, H, W, generator=gen) * 190 + 1).pin_memory() for _ in range(rot)]
    dev_left = [t.to(dev) for t in host_left]
    dev_right = [t.to(dev) for t in host_right]
    dev_gt = [t.to(dev) for t in host_gt]
    host_epe = torch.empty(B, 2).pin_memory()

    def step_resident(i):
        k = i % rot
        with torch.no_grad():
            disp = model({"left": dev_left[k], "right": dev_right[k]})["disp_pred"]
            return disp, ops.epe_partial(disp, dev_gt[k], CFG["MAX_DISP"])

    def step_e2e(i):
        k = i % rot
        with torch.no_grad():
            left = host_left[k].to(dev, non_blocking=True)
            right = host_right[k].to(dev, non_blocking=True)
            gt = host_gt[k].to(dev, non_blocking=True)
            disp = model({"left": left, "right": right})["disp_pred"]
            part = ops.epe_partial(disp, gt, CFG["MAX_DISP"])
            host_epe.copy_(part, non_blocking=True)
            torch.cuda.current_stream().synchronize()               # the caller reads the metric every step
            return disp, part

    from openstereo_b200.distributed import gather_epe_partials

    def gather(part):
        return gather_epe_partials(part)[0]                         # the single collective of the path (NCCL all_gather)

    def timed(step_fn, steps, profile):
        barrier(world)
        torch.cuda.synchronize()
        if profile:
            ops.profile_start()
        launches0 = _lib.launch_count()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        disp = part = None
        for i in range(steps):
            disp, part = step_fn(i)
        allparts = gather(part)
        stop.record()
        torch.cuda.synchronize()
        barrier(world)
        ms = start.elapsed_time(stop)
        prof = ops.profile_stop() if profile else None
        launches = _lib.launch_count() - launches0
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([ms, float(launches)], device=dev, dtype=torch.float64)
            mx = t.clone()
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            sm = t.clone()
            dist.all_reduce(sm, op=dist.ReduceOp.SUM)
            ms, launches = mx[0].item(), int(sm[1].item())
        return ms, launches, prof, allparts, disp

    for i in range(max(args.warmup, 3)):
        step_resident(i)
        step_e2e(i)
    torch.cuda.synchronize()

    sampler = ClockSampler()
    if rank == 0:
        sampler.start()
    if os.environ.get("OSB_NCU_RANGE"):                             # `ncu --profile-from-start off`: capture only the timed steps
        torch.cuda.cudart().cudaProfilerStart()
    ms, launches, prof, parts, last_disp = timed(step_resident, args.steps, profile=True)
    if os.environ.get("OSB_NCU_RANGE"):
        torch.cuda.cudart().cudaProfilerStop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"disp_pred": last_disp, "epe_partials": parts})
    del last_disp
    ms_e2e, _, _, _, _ = timed(step_e2e, args.steps, profile=False)
    clocks = sampler.stop(args.gpus) if rank == 0 else None
    if rank != 0:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()
        return

    pairs = B * world * args.steps
    value = pairs / (ms / 1e3)
    e2e_value = pairs / (ms_e2e / 1e3)
    epe = (parts[:, 0] / parts[:, 1].clamp(min=1)).mean().item()
    hbm_peak, peak_src, sm_max = measured_peaks()

    def kernel_stats(name):
        ev = prof.get(name, [])
        t = [a.elapsed_time(b) for a, b in ev]
        return (sum(t) / len(t), len(t), sum(t)) if t else (None, 0, 0.0)

    step_ms = ms / args.steps
    vol_ms, vol_n, vol_total = kernel_stats("osb_gwc_concat_volume_fwd")
    vol_bytes = 4 * (2 * B * (320 + 12) * 64 * 128 + B * 64 * 48 * 64 * 128)        # BASELINE.md section 3
    roof_vol = None
    if vol_ms:
        ach = vol_bytes / vol_ms / 1e6
        roof_vol = {"kernel": "volume_kernel (gwc+concat fused)", "bound": "hbm", "achieved": round(ach, 1), "peak": hbm_peak,
                    "unit": "GB/s", "frac": round(ach / hbm_peak, 4), "frac_of_8TBs_nominal": round(ach / 8000.0, 4),
                    "peak_source": peak_src, "alg_bytes_per_launch": vol_bytes, "ms_per_launch": round(vol_ms, 4),
                    "traffic": NCU_TRAFFIC.get("volume_kernel") if B == 8 else None, "share_of_step": round(vol_total / ms, 4)}
    # ---- 3D aggregation (SURVEY.md section 8a row a6): MACs per pair of GwcNet-gc at D'=48, H'=64, W'=128
    vox = 48 * 64 * 128
    macs = {
        # stem dres0a (64->32) + dres0b, dres1a, dres1b, classif3a (32->32) at full resolution; 3 x (conv2, conv4)
        "osb_conv3d_k3_tc_fwd": vox * 27 * 32 * (64 + 4 * 32) + 3 * (vox // 8 * 27 * 64 * 64 + vox // 64 * 27 * 128 * 128),
        # 3 x (conv1 32->64 to 1/2, conv3 64->128 to 1/4): MACs counted at the OUTPUT voxels
        "osb_conv3d_k3_s2_tc_fwd": 3 * (vox // 8 * 27 * 32 * 64 + vox // 64 * 27 * 64 * 128),
        # 3 x (conv5 128->64, conv6 64->32): every INPUT voxel feeds 27 taps
        "osb_deconv3d_k3_tc_fwd": 3 * (vox // 64 * 27 * 128 * 64 + vox // 8 * 27 * 64 * 32),
        # redir1 (32->32, full) and redir2 (64->64, half) of the three hourglasses
        "osb_conv1x1_ndhwc_fwd": 3 * (vox * 32 * 32 + vox // 8 * 64 * 64),
        # classif3b 32->1 head
        "osb_conv3d_k3_c1_ndhwc_fwd": vox * 27 * 32,
        # 2D backbone residual blocks on the same kernels (two images per pair): 8 front convs 32->32 @128x256, 30 layer2 convs
        # 64->64, 4 layer3 + 6 dilated layer4 convs 128->128 @64x128 (gwcnet_backbone.py:38-60) + lastconv's 320->128 3x3
        "osb_conv2d_k3_tc_fwd": 2 * 9 * (8 * 128 * 256 * 32 * 32 + 30 * 64 * 128 * 64 * 64 + 10 * 64 * 128 * 128 * 128
                                         + 64 * 128 * 320 * 128),
    }
    agg_macs = sum(v for k, v in macs.items() if k != "osb_conv2d_k3_tc_fwd")      # = 116.30 GMAC, SURVEY.md section 8a row a6
    tc_names = ["osb_conv3d_k3_tc_fwd", "osb_conv3d_k3_s2_tc_fwd", "osb_deconv3d_k3_tc_fwd", "osb_conv2d_k3_tc_fwd"]
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            bf16_peak = float(json.load(f).get("bf16_tflops_sustained"))
    except Exception:
        bf16_peak = 1400.0
    mma_kind = ops.tc_operand_kind()                                # "tf32" (3xTF32) or "f16" (3xFP16 split)
    tc_peak = bf16_peak / (2.0 if mma_kind == "tf32" else 1.0)      # dense tf32 = half the 16-bit rate
    roofline = None
    tc_total = sum(kernel_stats(n)[2] for n in tc_names)
    if tc_total > 0:
        per = {}
        for n in tc_names:
            _, cnt, tot = kernel_stats(n)
            if tot > 0:
                per[n] = {"launches_per_step": cnt // args.steps, "ms_per_step": round(tot / args.steps, 3),
                          "useful_tflops": round(2 * macs[n] * B * args.steps / (tot / 1e3) / 1e12, 1)}
        ran = [n for n in tc_names if kernel_stats(n)[2] > 0]
        useful = 2 * sum(macs[n] for n in ran) * B * args.steps / (tc_total / 1e3) / 1e12
        roofline = {"kernel": "tcgen05 conv family (conv3d_tc / tcg / tcs2 / tcdc kernels: 3x3x3 s1, s2, transposed; the backbone's 3x3 "
                              "blocks as one-plane volumes), kind::%s, 3 split-operand MMAs per fp32-accurate product" % mma_kind,
                    "bound": "tensor", "achieved": round(3 * useful, 1), "peak": round(tc_peak, 1), "unit": "TFLOP/s",
                    "frac": round(3 * useful / tc_peak, 4), "useful_fp32_equivalent_tflops": round(useful, 1),
                    "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained%s; achieved counts the 3 issued MMAs"
                                   % (" / 2 (dense tf32)" if mma_kind == "tf32" else " (dense 16-bit)"),
                    "alg_flops_per_step": 2 * sum(macs[n] for n in ran) * B, "share_of_step": round(tc_total / ms, 4),
                    "traffic": NCU_TRAFFIC.get("conv3d_tc_kernel") if B == 8 else None, "per_kernel": per}
    cc_names = ["osb_conv3d_k3_bn_act_fwd", "osb_deconv3d_bn_act_fwd", "osb_conv3d_1x1_bn_act_fwd", "osb_conv1x1_ndhwc_fwd",
                "osb_conv3d_k3_c1_ndhwc_fwd"]
    cc_total = sum(kernel_stats(n)[2] for n in cc_names)
    fp32_peak = 148 * 128 * 2 * sm_max * 1e6 / 1e12                 # derived: SMs x fp32 lanes x 2 x max clock
    roof_cc = None
    if cc_total > 0:
        cc_flops = 2 * (agg_macs - (sum(macs[n] for n in tc_names[:3]) if tc_total > 0 else 0)) * B
        ach = cc_flops * args.steps / (cc_total / 1e3) / 1e12
        roof_cc = {"kernel": "fp32 CUDA-core layers left in the aggregation", "bound": "fp32_fma", "achieved": round(ach, 2),
                   "peak": round(fp32_peak, 1), "unit": "TFLOP/s", "frac": round(ach / fp32_peak, 4),
                   "peak_source": "derived 148 SM x 128 lanes x 2 x %.0f MHz" % sm_max,
                   "alg_flops_per_step": cc_flops, "share_of_step": round(cc_total / ms, 4), "traffic": None}
    shares = {}
    for name, ev in prof.items():
        shares[name] = round(sum(a.elapsed_time(b) for a, b in ev) / ms, 4)

    # ---- checker / baseline legs (rank 0, N = 1 only): the reference on the host cores, parity of one timed pair against it,
    # the reference's own class through patch(), the reference on this GPU, its Triton gwc kernel.
    cpu, parity, dropin, comparators = None, None, None, None
    if world == 1 and not args.no_cpu_baseline:
        cores = usable_cores()
        torch.set_num_threads(cores)
        cm, kind = reference_model()
        n = 4
        x1 = {"left": host_left[0][:1].clone(), "right": host_right[0][:1].clone()}       # pair 0 of the first timed batch
        dt, want = time_cpu(cm, 1, n, 1, x=x1)
        cpu = {"value": round(n / dt, 4), "unit": "pairs/s", "cores": cores, "kind": kind,
               "sample": "%d forwards of 1 pair (pair 0 of the B=%d batch) through %s, %d threads"
                         % (n, B, "the unmodified reference GwcNet class (oracle/_ref)" if kind == "reference"
                            else "the oracle port of the reference", cores)}
        with torch.no_grad():
            got = model({"left": dev_left[0], "right": dev_right[0]})["disp_pred"][:1].cpu()  # the timed B=8 batch, image 0
        parity = {"epe_px": float("%.3e" % (got - want).abs().mean().item()), "bar_px": 1e-3, "against": kind + " on CPU",
                  "disparity_std_px": round(want.std().item(), 2), "pair": "image 0 of timed batch 0 (inside the B=%d forward)" % B}
        del cm
    if world == 1 and not args.no_comparators and reference_available():
        dropin, comparators = run_comparators(args, dev, B, dev_left, dev_right, dev_gt, value)

    line = {
        "metric": METRIC, "value": round(value, 3), "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": round(step_ms, 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "GwcNet cfgs/gwcnet/gwcnet_sceneflow.yaml, batch %d/GPU @256x512 D=192 (BASELINE configs[1])" % B,
                   "global_batch": B * world, "parallelism": "dp%d batch-shard, 1 all_gather of per-image EPE" % world,
                   "model_path": "openstereo_b200.host_models.GwcNet (state_dict-compatible mirror; `dropin` = the reference's class + patch())",
                   "l2": "inputs rotate over %d distinct batches (%.0f MB > 126 MB L2); per-step activations ~6 GB" % (rot, rot * 2 * B * 3 * H * W * 4 / 1e6),
                   "weights": "synthetic seeded init (no checkpoints ship with the reference)"},
        "clocks": clocks,
        "e2e": {"value": round(e2e_value, 3), "unit": "pairs/s", "ms_per_step": round(ms_e2e / args.steps, 4),
                "h2d_bytes_per_step": (2 * B * 3 * H * W + B * H * W) * 4, "d2h_bytes_per_step": B * 2 * 4},
        "gpu_launches": launches,
        "roofline": roofline, "cpu_baseline": cpu, "parity": parity, "parity_epe_px": parity["epe_px"] if parity else None,
        "dropin": dropin, "comparators": comparators,
        "roofline_volume": roof_vol, "roofline_cuda_core": roof_cc, "kernel_share_of_step": shares,
        "mean_epe_vs_synthetic_gt": round(epe, 3),
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def dump_outputs(path, arrays):
    """name -> tensor, written as path/<name>.npy in float32."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.detach().float().cpu().numpy())


def run_comparators(args, dev, B, dev_left, dev_right, dev_gt, mirror_value):
    """N = 1 legs that need the staged reference (oracle/_ref).  Each is CUDA-event timed after warm-up, resident inputs, same
    synthetic weights and batches as the main arm.
      dropin                     the reference's own GwcNet class + patch(): pairs/s and its ratio to the mirror's value
      reference_gpu_cudnn_fp32   the UNMODIFIED reference forward on this B200 (cuDNN fp32, TF32 off) -- SURVEY.md section 8d's GPU bar
      triton_gwc                 the reference's Triton gwc kernel (normalize=False, / K to match build_gwc_volume's mean)
                                 against osb_gwc_volume_fwd at the config-2 shape (8, 320, 64, 128), D' = 48, G = 40"""
    from oracle import _reference_shim as shim
    from openstereo_b200 import ops
    from openstereo_b200.patch import patch
    rot = len(dev_left)

    def timed_model(m, steps, warm):
        with torch.no_grad():
            for i in range(warm):
                m({"left": dev_left[i % rot], "right": dev_right[i % rot]})
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(steps):
                d = m({"left": dev_left[i % rot], "right": dev_right[i % rot]})["disp_pred"]
                ops.epe_partial(d.float().contiguous(), dev_gt[i % rot], CFG["MAX_DISP"])
            b.record()
            torch.cuda.synchronize()
        return a.elapsed_time(b) / steps, d

    dropin, comp = None, {}
    try:
        ref, _ = reference_model()
        ref = ref.to(dev)
        ms_ref, _ = timed_model(ref, 3, 2)
        with torch.no_grad():
            d_ref = ref({"left": dev_left[0], "right": dev_right[0]})["disp_pred"]
        comp["reference_gpu_cudnn_fp32"] = {"value": round(B / (ms_ref / 1e3), 2), "unit": "pairs/s", "ms_per_step": round(ms_ref, 2),
                                            "what": "unmodified reference GwcNet forward on this GPU, B=%d, cuDNN fp32, allow_tf32=False" % B}
        patch(ref)                                                  # same instance, now on this library's kernels
        ms_pat, _ = timed_model(ref, args.steps, 3)
        with torch.no_grad():
            d_pat = ref({"left": dev_left[0], "right": dev_right[0]})["disp_pred"]
        dropin = {"value": round(B / (ms_pat / 1e3), 3), "unit": "pairs/s", "ms_per_step": round(ms_pat, 4),
                  "path": "reference GwcNet class (oracle/_ref) + openstereo_b200.patch.patch(model)",
                  "ratio_to_mirror": round(B / (ms_pat / 1e3) / mirror_value, 4),
                  "epe_vs_reference_on_this_gpu_px": float("%.3e" % (d_pat - d_ref).abs().mean().item())}
        del ref
    except Exception as exc:                                        # a comparator must never take the bench line down
        comp["reference_gpu_cudnn_fp32"] = comp.get("reference_gpu_cudnn_fp32") or {"error": repr(exc)[:200]}
    try:
        sub = shim.load("stereo.modeling.models.fast_foundationstereo.core.submodule")
        g = torch.Generator(device=dev).manual_seed(5)
        lf, rf = torch.randn(B, 320, 64, 128, device=dev, generator=g), torch.randn(B, 320, 64, 128, device=dev, generator=g)
        # the reference's wrapper views permute(0,2,3,1) as (B*H, W, C): it expects channels_last features (as its own backbone emits)
        lf_cl, rf_cl = lf.contiguous(memory_format=torch.channels_last), rf.contiguous(memory_format=torch.channels_last)

        def timeit(fn, n=10):
            for _ in range(3):
                out = fn()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(n):
                out = fn()
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / n, out

        ms_tr, v_tr = timeit(lambda: sub.build_gwc_volume_triton(lf_cl, rf_cl, 48, 40, normalize=False))
        ms_us, v_us = timeit(lambda: ops.build_gwc_volume(lf, rf, 48, 40))
        comp["triton_gwc"] = {"reference_triton_ms": round(ms_tr, 4), "this_library_ms": round(ms_us, 4), "speedup": round(ms_tr / ms_us, 2),
                              "max_abs_diff": float("%.2e" % (v_tr / 8.0 - v_us).abs().max().item()),
                              "what": "build_gwc_volume_triton(normalize=False) [sum over K=8; /8 for the mean] vs osb_gwc_volume_fwd, "
                                      "(%d,320,64,128) D'=48 G=40" % B}
    except Exception as exc:
        comp["triton_gwc"] = {"error": repr(exc)[:200]}
    return dropin, comp


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--rotate", type=int, default=12)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-comparators", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
