#!/usr/bin/env python
"""bench.py -- diffusion-steps/sec of the CLIP-guided sampling step (BASELINE.json metric) on N B200s.

    python bench.py --gpus 1 --steps 20 --warmup 5                       # this framework, cfg2 per GPU
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference --steps K --warmup W               # the oracle port on the host CPU cores
    python bench.py --steps K --warmup W --dump-outputs DIR              # also DIR/sample.npy, DIR/pred_xstart.npy of the last timed step

A "step" is one ddim_sample_with_grad iteration (UNet fwd -> cutouts -> CLIP ViT fwd/bwd -> losses -> UNet dgrad ->
DDIM update) of BASELINE.json configs[1]: 256x256, ddim250, 1 image per GPU, 16 cutouts, ViT-B/32, synthetic noise and
seeded random weights of the published architectures.  With N GPUs every rank owns one image (weak scaling, no
data-path collective; one NCCL all-gather of the final images), and `value` counts image-steps per second.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch as th

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# per-GPU shards of the BASELINE.json configurations; cfg2 is the metric's configuration (the default and the only one the driver
# runs), the others are extra measurements (--workload).  tflop = algorithmic FLOPs per image-step (SURVEY.md 8d, fwd + dgrad).
WORKLOADS = {
    "cfg2": dict(image_size=256, respacing="ddim250", per_gpu_batch=1, cutn=16, clip="ViT-B/32", lpips=False, tflop=4.775,
                 name="BASELINE configs[1]: image_size=256, respace=ddim250, batch=1 per GPU, cutn=16, ViT-B/32"),
    "cfg3": dict(image_size=256, respacing="1000", per_gpu_batch=1, cutn=32, clip="ViT-B/32", lpips=False, tflop=5.059,
                 name="BASELINE configs[2] shard: image_size=256, respace=1000 (ancestral), batch=1 per GPU, cutn=32, ViT-B/32"),
    "cfg4": dict(image_size=512, respacing="ddim250", per_gpu_batch=1, cutn=16, clip="ViT-B/16", lpips=False, tflop=9.09,
                 name="BASELINE configs[3] shard: image_size=512, respace=ddim250, batch=1 per GPU, cutn=16, ViT-B/16"),
    "cfg5": dict(image_size=512, respacing="1000", per_gpu_batch=1, cutn=64, clip="ViT-L/14", lpips=True, tflop=29.1,
                 name="BASELINE configs[4] shard: image_size=512, respace=1000 (ancestral), batch=1 per GPU, cutn=64, ViT-L/14, "
                      "init image + LPIPS init_scale=1000 (LPIPS FLOPs not counted)"),
    # not a BASELINE configuration: the reference's default arguments (cgd/cgd.py:20-33) -- the 128x128 checkpoint (4 heads of 128 / 192 /
    # 256 channels: csrc/attention_wide.cu); tflop = the executed contractions of the op list (Plan.conv_flops)
    "default128": dict(image_size=128, respacing="1000", per_gpu_batch=1, cutn=16, clip="ViT-B/32", lpips=False, tflop=1.492,
                       name="reference defaults: image_size=128, respace=1000 (ancestral), batch=1 per GPU, cutn=16, ViT-B/32"),
}
CFG = WORKLOADS["cfg2"]
FLOP_PER_IMAGE_STEP = 4.775e12  # SURVEY.md 8d: UNet 2.240+2.252, CLIP 0.141+0.143 TFLOP (fwd + dgrad)
DOMINANT = dict(M=65536, N=256, K=2304)  # 256^2 x 256ch conv3x3: 31 % of the UNet FLOPs (SURVEY App. C)
DUMP_BYTES = 64 << 20  # --dump-outputs: the .npy files together stay below this


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    fb = dict(burst=1590.0, sustained=1400.0, hbm=6650.0, src="fallback")  # B200_PROFILING.md's stated fallback
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            burst = float(d["bf16_tflops"])
            return dict(burst=burst, sustained=float(d.get("bf16_tflops_sustained", burst)), hbm=float(d.get("hbm_gbs", fb["hbm"])), src="measured")
        except (OSError, ValueError, KeyError, TypeError):  # unreadable / other schema: say "fallback" rather than abort the bench line
            pass
    return fb


def dump_outputs(path, arrays):
    """One float32 DIR/<name>.npy per array.  Above DUMP_BYTES in all, each array is cut to the same fixed, seeded sample of its
    flattened elements on every run, so that two builds' dumps stay comparable element for element."""
    os.makedirs(path, exist_ok=True)
    arrays = {k: v.detach().float().cpu() for k, v in arrays.items()}
    total = sum(a.numel() * 4 for a in arrays.values())
    budget = DUMP_BYTES - 1024 * len(arrays)  # room for the .npy headers
    for name, a in arrays.items():
        if total > budget:
            keep = a.numel() * budget // total
            a = a.flatten()[th.randperm(a.numel(), generator=th.Generator().manual_seed(0))[:keep].sort().values]
        np.save(os.path.join(path, f"{name}.npy"), a.numpy())


class ClockSampler:
    """SM clock / throttle reasons during the timed region (B200_PROFILING.md).  NVML from a sampling thread (one query ~50 us, every
    10 ms: a 250 ms timed region yields ~25 samples); `nvidia-smi -lms 200` as the fallback when pynvml is not usable."""

    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None
        self.nvml, self.samples, self._stop, self._thread = None, [], threading.Event(), None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)  # probe once: any failure falls back to nvidia-smi
            self.nvml, self.handle = pynvml, h
            self._thread = threading.Thread(target=self._poll, daemon=True)
            self._thread.start()
            return
        except Exception:
            self.nvml = None
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        get_reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(n, "nvmlDeviceGetCurrentClocksThrottleReasons", None)
        while not self._stop.is_set():
            try:
                mhz = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                bits = int(get_reasons(self.handle)) if get_reasons else 0
                self.samples.append((float(mhz), bits))
            except Exception:
                pass
            self._stop.wait(0.010)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            try:
                self._stop.set()
                self._thread.join(timeout=1.0)
                n = self.nvml
                mx = float(n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM))
                masks = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}  # nvml.h
                reasons = sorted(k for k, m in masks.items() if any(b & m for _, b in self.samples))
                sm = [v for v, _ in self.samples]
                return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": reasons, "samples": len(sm),
                        "source": "nvml, 10 ms"}
            except Exception as e:  # never let the sampler take the bench line down
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"nvml sampler failed: {type(e).__name__}"], "samples": 0}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = self.NAMES
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "source": "nvidia-smi -lms 200"}


# ------------------------------------------------------------------------------------------------ our arm
def build_engine(device, rank, world):
    from clip_guided_diffusion_b200 import gaussian_diffusion as gd
    from clip_guided_diffusion_b200 import guidance as pg
    from clip_guided_diffusion_b200 import unet as pu
    from clip_guided_diffusion_b200 import vit as pv
    from clip_guided_diffusion_b200 import weights as pw
    ucfg = pu.config_for(CFG["image_size"], class_cond=True)
    vcfg = pv.VIT_CONFIGS[CFG["clip"]]
    usd = pw.seeded_state_dict(pw.unet_param_shapes(ucfg), seed=1234)
    vsd = pw.seeded_state_dict(pw.vit_param_shapes(vcfg), seed=1235)
    extra = dict(lpips_sd=pw.seeded_lpips_state_dict(), init_scale=1000.0) if CFG["lpips"] else {}
    eng = pg.GuidedStepB200(ucfg, usd, vcfg, vsd, batch=CFG["per_gpu_batch"], num_cutouts=CFG["cutn"], device=device, rank=rank,
                            world_size=world, vit_streams=int(os.environ.get("CGD_VIT_STREAMS", "1")), **extra)
    if CFG["lpips"]:
        eng.set_init_image((th.rand(1, 3, CFG["image_size"], CFG["image_size"], generator=th.Generator().manual_seed(5)) * 2 - 1).to(device))
    del usd, vsd
    diff = gd.create_gaussian_diffusion(1000, "linear", CFG["respacing"], rescale_timesteps=ucfg.rescale_timesteps)
    th.manual_seed(0)
    tgt = th.nn.functional.normalize(th.randn(1, vcfg.output_dim), dim=-1)
    eng.set_targets(tgt, th.ones(1))
    mk = pg.MakeCutouts(vcfg.input_resolution, CFG["cutn"])
    cond = pg.CondFnB200(eng, diff, mk)
    return eng, diff, cond


def dominant_kernel_time(device, reps=24):
    """Average duration of the dominant conv launch (256x256 pixels, 256 -> 256 channels, 3x3), rotating over buffers that
    together exceed the 126 MB L2, CUDA events on the launching stream."""
    from clip_guided_diffusion_b200.plan import Plan, pack_conv
    th.manual_seed(0)
    plan = Plan()
    w = th.randn(256, 256, 3, 3) * (9 * 256) ** -0.5
    cw = pack_conv(plan, w, th.zeros(256), need_bwd=False, name="dom")
    nbuf = 4
    for _ in range(nbuf):
        x = plan.act(1, 256, 256, 256, "x")
        plan.conv(x, cw, name="dom")
    plan.finalize(device)
    for b in plan.bufs:
        if b.name == "x":
            plan.view(b).normal_()
    for _ in range(2):
        plan.run()
    th.cuda.synchronize()
    e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
    rounds = max(1, reps // nbuf)
    e0.record()
    for _ in range(rounds):
        plan.run()
    e1.record()
    th.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / (rounds * nbuf)


def conv_share(eng, mode, reps=3):
    """Summed duration and algorithmic FLOPs of every contraction (op CONV: 3x3 / 1x1 convs and the GEMMs, forward and dgrad) of
    one step, launched back to back on the current stream."""
    from clip_guided_diffusion_b200._lib import OP
    plan = eng.plan
    m = plan.marks
    segs = [("unet_emb", "unet_bwd"), ("vit_fwd", "vit_bwd"), ("vit_bwd", "vit_end"), ("unet_bwd", "unet_end")]
    if eng.lpips is not None:
        segs.append(("lpips", "lpips_end"))
    ks = [k for a, b in segs for k in range(m[a], m[b]) if plan.ops[k].code == OP["CONV"]]
    flop = 0.0
    for k in ks:
        flop += plan.conv_flops(k)
    for k in ks:
        plan.run(k, 1)
    th.cuda.synchronize()
    e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        for k in ks:
            plan.run(k, 1)
    e1.record()
    th.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / reps, flop, len(ks)


def run_ours(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run for N>1)"
    assert th.cuda.is_available(), "bench.py (own arm) needs a CUDA device; there is no CPU fallback"
    th.cuda.set_device(local)
    device = th.device("cuda", local)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    eng, diff, cond = build_engine(device, rank, world)
    MODE = "ddim" if CFG["respacing"].startswith("ddim") else "ancestral"
    B = eng.B
    T = diff.num_timesteps
    y0 = th.zeros(eng.global_batch, dtype=th.long)
    last = {}

    def step_resident(i, img):
        # x_t is fresh synthetic noise every step: with random (non-denoising) weights a chained trajectory diverges within a
        # few steps (pred_xstart ~ 1e3 and growing), which says nothing about throughput; timing is value-independent
        img = eng.draw_initial_noise()
        y = eng.draw_classes()
        out = eng.fused_step(diff, MODE, i, img, y, cond, 0.0)
        cond.current_timestep = max(cond.current_timestep - 1, 0)
        last.update(out)
        return out["sample"]

    # ---------------- device-resident loop (value)
    th.manual_seed(0)
    img = eng.draw_initial_noise()
    idx = T - 1
    for _ in range(args.warmup):
        img = step_resident(idx, img)
        idx = max(idx - 1, 0)
    eng.gather_final(img)  # warm-up of the collective too: communicator / channel set-up stays out of the timed region
    if world > 1:
        dist.barrier()
    th.cuda.synchronize()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        img = step_resident(idx, img)
        idx = max(idx - 1, 0)
    gathered = eng.gather_final(img)  # the run's single collective (one all_gather_into_tensor; identity at N = 1)
    e1.record()
    th.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = th.tensor([e0.elapsed_time(e1)], device=device)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    clocks = sampler.stop() if rank == 0 else None
    ms_total = float(ms.item())
    finite = bool(th.isfinite(img).all()) and tuple(gathered.shape) == (eng.global_batch, 3, eng.H, eng.W)
    if args.dump_outputs:
        # what the last timed step returned, every rank's rows in rank order; .cpu() before the next gather reuses its buffer
        outs = {k: eng.gather_final(v).cpu() for k, v in sorted(last.items())}
        if rank == 0:
            dump_outputs(args.dump_outputs, outs)

    # ---------------- end-to-end loop: host buffers, H2D of x_t and D2H of the sample inside every step
    host_x = th.empty(B, 3, eng.H, eng.W, pin_memory=True)
    host_out = th.empty(B, 3, eng.H, eng.W, pin_memory=True)
    host_x.copy_(th.randn(B, 3, eng.H, eng.W))
    idx_e = max(idx, 1)

    def step_host(i):
        y = th.randint(0, eng.unet.num_classes, (B,))  # host-side class draw, staged with the other per-step data
        eng.img(eng.unet.x_in).copy_(host_x, non_blocking=True)
        out = eng.fused_step(diff, MODE, i, eng.img(eng.unet.x_in), y, cond, 0.0)
        host_out.copy_(out["sample"], non_blocking=True)
        th.cuda.current_stream().synchronize()

    for _ in range(min(3, args.warmup)):
        step_host(idx_e)
    if world > 1:
        dist.barrier()
    th.cuda.synchronize()
    e0.record()
    for _ in range(args.steps):
        step_host(idx_e)
        idx_e = max(idx_e - 1, 0)
    e1.record()
    th.cuda.synchronize()
    ms_e = th.tensor([e0.elapsed_time(e1)], device=device)
    if world > 1:
        dist.all_reduce(ms_e, op=dist.ReduceOp.MAX)
    ms_e2e = float(ms_e.item())
    h2d = B * 3 * eng.H * eng.W * 4 + eng.h2d_bytes
    d2h = B * 3 * eng.H * eng.W * 4

    # ---------------- the PyTorch-CUDA build of the same step (north_star's ">= 2.5x" denominator), on every rank like our arm
    torch_base = None
    if not args.no_torch_baseline:
        try:
            torch_base = torch_cuda_baseline(device, max(5, min(10, args.steps)), dist if world > 1 else None, world)
        except Exception as e:  # context only: never lose the measured line
            torch_base = {"error": repr(e)[:300]}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk = peaks()
    conv_s, conv_flop, n_conv = conv_share(eng, MODE)
    launches = eng.launches_per_step(MODE)
    value = args.steps * eng.global_batch / (ms_total * 1e-3)
    e2e = args.steps * eng.global_batch / (ms_e2e * 1e-3)
    # roofline of the dominant kernel, timed alone right after the step loops
    t_dom = dominant_kernel_time(device)
    flops_dom = 2.0 * DOMINANT["M"] * DOMINANT["N"] * DOMINANT["K"]
    ach = flops_dom / t_dom / 1e12
    traffic = None
    tp = os.path.join(ROOT, "profiles", "dominant_conv_traffic.json")
    if os.path.exists(tp):
        traffic = json.load(open(tp)).get("dram_bytes_per_launch")
    line = {
        "metric": "diffusion-steps/sec", "value": value,
        "unit": f"image-steps/s (1 step of one {CFG['image_size']}x{CFG['image_size']} image, {CFG['cutn']} cutouts)",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "fp16 (fp32 accumulate / norm / softmax / sampler)", "data": "synthetic (x_t ~ N(0,1) redrawn every step, seeded random weights)",
        "config": {"workload": CFG["name"] + ", class-cond UNet, seeded random weights", "global_batch": eng.global_batch, "parallelism": f"dp{world} (batch shard, no data-path collective)",
                   "l2": "per-step working set (2.3 GB of packed weights + activations) exceeds the 126 MB L2; no explicit flush",
                   "finite": finite},
        "e2e": {"value": e2e, "unit": "image-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches * args.steps,
        "launches_per_step": launches,
        "clocks": clocks,
        "roofline": {"bound": "tensor", "achieved": ach, "peak": pk["burst"], "unit": "TFLOP/s", "frac": ach / pk["burst"], "traffic": traffic,
                     "kernel": "conv_tc2_kernel<256> 256x256x256->256 3x3 (M=65536,N=256,K=2304)", "peak_source": pk["src"] + " burst (kernel timed alone)",
                     "avg_launch_s": t_dom},
        "step_tensor_frac": CFG["tflop"] * 1e12 * value / world / (pk["sustained"] * 1e12),
    }
    # time-weighted fraction over EVERY contraction of the step (convs + GEMMs, both directions), so that `frac` above -- one layer
    # shape -- cannot be read as "the step runs at that fraction": their algorithmic FLOPs / their summed duration / peak
    line["roofline"].update({"step_conv_frac": conv_flop / conv_s / 1e12 / pk["sustained"], "step_conv_tflops": conv_flop / conv_s / 1e12,
                             "step_conv_ms": conv_s * 1e3, "step_conv_launches": n_conv,
                             "step_conv_note": "all CONV ops of one step launched back to back (no graph), CUDA events; vs the sustained peak"})
    if torch_base is not None:
        line["torch_cuda_baseline"] = torch_base
        if "value" in torch_base:
            line["vs_torch_cuda"] = value / torch_base["value"]
            line["vs_torch_cuda_e2e"] = e2e / torch_base["value_with_item_logging"]
    if world == 1 and not args.no_cpu_baseline and args.workload == "cfg2":
        line["cpu_baseline"] = cpu_baseline(sample_steps=3)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ CPU arms (oracle port)
_CPU_THREADS = None


def pick_cpu_threads() -> int:
    """Deterministic thread count of the CPU arms: every host core up to 32 (PyTorch's CPU convs stop scaling there: the build box'
    8 cores take 30 s/step, the B200 host ran 5-6 s/step with 16-48 threads and 206 s/step with 128; CGD_CPU_THREADS overrides)."""
    global _CPU_THREADS
    if _CPU_THREADS is None:
        _CPU_THREADS = int(os.environ.get("CGD_CPU_THREADS", "0")) or min(os.cpu_count() or 1, 32)
    return _CPU_THREADS


def oracle_cpu_setup():
    """The oracle (fp32 PyTorch restatement of the reference path) on the host cores -- the checker timed as the CPU baseline."""
    from oracle import diffusion as od
    from oracle import guidance as og
    from oracle.clip_vit import VIT_CONFIGS, CLIPVisualOnly
    from oracle.unet import UNetModel, config_for, seeded_init_
    th.set_num_threads(pick_cpu_threads())
    unet = seeded_init_(UNetModel(config_for(CFG["image_size"], True))).eval()
    clip = seeded_init_(CLIPVisualOnly(VIT_CONFIGS[CFG["clip"]]), seed=1235).eval()
    for p in list(unet.parameters()) + list(clip.parameters()):
        p.requires_grad_(False)
    from clip_guided_diffusion_b200 import unet as pu
    diff = od.create_gaussian_diffusion(1000, "linear", CFG["respacing"], rescale_timesteps=pu.config_for(CFG["image_size"], True).rescale_timesteps)
    tgt = th.nn.functional.normalize(th.randn(1, VIT_CONFIGS[CFG["clip"]].output_dim), dim=-1)
    extra = {}
    if CFG["lpips"]:  # cfg5: init image + LPIPS-VGG init loss (cgd/cgd.py:220-224), same synthetic weights / image as our arm
        from clip_guided_diffusion_b200 import weights as pw
        from oracle import lpips as ol
        init = th.rand(1, 3, CFG["image_size"], CFG["image_size"], generator=th.Generator().manual_seed(5)) * 2 - 1
        extra = dict(lpips_model=ol.LPIPSVgg(pw.seeded_lpips_state_dict()), init_tensor=init, init_scale=1000.0)
    cond = og.OracleCondFn(diff, clip, tgt, th.ones(1), cut_size=224, num_cutouts=CFG["cutn"], **extra)
    return unet, diff, cond


def oracle_cpu_steps(unet, diff, cond, n_steps, x=None):
    th.manual_seed(0)
    B = CFG["per_gpu_batch"]
    x = th.randn(B, 3, CFG["image_size"], CFG["image_size"]) if x is None else x
    times = []
    i = diff.num_timesteps - 1
    for _ in range(n_steps):
        t = th.full((B,), i, dtype=th.long)
        y = th.randint(0, 1000, (B,))
        t0 = time.perf_counter()
        out = diff.ddim_sample_with_grad(unet, x, t, clip_denoised=False, cond_fn=cond, model_kwargs={"y": y})
        times.append(time.perf_counter() - t0)
        x = out["sample"]
        cond.step_done()
        i -= 1
    return times, x


def torch_cuda_baseline(device, n_steps, dist=None, world=1):
    """The reference's PyTorch-CUDA configuration (BASELINE.md section 5): the same op sequence on cuDNN / cuBLAS / ATen with eager
    autograd -- fp16 UNet trunk (convert_to_fp16: conv weights of input/middle/output blocks), fp16 CLIP, fp32 norms -- via the
    oracle port because the reference's third-party packages cannot be installed offline.  One image per rank like our arm (weak
    scaling), time = max over ranks, measured twice: with the reference's per-step `.item()` loss logging (cgd/cgd.py:234-236,
    three host syncs per step) and without it."""
    from oracle import guidance as og
    th.backends.cudnn.benchmark = True
    unet, diff, cond = oracle_cpu_setup()
    unet = unet.to(device)
    for blocks in (unet.input_blocks, unet.middle_block, unet.output_blocks):
        for m in blocks.modules():
            if isinstance(m, (th.nn.Conv1d, th.nn.Conv2d)):
                m.half()
    unet.dtype = th.float16
    clip = cond.clip_model.to(device).half()
    for m in clip.modules():  # clip.model.convert_weights leaves LayerNorm in fp32
        if isinstance(m, th.nn.LayerNorm):
            m.float()
    extra = {}
    if cond.kw.get("lpips_model") is not None:
        lp = cond.kw["lpips_model"].to(device)
        lp.sd = {k: v.to(device) for k, v in lp.sd.items()}
        extra = dict(lpips_model=lp, init_tensor=cond.kw["init_tensor"].to(device), init_scale=cond.kw["init_scale"])
    cond = og.OracleCondFn(diff, clip, cond.target_embeds.to(device), cond.weights.to(device), cut_size=224, num_cutouts=CFG["cutn"], **extra)
    B = CFG["per_gpu_batch"]
    i = diff.num_timesteps - 1
    fn = diff.ddim_sample_with_grad if CFG["respacing"].startswith("ddim") else diff.p_sample_with_grad

    def one(i):
        x = th.randn(B, 3, CFG["image_size"], CFG["image_size"], device=device)
        t = th.full((B,), i, dtype=th.long, device=device)
        y = th.randint(0, 1000, (B,), device=device)
        return fn(unet, x, t, clip_denoised=False, cond_fn=cond, model_kwargs={"y": y})["sample"]

    res = {}
    for key, log_items in (("value", False), ("value_with_item_logging", True)):
        cond.log_items = log_items
        for _ in range(3):
            one(i)
        if dist is not None:
            dist.barrier()
        th.cuda.synchronize()
        e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(n_steps):
            out = one(i - k)
        e1.record()
        th.cuda.synchronize()
        ms = th.tensor([e0.elapsed_time(e1) / n_steps], device=device)
        if dist is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        res[key] = 1e3 * world * B / float(ms.item())
    return {"value": res["value"], "value_with_item_logging": res["value_with_item_logging"], "unit": "image-steps/s (whole job)",
            "ms_per_step": 1e3 * world * B / res["value"], "steps": n_steps, "n_gpus": world,
            "what": "oracle port on cuda: eager PyTorch autograd, fp16 UNet trunk + fp16 CLIP (cuDNN benchmark mode / cuBLAS / ATen), "
                    "one image per rank, max over ranks; with and without the reference's per-step .item() loss logging",
            "torch": th.__version__, "finite": bool(th.isfinite(out).all())}


def cpu_baseline(sample_steps=3):
    """rank 0, N = 1: one untimed (cold) step, then `sample_steps` timed ones -- the same protocol as the reference arm"""
    unet, diff, cond = oracle_cpu_setup()
    _, x = oracle_cpu_steps(unet, diff, cond, 1)
    times, _ = oracle_cpu_steps(unet, diff, cond, sample_steps, x)
    t = float(np.mean(times))
    return {"value": 1.0 / t, "unit": "image-steps/s", "cores": pick_cpu_threads(), "host_cpus": os.cpu_count(), "kind": "port",
            "sample": f"{sample_steps} full cfg2 steps of the fp32 oracle port after 1 untimed step (PyTorch CPU, {pick_cpu_threads()} threads), "
                      f"{t:.2f} s/step"}


def run_reference(args):
    """The reference's own algorithm on the host cores (fp32 oracle port: guided_diffusion / clip / lpips are not installable
    offline, DESIGN.md section 5).  Same metric / unit / config strings as our arm; --warmup W untimed steps, --steps K timed ones.
    One cfg2 step takes 5-6 s on a B200 host's CPU cores."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    unet, diff, cond = oracle_cpu_setup()
    _, x = oracle_cpu_steps(unet, diff, cond, args.warmup)  # the first one is the cold step (allocator, thread pool)
    n_timed = args.steps
    times, _ = oracle_cpu_steps(unet, diff, cond, n_timed, x)
    total = float(sum(times))
    value = n_timed / total
    line = {"impl": "reference", "metric": "diffusion-steps/sec", "value": value,
            "unit": f"image-steps/s (1 step of one {CFG['image_size']}x{CFG['image_size']} image, {CFG['cutn']} cutouts)",
            "n_gpus": args.gpus, "steps": n_timed, "warmup": args.warmup,
            "ms_per_step": total / n_timed * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic (seeded random weights)",
            "config": {"workload": CFG["name"] + ", class-cond UNet, seeded random weights", "global_batch": 1,
                       "parallelism": "host CPU threads (rank 0 only)",
                       "note": "the reference's own algorithm as the fp32 oracle port on the host CPU; guided_diffusion / clip are not "
                               "installable offline"},
            "cpu_baseline": {"value": value, "unit": "image-steps/s", "cores": pick_cpu_threads(), "host_cpus": os.cpu_count(), "kind": "port",
                             "sample": f"{n_timed} full cfg2 steps after {args.warmup} untimed"},
            "e2e": {"value": value, "unit": "image-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-torch-baseline", action="store_true", help="skip the PyTorch-CUDA (cuDNN/cuBLAS eager autograd) oracle-port arm")
    ap.add_argument("--torch-baseline", action="store_true", help="(default now; kept for old command lines)")
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS), help="per-GPU shard of a BASELINE.json configuration (default: the metric's)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last step's sample and pred_xstart "
                                                          "(float32, the whole batch) to DIR/<name>.npy; same arguments, same inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what --impl ours computed")
    global CFG
    CFG = WORKLOADS[args.workload]
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
