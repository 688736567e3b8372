#!/usr/bin/env python
"""Headline benchmark: denoised frames/s at 512x512, 16-frame window, 20 DDIM steps (BASELINE.json, config 2).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
  (N > 1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...)

One "step" = one complete denoise of the workload: 20 DDIM steps of the Visual-Conditioned Parallel-Denoise loop
(every window: UNet3D forward with CFG batch 2 -> overlap mean -> CFG -> DDIM update) on synthetic latents.
N = 1: config 2 of BASELINE.json (one 16-frame window + 1 vision-condition frame, 64x64 latents, `musev` preset).
N > 1: weak scaling -- one 16-frame window per GPU (video length 16 + 12 (N-1), window 16, overlap 4), windows sharded
over the ranks, one NCCL all-reduce of the eps accumulator per DDIM step.
Prints ONE JSON line on rank 0 (contract in the task statement; extra keys: roofline, cpu_baseline, e2e, clocks).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only: no __pycache__ is written next to the sources

DDIM_STEPS = 20
WINDOW, OVERLAP = 16, 4
LAT_H = LAT_W = 64
GUIDANCE = 3.5
PRESET = "musev"
METRIC = "denoised frames/sec at 512x512, 16-frame window, 20 DDIM steps"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="musev_b200", choices=["musev_b200", "reference"])
    ap.add_argument("--preset", default=PRESET)
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--cfg-split", action="store_true",
                    help="pair the GPUs: one window per PAIR, each GPU of a pair runs one half of the CFG batch (N=2 = config 2 itself)")
    ap.add_argument("--controlnet", action="store_true", help="config-4 style: ControlNet encoder per window-step")
    ap.add_argument("--cpu-frames", type=int, default=4, help="frames of the bounded cpu_baseline sample (GPU arm)")
    ap.add_argument("--ref-frames", type=int, default=16, help="frames of one reference-arm step (16 = the config-2 window)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the denoised latents of the last timed step to DIR/latents.npy (float32); the inputs are "
                         "seeded, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "musev_b200":
        ap.error("--dump-outputs needs --impl musev_b200")
    return args


def video_frames(n_gpus: int) -> int:
    return WINDOW + (WINDOW - OVERLAP) * (n_gpus - 1)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = [float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(s) > 3 + i and s[3 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.samples)}


_ORACLE_CACHE = {}


def _oracle_forward_seconds(preset: str, frames: int, cores: int) -> float:
    from musev_b200.schema import preset_config
    from musev_b200.synth import make_inputs, make_state_dict
    from oracle.unet3d_oracle import UNet3DOracle
    torch.set_num_threads(cores)
    cfg = preset_config(preset)
    if preset not in _ORACLE_CACHE:
        _ORACLE_CACHE[preset] = UNet3DOracle(cfg, make_state_dict(cfg, seed=0))
    o = _ORACLE_CACHE[preset]
    inp = make_inputs(cfg, batch=2, frames=frames, h=LAT_H, w=LAT_W, n_vis_cond=1)
    kw = dict(sample_index=inp["sample_index"], vision_conditon_frames_sample_index=inp["vision_conditon_frames_sample_index"],
              sample_frame_rate=8)
    t0 = time.perf_counter()
    o(inp["sample"], 601, inp["encoder_hidden_states"], **kw)
    return time.perf_counter() - t0


def _frames_per_s(seconds_per_computed_frame: float) -> float:
    """Denoised frames/s of config 2 from the CPU cost of one computed frame: a window-step computes 16 + 1 frames (the
    vision-condition frame rides along) and 20 window-steps denoise 16 frames."""
    return WINDOW / ((WINDOW + 1) * seconds_per_computed_frame * DDIM_STEPS)


def cpu_baseline(preset: str, frames: int = 4, threads: int | None = None):
    """The oracle (CPU restatement of the reference, oracle/unet3d_oracle.py) timed on the host cores on a bounded sample:
    ONE window-step forward (CFG batch 2, 64x64 latents) with `frames`+1 frames instead of 16+1; the cost per computed
    frame is scaled to the 17 computed frames of the real window-step and to 20 DDIM steps.
    torch's CPU convolutions stop scaling (and regress) far below the box's 128 hardware threads -- the first measurement
    with all 128 was slower than 8 cores of the build container -- so at most 32 threads are used and `cores` says so."""
    cores = threads or min(32, os.cpu_count() or 1)
    dt = _oracle_forward_seconds(preset, frames, cores)
    return {"value": _frames_per_s(dt / (frames + 1)), "unit": "frames/s", "cores": cores, "kind": "port",
            "seconds_per_forward": dt, "sample_frames": frames + 1,
            "sample": f"1 oracle UNet3D window-step forward (fp32, B=2 CFG, {frames}+1 frames, 64x64 latents, {preset}) = {dt:.1f} s "
                      f"-> {dt / (frames + 1):.2f} s per computed frame, x17 frames per window-step, x{DDIM_STEPS} DDIM steps"}


def bench_config(preset: str, world: int, T: int, extra: dict | None = None) -> dict:
    """`config` of the JSON line; shared by both arms so that the driver sees the same workload description."""
    c = {"workload": f"config2 image2video 16-frame window 512x512, {DDIM_STEPS} DDIM steps, CFG, {preset} UNet3D"
                     + ("" if world == 1 else f"; weak scaling: {T} frames = {world} windows (16, overlap 4), 1 per GPU"),
         "preset": preset, "frames": T, "latent_hw": [LAT_H, LAT_W], "ddim_steps": DDIM_STEPS, "windows": world}
    if extra:
        c.update(extra)
    return c


def run_reference(args):
    """`--impl reference`: the reference's CPU path (the oracle port -- a Python reference cannot travel to the GPU box),
    `--warmup W` untimed + `--steps K` timed steps. One step = one bounded window-step forward of F+1 frames (F = 1 when
    K + W is large, up to 4) whose per-computed-frame cost is scaled to the real 16+1-frame window-step; ONE real
    16+1-frame forward is timed after the loop and reported next to it (`full_window_step`), so the scaling can be checked."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = min(32, os.cpu_count() or 1)
    n = args.warmup + args.steps
    probe = _oracle_forward_seconds(args.preset, 1, cores)                   # also loads the weights / warms the allocator
    frames = 1
    for f in (4, 2):
        if n * probe * (f + 1) / 2.0 <= 200.0:
            frames = f
            break
    dts = []
    for i in range(n):
        dt = _oracle_forward_seconds(args.preset, frames, cores)
        if i >= args.warmup:
            dts.append(dt)
    per_frame = (sum(dts) / len(dts)) / (frames + 1)
    v = _frames_per_s(per_frame)
    full = _oracle_forward_seconds(args.preset, WINDOW, cores)               # the real config-2 window-step, once
    cb = {"value": v, "unit": "frames/s", "cores": cores, "kind": "port", "sample_frames": frames + 1,
          "seconds_per_forward": sum(dts) / len(dts),
          "full_window_step": {"frames": WINDOW + 1, "seconds": full, "value_frames_per_s": WINDOW / (full * DDIM_STEPS)},
          "sample": f"each step = 1 oracle UNet3D window-step forward (fp32, B=2 CFG, {frames}+1 frames, 64x64, {args.preset}); "
                    f"{per_frame:.2f} s per computed frame x17 x{DDIM_STEPS}; one real 16+1-frame forward afterwards: {full:.1f} s"}
    T = video_frames(1)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * (WINDOW + 1) * per_frame * DDIM_STEPS, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(args.preset, 1, T),
        "cpu_baseline": cb,
        "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if args.gpus != 1 or world != 1:
            raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # stdout carries exactly one JSON line: anything a library prints while the bench runs (NCCL's version banner, ...)
    # is sent to stderr by pointing fd 1 at fd 2 until the result is ready
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    import torch.distributed as dist
    if world > 1:
        import datetime
        # the image exports NCCL_DEBUG=VERSION, which makes NCCL print a banner on stdout next to the one JSON line
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=240))

    from musev_b200 import _capi
    from musev_b200.flops import unet_forward_flops
    from musev_b200.pipeline import ParallelDenoiser
    from musev_b200.scheduler import SD15_DDIM_CONFIG, DDIMScheduler
    from musev_b200.schema import preset_config
    from musev_b200.synth import make_state_dict
    from musev_b200.unet import UNet3DConditionModel

    cfg = preset_config(args.preset)
    unet = UNet3DConditionModel(cfg, device=dev, dtype=torch.float16)
    sd = make_state_dict(cfg, seed=0, dtype=torch.float16)          # random-init weights of the named architecture
    unet.load_state_dict(sd)
    del sd
    sched = DDIMScheduler(**SD15_DDIM_CONFIG)
    den = ParallelDenoiser(unet, sched)
    if args.cfg_split and world % 2:
        raise SystemExit("--cfg-split needs an even number of GPUs")
    n_windows = world // 2 if args.cfg_split else world        # one window per GPU, or per GPU pair
    T = video_frames(n_windows)
    cnet_fn = None
    g = torch.Generator().manual_seed(1234)
    lat_host = torch.randn(1, 4, T, LAT_H, LAT_W, generator=g).half().pin_memory()
    cond_host = (torch.randn(1, 4, 1, LAT_H, LAT_W, generator=g) * 0.18215).half().pin_memory()
    prompt_host = torch.randn(2, 77, cfg.cross_attention_dim, generator=g).half().pin_memory()
    out_host = torch.empty(1, 4, T, LAT_H, LAT_W, dtype=torch.float16).pin_memory()
    lat, cond, prompt = lat_host.to(dev), cond_host.to(dev), prompt_host.to(dev)
    if args.controlnet:
        # config-4 style: the ControlNet encoder runs on the engine every window-step (+9.63 TFLOP per 34-frame call)
        from musev_b200.controlnet import ControlNetModel
        from musev_b200.pipeline import make_controlnet_fn
        from musev_b200.schema import ControlNetConfig
        ccfg = ControlNetConfig()
        cnet = ControlNetModel(ccfg, device=dev, dtype=torch.float16)
        cnet.load_state_dict(make_state_dict(ccfg, seed=3, dtype=torch.float16))
        cn_lat = (torch.randn(2, ccfg.block_out_channels[0], 1 + T, LAT_H, LAT_W, generator=g) * 0.3).half().to(dev)
        cnet_fn = make_controlnet_fn(cnet, cn_lat, prompt, 1)

    def one_step(latents, cond_l, prompt_e, single_window=False):
        if single_window:                       # the N = 1 workload on this rank alone (no collective): step-time reference
            return single(latents[:, :, :WINDOW].contiguous(), cond_l, prompt_e, num_inference_steps=DDIM_STEPS,
                          guidance_scale=GUIDANCE, context_frames=WINDOW, context_overlap=OVERLAP,
                          context_schedule="uniform_v2", motion_speed=8.0).latents
        return den(latents, cond_l, prompt_e, num_inference_steps=DDIM_STEPS, guidance_scale=GUIDANCE,
                   context_frames=WINDOW, context_overlap=OVERLAP, context_schedule="uniform_v2", motion_speed=8.0,
                   controlnet_fn=cnet_fn, cfg_split=args.cfg_split).latents

    single = ParallelDenoiser(unet, sched)
    single._dist, single.rank, single.world = None, 0, 1      # local: never enters a collective

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        one_step(lat, cond, prompt)
    # ---- timed region 1: inputs resident in HBM
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = _capi.launch_count(-1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        res = one_step(lat, cond, prompt)
    e1.record()
    barrier()
    launches = _capi.launch_count(-1) - l0
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    # ---- timed region 2 (e2e): host buffers, H2D of the step's inputs and D2H of its result inside the region
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for _ in range(args.steps):
        l_d = lat_host.to(dev, non_blocking=True)
        c_d = cond_host.to(dev, non_blocking=True)
        p_d = prompt_host.to(dev, non_blocking=True)
        r = one_step(l_d, c_d, p_d)
        out_host.copy_(r, non_blocking=True)
    e3.record()
    barrier()
    sampler.stop_flag = True
    ms2 = torch.tensor([e2.elapsed_time(e3)], device=dev)
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    ms2_total = float(ms2.item())
    h2d = lat_host.numel() * 2 + cond_host.numel() * 2 + prompt_host.numel() * 2
    d2h = out_host.numel() * 2

    # ---- step-time reference for the scaling record: the N = 1 workload (one 16-frame window, CFG batch 2) on this GPU
    ms_single = None
    if world > 1:
        barrier()
        one_step(lat, cond, prompt, single_window=True)
        torch.cuda.synchronize()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        one_step(lat, cond, prompt, single_window=True)
        s1.record()
        torch.cuda.synchronize()
        t_single = torch.tensor([s0.elapsed_time(s1)], device=dev)
        dist.all_reduce(t_single, op=dist.ReduceOp.MAX)
        ms_single = float(t_single.item())
    # ---- one UNet forward of each released preset at the config-2 shape (N = 1 only; CUDA events, 3 forwards)
    forward_ms = {}
    if world == 1:
        from musev_b200.synth import make_inputs

        def time_forward(model, mcfg):
            inp = make_inputs(mcfg, batch=2, frames=WINDOW, h=LAT_H, w=LAT_W, n_vis_cond=1)
            kw = dict(sample_index=inp["sample_index"], vision_conditon_frames_sample_index=inp["vision_conditon_frames_sample_index"],
                      sample_frame_rate=8)
            for k in ("down_block_refer_embs", "mid_block_refer_emb", "vision_clip_emb"):
                if k in inp:
                    kw[k] = [x.half().to(dev) for x in inp[k]] if isinstance(inp[k], list) else inp[k].half().to(dev)
            x, enc = inp["sample"].half().to(dev), inp["encoder_hidden_states"].half().to(dev)
            for _ in range(2):
                model(x, 601, enc, **kw)
            torch.cuda.synchronize()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
            for _ in range(3):
                model(x, 601, enc, **kw)
            f1.record()
            torch.cuda.synchronize()
            return f0.elapsed_time(f1) / 3
        forward_ms[args.preset] = time_forward(unet, cfg)
        other = "musev_referencenet" if args.preset == "musev" else "musev"
        try:
            ocfg = preset_config(other)
            om = UNet3DConditionModel(ocfg, device=dev, dtype=torch.float16)
            om.load_state_dict(make_state_dict(ocfg, seed=0, dtype=torch.float16))
            forward_ms[other] = time_forward(om, ocfg)
            del om
            torch.cuda.empty_cache()
        except Exception as e:   # never fail the headline on the side measurement
            forward_ms[other] = f"error: {e}"

    # ---- roofline of the dominant kernel (conv/linear tcgen05 GEMM): CUDA events around every launch of one more
    # denoise step on the launching stream (separate pass so the event records do not perturb the timed regions)
    roof = None
    # every rank runs the pass (the loop contains a collective); only rank 0 reports it
    barrier()
    _capi.profile_enable(True)
    one_step(lat, cond, prompt)
    prof = _capi.profile_collect()
    _capi.profile_enable(False)
    barrier()
    if rank == 0:
        fl = unet_forward_flops(cfg, 2, WINDOW + 1, LAT_H, LAT_W)
        n_fwd = DDIM_STEPS          # one window per rank -> one UNet forward per DDIM step
        if args.cfg_split:
            fl = unet_forward_flops(cfg, 1, WINDOW + 1, LAT_H, LAT_W)      # each rank runs one half of the CFG batch
        gemm_ms, gemm_n = prof["gemm"]["ms"], prof["gemm"]["launches"]
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = peaks.get("bf16_tflops_sustained", 1400.0)
        achieved = fl["gemm"] * n_fwd / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else None
        # DRAM bytes per launch of this kernel from the committed ncu capture of one forward (same shapes as here)
        traffic, traffic_src = None, None
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "r01_gemm_dram_traffic.json")))
            traffic, traffic_src = tr["dram_bytes_per_launch"], "profiles/r01_gemm_dram_traffic.json (ncu dram__bytes_read+write, mean over the 440 GEMM launches of a forward; algorithmic %.0f MB/launch)" % (tr["algorithmic_bytes_per_launch"] / 1e6)
        except Exception:
            pass
        roof = {"kernel": "conv_gemm_kernel (tcgen05 implicit-GEMM conv / linear)", "bound": "tensor",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak if achieved else None,
                "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback 1.4 PFLOP/s sustained",
                "traffic": traffic, "traffic_unit": "bytes/launch", "traffic_source": traffic_src, "launches_per_step": gemm_n, "avg_launch_ms": gemm_ms / max(gemm_n, 1),
                "algorithmic_tflop_per_forward": fl["gemm"] / 1e12,
                "step_share": {k: round(v["ms"], 2) for k, v in prof.items()}}

    if args.dump_outputs and rank == 0:
        # `res` is what the last step of timed region 1 returned; the latents are replicated on every rank
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "latents.npy"), res.float().cpu().numpy())

    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    os.close(saved_stdout)
    if rank == 0:
        frames = T * args.steps
        value = frames / (ms_total * 1e-3)
        e2e = frames / (ms2_total * 1e-3)
        cb = None
        if world == 1 and not args.skip_cpu_baseline:
            try:
                cb = cpu_baseline(args.preset)
            except Exception as e:  # reported baseline only; never fail the GPU number on it
                cb = {"error": str(e)}
        fl_total = unet_forward_flops(cfg, 2, WINDOW + 1, LAT_H, LAT_W)["total"]
        extra = {"parallelism": (f"windows sharded over {world} GPU(s), 1 NCCL all-reduce/step" if not args.cfg_split else
                                 f"CFG split: {n_windows} window(s) over {world} GPUs, each GPU of a pair runs one half of the CFG batch, 1 NCCL all-reduce/step"),
                 "l2_policy": "per-forward activation working set (~4 GB) >> 126 MB L2; no explicit flush",
                 "achieved_tflops_whole_step": fl_total * DDIM_STEPS * args.steps * n_windows / (ms_total * 1e-3) / 1e12,
                 # what bounds the weak-scaling curve: each added window brings 12 new frames for 17 computed ones
                 "ideal_efficiency": T / (WINDOW * world),
                 "step_time_efficiency": (ms_single / (ms_total / args.steps)) if ms_single else 1.0,
                 "single_window_ms_per_step": ms_single}
        if forward_ms:
            extra["unet_forward_ms"] = forward_ms
        if args.controlnet:
            extra["controlnet"] = "SD-1.5 ControlNet encoder on the engine every window-step (config-4 style)"
        conf = bench_config(args.preset, n_windows, T, extra)
        if args.cfg_split:
            conf["workload"] = (f"config2 image2video 16-frame window 512x512, {DDIM_STEPS} DDIM steps, CFG, {args.preset} UNet3D; "
                                f"CFG split over {world} GPUs: {T} frames = {n_windows} window(s)")
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "strong" if args.cfg_split else "weak",
            "vs_baseline": None, "dtype": "f16 (fp32 accumulate)", "data": "synthetic",
            "config": conf,
            "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches),
            "clocks": sampler.summary(),
            "roofline": roof,
            "cpu_baseline": cb,
        }), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
