#!/usr/bin/env python
"""Benchmark of the multi-view denoising hot path (BASELINE.json: "6-view 224x400 denoising-steps/sec").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload full|cam] [--scenes S]
                  [--dump-outputs DIR]

One "step" = ControlNet forward + multi-view UNet forward + classifier-free-guidance combine + DDIM update for S
six-view scenes per GPU (CFG on: 12 view-samples per scene-step, the reference default guidance_scale = 2).
Default workload = BASELINE.json configs[2] (full conditioning: 20 boxes/view + BEV map + text), the configuration
BASELINE.md section 2's 4.75 TFLOP/scene-step is quoted on; `--workload cam` = configs[1].
N > 1 (torchrun, one process per GPU): scenes are sharded across ranks, no data-path collective ("weak" scaling);
time = max over ranks of the device-timed loop, value = all scene-steps / time.
`--impl reference` times the UNMODIFIED reference (its own pipeline __call__, loaded from the oracle/_ref snapshot through
oracle/ref_shim.py) on the host CPU cores in fp32, rank 0 only.  The default arm also reports `cpu_baseline` (same thing,
1 step) and `gpu_reference`: the same reference modules in bf16 on the same GPU (torch SDPA attention).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TFLOP_PER_SCENE_STEP_CFG = {"224x400": 4.75, "424x800": 24.0}  # BASELINE.md section 2 (algorithmic, CFG on, ctx 1+77+20)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30, help="timed denoising steps (>= 1)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="full", choices=["cam", "full"],
                    help="full = configs[2] (20 boxes/view + BEV map + text, default); cam = configs[1] (text + camera only)")
    ap.add_argument("--scenes", type=int, default=1, help="six-view scenes per GPU")
    ap.add_argument("--res", default="224x400", choices=["224x400", "424x800"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-reference", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-overlap", action="store_true", help="run ControlNet and UNet encoder on one stream")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--scheduler", default="ddim", choices=["ddim", "unipc"],
                    help="sampler fused into the step: ddim (BASELINE.json configs: 50-step DDIM) or unipc (the reference's default)")
    ap.add_argument("--cfg-streams", action="store_true",
                    help="opt-in: run the unconditional / conditional guidance halves as two concurrent graph branches")
    ap.add_argument("--no-hires", action="store_true", help="skip the configs[3] (424x800) sub-record of the default run")
    ap.add_argument("--no-decode", action="store_true",
                    help="skip timing the VAE decode of the scene's 6 views (SURVEY.md section 8 f2, reported as vae_decode)")
    ap.add_argument("--shard", default="scenes", choices=["scenes", "views"],
                    help="N>1: scenes = independent scenes per GPU (default, weak scaling, no data-path collective); "
                         "views = the 6 cameras of the SAME scenes split across GPUs with an exchange of the "
                         "cross-view K/V per multiview block (strong scaling, latency mode)")
    ap.add_argument("--strong-scaling", action="store_true",
                    help="N>1, default sharding: after the replica measurement also time ONE scene spread over all N GPUs "
                         "(guidance halves x views through NVLink peer memory) and report it as `strong_scaling`")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed loop's last step returned (the scene latents, float32) as DIR/<name>.npy, "
                         "at most 64 MB in all, so that two builds can be compared output for output on identical inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(dirname, arrays):
    """Write each tensor of `arrays` as <dirname>/<name>.npy in float32.  When they exceed DUMP_LIMIT_BYTES in all, each is
    replaced by the same share of its elements at positions drawn from a fixed seed, so that every run writes the same ones."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    total = sum(a.numel() for a in arrays.values()) * 4
    for name, a in arrays.items():
        a = a.detach().float().cpu()
        if total > DUMP_LIMIT_BYTES:
            flat = a.reshape(-1)
            keep = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:flat.numel() * DUMP_LIMIT_BYTES // total]
            a = flat[keep.sort().values]
        np.save(os.path.join(dirname, name + ".npy"), a.numpy())


def make_inputs(args, rank):
    from magicdrive_b200.synthetic import synthetic_inputs  # seeded input generator (no model arithmetic)
    h, w = (28, 50) if args.res == "224x400" else (53, 100)
    mhw = 200 if args.res == "224x400" else 400
    inp = synthetic_inputs(args.scenes, 6, h, w, n_box=20 if args.workload == "full" else 0, map_hw=mhw,
                           seed=args.seed + 1000 * rank)
    if args.workload == "cam":
        inp["bev_map"] = torch.zeros_like(inp["bev_map"])  # configs[1]: no map / no boxes; the ControlNet still runs
    return inp, h, w


def workload_config(args, sharding):
    """Identical for both arms (the driver compares the `config` objects of the two lines)."""
    return {"workload": f"configs[{1 if args.workload == 'cam' else 2}]: 6-view {args.res}, "
                        + ("text+camera-pose cond" if args.workload == "cam" else "full cond (20 boxes/view + BEV map + text)")
                        + ", CFG 2.0 (12 view-samples per scene-step), DDIM eta=0, SD-1.5-config UNet + BEVControlNet, random-init weights",
            "scenes_per_gpu": args.scenes, "views": 6, "latent_hw": [28, 50] if args.res == "224x400" else [53, 100],
            "sharding": sharding, "scheduler": args.scheduler,
            "l2": "2.6 GB of weights are streamed every step (>> 126 MB L2), no explicit flush needed"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def calibrate_cpu_threads():
    """All host threads the arithmetic can actually use: torch's CPU conv / GEMM stop scaling (and regress) well before
    128 threads on this workload, so the thread count is calibrated on a representative 3x3 convolution first."""
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (ncpu, ncpu // 2, ncpu // 4, 32, 16, 8) if 1 <= c <= ncpu}, reverse=True)
    xcal, wcal = torch.randn(12, 320, 28, 50), torch.randn(320, 320, 3, 3)
    best_t, best_c = None, ncpu
    for c in cands:
        torch.set_num_threads(c)
        torch.nn.functional.conv2d(xcal, wcal, padding=1)
        t0 = time.perf_counter()
        for _ in range(2):
            torch.nn.functional.conv2d(xcal, wcal, padding=1)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best_t, best_c = dt, c
    torch.set_num_threads(best_c)
    return best_c


class ReferenceArm:
    """The reference's own implementation of the path on this workload (oracle/ref_runner.py: the unmodified
    StableDiffusionBEVControlNetPipeline.__call__ with its own networks), or — if neither /root/reference nor the
    oracle/_ref snapshot exists — the oracle port (oracle/torch_oracle.py).  Measurement code only."""

    def __init__(self, args):
        from oracle import ref_runner
        self.args = args
        self.kind = "reference" if ref_runner.available() else "port"
        self.pipe = None
        self.inp, self.h, self.w = make_inputs(args, 0)

    def _pipe(self):
        if self.pipe is None:
            from oracle import ref_runner
            self.pipe = ref_runner.build_pipeline(self.args.res, "cpu", torch.float32)
        return self.pipe

    def cpu(self, steps, warmup):
        """(scene-steps/s, seconds/step, threads) on the host cores, fp32."""
        cores = calibrate_cpu_threads()
        if self.kind == "reference":
            from oracle import ref_runner
            sec, _ = ref_runner.time_steps(self._pipe(), self.inp, self.h, self.w, steps, max(warmup, 1), "cpu", torch.float32)
        else:
            sec = self._port_cpu(steps, warmup)
        return self.args.scenes / sec, sec, cores

    def gpu(self, device, steps, warmup):
        """The same reference modules in bf16 on `device` (diffusers AttnProcessor2_0 -> torch SDPA)."""
        if self.kind != "reference":
            return None
        from oracle import ref_runner
        pipe = self._pipe().to(device, torch.bfloat16)
        sec, _ = ref_runner.time_steps(pipe, self.inp, self.h, self.w, steps, warmup, device, torch.bfloat16)
        self.pipe = None  # the pipeline now lives on the GPU in bf16; drop it
        del pipe
        torch.cuda.empty_cache()
        return sec

    def _port_cpu(self, steps, warmup):
        from magicdrive_b200 import arch
        from oracle import torch_oracle as O
        args, inp = self.args, self.inp
        ucfg, ccfg = arch.UNetConfig(), arch.ControlNetConfig(map_size=(8, 200, 200) if args.res == "224x400" else (8, 400, 400))
        usd = arch.synthetic_state_dict(arch.unet_param_shapes(ucfg), 11)
        csd = arch.synthetic_state_dict(arch.controlnet_param_shapes(ccfg), 12)
        sched = O.DDIM()
        ts = sched.set_timesteps(50).tolist()
        cam, boxes = O.add_uncond_to_kwargs(csd, ccfg, inp["camera_param"], inp["bboxes_3d_data"])
        text = torch.cat([inp["negative_prompt_embeds"], inp["prompt_embeds"]])
        image = torch.cat([inp["bev_map"]] * 2)
        lat = torch.stack([inp["latents"]] * 6, 1)
        times = []
        with torch.no_grad():
            for i in range(warmup + steps):
                t = ts[i % len(ts)]
                t0 = time.perf_counter()
                x2 = torch.cat([lat] * 2)
                tt = torch.full((x2.shape[0],), t, dtype=torch.int64)
                down, mid, ctx = O.controlnet_forward(csd, ccfg, x2, tt, cam, boxes, text, image)
                eps = O.unet_forward(usd, ucfg, x2.reshape(-1, *x2.shape[2:]), torch.tensor(t), ctx, down, mid)
                eu, ec = eps.chunk(2)
                eps = eu + 2.0 * (ec - eu)
                lat = sched.step(eps, t, lat.reshape(-1, *lat.shape[2:])).reshape(lat.shape)
                if i >= warmup:
                    times.append(time.perf_counter() - t0)
        return sum(times) / len(times)


def context_delta_tflop(args, n_box_tokens):
    """FLOPs that `n_box_tokens` extra conditioning tokens add to one CFG scene-step (attn2 QK^T + PV, and the hoisted
    K/V projections), for the SD-1.5 layer sheet (SURVEY.md Appendix A): used to state the cam workload's algorithmic
    work relative to BASELINE.md's full-cond figure."""
    h, w = (28, 50) if args.res == "224x400" else (53, 100)
    sizes = []
    hh, ww = h, w
    for c in (320, 640, 1280):
        sizes.append((hh * ww, c))
        hh, ww = (hh - 1) // 2 + 1, (ww - 1) // 2 + 1
    mid = (hh * ww, 1280)
    # transformer layers: UNet down 2+2+2, mid 1, up 3+3+3; ControlNet down 2+2+2, mid 1
    layers = [sizes[0]] * (2 + 3 + 2) + [sizes[1]] * (2 + 3 + 2) + [sizes[2]] * (2 + 3 + 2) + [mid] * 2
    V = 12 * args.scenes
    core = sum(4.0 * V * L * n_box_tokens * c for L, c in layers)
    kv = sum(2.0 * 2.0 * V * n_box_tokens * 768 * c for _, c in layers)
    return core / 1e12, kv / 1e12


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n_gpus = max(args.gpus, world)
    by_views = args.shard == "views" and world > 1
    sharding = (f"one scene over {world} GPUs: guidance halves x camera views; neighbour K/V and the partner half's noise read in "
                "place through NVLink peer memory (no NCCL on the data path)" if by_views else "scene-per-GPU replicas, no data-path collective")
    config = workload_config(args, sharding)
    metric = "6-view 224x400 denoising-steps/sec" if args.res == "224x400" else "6-view 424x800 denoising-steps/sec"

    if args.impl == "reference":
        if rank != 0:
            return 0
        steps, warm = min(args.steps, 3), max(1, min(args.warmup, 1))
        arm = ReferenceArm(args)
        val, sec, cores = arm.cpu(steps, warm)
        what = ("the unmodified reference pipeline __call__ (oracle/_ref snapshot)" if arm.kind == "reference"
                else "the oracle port of the reference arithmetic")
        sample = f"{steps} full scene-steps (CFG, V=12) after {warm} warm-up, fp32, torch CPU kernels, {what}"
        line = {"impl": "reference", "metric": metric, "value": val, "unit": "scene-steps/s",
                "n_gpus": n_gpus, "steps": steps, "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": val, "unit": "scene-steps/s", "cores": cores, "kind": arm.kind, "sample": sample},
                "e2e": {"value": val, "unit": "scene-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ our arm (CUDA)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from dataclasses import asdict

    from magicdrive_b200 import arch, ops
    from magicdrive_b200.models import BEVControlNetModel, UNet2DConditionModelMultiview
    from magicdrive_b200.pipeline import BEVControlNetDenoiser

    ucfg = arch.UNetConfig()
    ccfg = arch.ControlNetConfig(map_size=(8, 200, 200) if args.res == "224x400" else (8, 400, 400))
    un = UNet2DConditionModelMultiview(**asdict(ucfg)).reset_parameters_synthetic(11).to(dev, torch.bfloat16)
    cn = BEVControlNetModel(**asdict(ccfg)).reset_parameters_synthetic(12).to(dev, torch.bfloat16)
    shard = None
    if by_views:
        from magicdrive_b200.dist import ShardContext
        shard = ShardContext(6, True, [ucfg.neighboring_view_pair[i] for i in range(6)], dev)
    pipe = BEVControlNetDenoiser(un, cn, use_cuda_graph=not args.no_graph, overlap_controlnet=not args.no_overlap,
                                 view_shard=shard, scheduler=args.scheduler, cfg_streams=args.cfg_streams)
    inp, h, w = make_inputs(args, 0 if by_views else rank)
    job_scenes = args.scenes if by_views else n_gpus * args.scenes  # scenes the whole job advances per step
    views_local = shard.plan.n_local * (0.5 if shard.plan.split_cfg else 1.0) if by_views else 6  # view-samples share of this rank
    boxes = inp["bboxes_3d_data"]
    host = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in inp.items()}
    if boxes is not None:
        host["bboxes_3d_data"] = {k: v.pin_memory() for k, v in boxes.items()}

    def prepare():
        return pipe.prepare(host["latents"], host["prompt_embeds"], host["negative_prompt_embeds"], host["camera_param"],
                            host["bboxes_3d_data"], host["bev_map"], guidance_scale=2.0)

    st = prepare()
    pipe.set_schedule(st, 50)
    sched_len = 50

    def run(i):
        pipe.run_steps(st, i % sched_len, i % sched_len + 1)

    ops.reset_launch_count()
    run(0)  # eager (sizes workspaces) + graph capture + first replay
    for i in range(1, args.warmup):
        run(i)
    # kernels of one step, counted on an eager pass (the graph replays the same kernel nodes)
    was = pipe.use_cuda_graph
    pipe.use_cuda_graph = False
    ops.reset_launch_count()
    run(args.warmup)
    launches_per_step = ops.launch_count()
    pipe.use_cuda_graph = was
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- timed region (device-timed, CUDA events on the launching stream)
    sampler = ClockSampler(local_rank)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.start()
    e0.record()
    for i in range(args.steps):
        run(args.warmup + 1 + i)
    e1.record()
    barrier()
    clocks = sampler.stop()
    ms_total = e0.elapsed_time(e1)
    # the latents a caller of the timed path receives after its last step; the sections below reuse and overwrite `st`
    dumped = {"latents": pipe.latents_out(st)} if args.dump_outputs else None
    if world > 1:
        tt = torch.tensor([ms_total], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_total = tt.item()
    ms_step = ms_total / args.steps
    value = job_scenes / (ms_step * 1e-3)

    # ---- end-to-end through the host-facing call.  A denoising step's inputs are (x_t, t): every timed step copies
    #      the scene's latents from pinned host memory to the device, runs the step (graph replay) and reads x_{t-1}
    #      back to the host.  The conditioning is a per-call constant staged before the loop (exactly as the reference
    #      pipeline moves it once, pipeline_bev_controlnet.py:329,343); the cost of re-staging + re-encoding it on
    #      EVERY step is reported separately as e2e_full_reencode.
    n_loc = shard.plan.n_local if by_views else 6
    lat_host = torch.stack([host["latents"]] * n_loc, 1).permute(0, 1, 3, 4, 2).contiguous().view(-1, 4).pin_memory()
    out_host = torch.empty_like(lat_host).pin_memory()
    h2d = lat_host.numel() * 4 + 4 * st["V"]
    d2h = out_host.numel() * 4
    barrier()
    e0.record()
    for i in range(args.steps):
        st["latents"].copy_(lat_host, non_blocking=True)
        run(i)
        out_host.copy_(st["latents"], non_blocking=True)
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1)
    full_h2d = sum(v.numel() * v.element_size() for v in [host["latents"], host["prompt_embeds"], host["negative_prompt_embeds"],
                                                          host["camera_param"], host["bev_map"]])
    if boxes is not None:
        full_h2d += sum(v.numel() * v.element_size() for v in host["bboxes_3d_data"].values())
    for i in range(2):
        s2 = prepare()
        pipe.run_steps(s2, i, i + 1)
    barrier()
    e0.record()
    nfull = max(3, args.steps // 4)
    for i in range(nfull):
        s2 = prepare()
        pipe.run_steps(s2, i % sched_len, i % sched_len + 1)
        out_host.copy_(s2["latents"], non_blocking=True)
    e1.record()
    barrier()
    ms_full = e0.elapsed_time(e1) / nfull
    if world > 1:
        tt = torch.tensor([ms_e2e, ms_full], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_e2e, ms_full = tt[0].item(), tt[1].item()
    e2e_value = job_scenes / (ms_e2e / args.steps * 1e-3)

    # ---- roofline of the dominant kernel (tcgen05 GEMM / implicit-GEMM conv): per-launch CUDA events, eager pass
    pipe.use_cuda_graph = False
    overlap_was, pipe.overlap_controlnet = pipe.overlap_controlnet, False  # serial launches: per-kernel times are not inflated by co-running kernels
    st = prepare()
    pipe.set_schedule(st, 50)
    run(0)
    torch.cuda.synchronize()
    # park the stream behind a ~25 ms spin so the whole step (launches + event records) is enqueued before the GPU
    # starts it: the per-launch events then bracket back-to-back device execution, not host enqueue latency
    torch.cuda._sleep(int(50e6))
    ops.start_profile()
    run(1)
    prof = ops.stop_profile()
    pipe.use_cuda_graph = was
    pipe.overlap_controlnet = overlap_was
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    # burst peak when the sampled clocks were un-capped (no power cap, SM clock at max): that is the regime the cuBLAS
    # burst figure was taken in; the sustained figure otherwise
    capped = ("sw_power_cap" in (clocks.get("reasons") or [])) or not clocks.get("sm_mhz") or \
        clocks["sm_mhz"] < 0.95 * (clocks.get("sm_max_mhz") or 1e9)
    if peaks:
        key = "bf16_tflops_sustained" if capped else "bf16_tflops"
        peak_tf = peaks.get(key) or peaks.get("bf16_tflops_sustained") or 1400.0
        peak_src = f"MEASURED_PEAKS.json {key} (of measured; clocks during the timed region {'capped' if capped else 'un-capped at max'})"
    else:
        peak_tf = 1400.0 if capped else 1590.0
        peak_src = "fallback " + ("1.4 PF/s sustained" if capped else "1.59 PF/s burst") + " (of fallback)"
    g = [(f, s) for k, f, s in prof if k == "gemm_conv"]
    a = [(f, s) for k, f, s in prof if k == "attention"]
    gf, gs = sum(f for f, _ in g), sum(s for _, s in g)
    af, as_ = sum(f for f, _ in a), sum(s for _, s in a)
    achieved = gf / gs / 1e12 if gs > 0 else 0.0
    traffic, traffic_src = None, None
    try:  # per-launch DRAM bytes of the dominant kernel from this round's committed ncu capture, if one exists
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic_r2.json")))
        traffic, traffic_src = tj["dram_bytes_per_launch"], "profiles/traffic_r2.json (ncu dram__bytes_read+write per launch, committed capture)"
    except Exception:
        pass
    scale = args.scenes * views_local / 6
    alg_full = TFLOP_PER_SCENE_STEP_CFG[args.res] * scale
    d_core, d_kv = context_delta_tflop(args, 20)
    alg = alg_full if args.workload == "full" else alg_full - (d_core + d_kv) * views_local / 6
    _, kv_all = context_delta_tflop(args, 98 if args.workload == "full" else 78)
    hoisted = kv_all * views_local / 6
    roofline = {"bound": "tensor", "kernel": "gemm_pair_kernel / gemm_tc2_kernel (tcgen05 GEMM / implicit-GEMM conv, all shapes of one step)",
                "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf, "peak_source": peak_src,
                "launches": len(g), "flops_per_step": gf, "kernel_ms_per_step": gs * 1e3, "traffic": traffic,
                "traffic_source": traffic_src,
                "timing_note": "per-launch CUDA events on an eager pass queued behind a spin kernel (no host enqueue gaps); "
                               "profiles/ has the ncu device times per shape",
                "attention": {"achieved": (af / as_ / 1e12 if as_ > 0 else 0.0), "launches": len(a),
                              "kernel_ms_per_step": as_ * 1e3, "flops_per_step": af},
                "whole_step": {"algorithmic_tflop": alg, "hoisted_tflop": hoisted, "executed_tensor_tflop": (gf + af) / 1e12,
                               "achieved": alg / (ms_step * 1e-3), "frac": alg / (ms_step * 1e-3) / peak_tf,
                               "note": "per GPU; algorithmic = BASELINE.md section 2 for this workload (context tokens accounted); "
                                       "hoisted = attn2 K/V projections, part of the algorithmic figure but computed once per "
                                       "call instead of every step; executed = tensor-core FLOPs the step actually launches"}}

    # ---- BASELINE.json configs[3]: the same networks at 424x800 (53x100 latents, 400x400 BEV map), a sub-record of the default line
    hires = None
    if args.res == "224x400" and not args.no_hires and not by_views and n_gpus == 1:
        import copy
        a3 = copy.copy(args)
        a3.res = "424x800"
        inp3, h3, w3 = make_inputs(a3, rank)
        pipe.release_graph()
        pipe3 = BEVControlNetDenoiser(un, cn, use_cuda_graph=not args.no_graph, overlap_controlnet=not args.no_overlap,
                                      scheduler=args.scheduler)
        st3 = pipe3.prepare(inp3["latents"], inp3["prompt_embeds"], inp3["negative_prompt_embeds"], inp3["camera_param"],
                            inp3["bboxes_3d_data"], inp3["bev_map"], guidance_scale=2.0)
        pipe3.set_schedule(st3, 50)
        for i in range(3):
            pipe3.run_steps(st3, i, i + 1)
        barrier()
        e0.record()
        n3 = 8
        for i in range(n3):
            pipe3.run_steps(st3, 3 + i, 4 + i)
        e1.record()
        barrier()
        ms3 = e0.elapsed_time(e1) / n3
        hires = {"workload": workload_config(a3, sharding)["workload"].replace("configs[2]", "configs[3]"), "latent_hw": [h3, w3],
                 "ms_per_step": ms3, "value": args.scenes / (ms3 * 1e-3), "unit": "scene-steps/s", "steps": n3, "warmup": 3,
                 "whole_step_tflops": TFLOP_PER_SCENE_STEP_CFG["424x800"] * args.scenes / (ms3 * 1e-3)}
        pipe3.release_graph()
        del pipe3, st3
        torch.cuda.empty_cache()

    vae_decode = None
    if not args.no_decode and not by_views and world == 1:  # a sub-record of the single-GPU line only
        from magicdrive_b200.models import AutoencoderKL
        vae = AutoencoderKL(**asdict(arch.VaeConfig())).reset_parameters_synthetic(13).to(dev, torch.bfloat16)
        lat5 = pipe.latents_out(st) * 0.18215
        for _ in range(3):
            vae.decode_latents(lat5)
        barrier()
        e0.record()
        for _ in range(5):
            vae.decode_latents(lat5)
        e1.record()
        barrier()
        vae_decode = {"ms_per_scene": e0.elapsed_time(e1) / 5 / args.scenes, "views": 6,
                      "note": "AutoencoderKL.decode_latents of the 6 views at full resolution (one CUDA-graph replay per call, latents "
                              "in / images out on the device), SD-1.5 VAE config, random-init weights; not part of `value`"}
        del vae
        torch.cuda.empty_cache()

    strong = None
    if world > 1 and not by_views and (args.strong_scaling or os.environ.get("MDB_BENCH_STRONG") == "1"):
        # the same scene on all N GPUs: latency mode (SURVEY.md section 8e); every rank runs its share, time = max over ranks
        from magicdrive_b200.dist import ShardContext
        ctx = ShardContext(6, True, [ucfg.neighboring_view_pair[i] for i in range(6)], dev)
        pipe.release_graph()
        pipe2 = BEVControlNetDenoiser(un, cn, use_cuda_graph=not args.no_graph, overlap_controlnet=not args.no_overlap,
                                      view_shard=ctx, scheduler=args.scheduler)
        inp0, _, _ = make_inputs(args, 0)
        st2 = pipe2.prepare(inp0["latents"], inp0["prompt_embeds"], inp0["negative_prompt_embeds"], inp0["camera_param"],
                            inp0["bboxes_3d_data"], inp0["bev_map"], guidance_scale=2.0)
        pipe2.set_schedule(st2, 50)
        for i in range(max(3, args.warmup)):
            pipe2.run_steps(st2, i, i + 1)
        barrier()
        e0.record()
        for i in range(args.steps):
            pipe2.run_steps(st2, (3 + i) % 50, (3 + i) % 50 + 1)
        e1.record()
        barrier()
        pipe2.check_peers()
        tt = torch.tensor([e0.elapsed_time(e1) / args.steps], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        strong = {"ms_per_step": tt.item(), "scenes": args.scenes, "value": args.scenes / (tt.item() * 1e-3), "unit": "scene-steps/s",
                  "speedup_vs_one_gpu_step": ms_step / tt.item(),
                  "layout": f"guidance halves x camera views over {world} GPUs: this rank half {ctx.plan.half}, views {list(ctx.plan.views)}",
                  "note": "one scene's 12 guidance x view samples spread over all GPUs; neighbour K/V and the partner half's noise "
                          "through NVLink peer memory (mdb_attention_multi / mdb_peer_barrier), no NCCL on the data path; "
                          "speed-up is against this run's own one-scene-per-GPU step time"}
        un.set_view_shard(None)
        pipe2.release_graph()
        pipe = pipe2  # torn down below

    if rank == 0:
        cpu, gpu_ref = None, None
        if n_gpus == 1 and not (args.no_cpu_baseline and args.no_gpu_reference):
            arm = ReferenceArm(args)
            if not args.no_cpu_baseline:
                v, sec, cores = arm.cpu(1, 1)
                cpu = {"value": v, "unit": "scene-steps/s", "cores": cores, "kind": arm.kind,
                       "sample": "1 full scene-step (CFG, V=12, ControlNet+UNet) after 1 warm-up, fp32, torch CPU kernels, "
                                 + ("unmodified reference pipeline __call__" if arm.kind == "reference" else "oracle port")}
            if not args.no_gpu_reference:
                sec = arm.gpu(dev, 20, 3)
                if sec is not None:
                    gpu_ref = {"value": args.scenes / sec, "unit": "scene-steps/s", "ms_per_step": sec * 1e3, "steps": 20, "warmup": 3,
                               "dtype": "bf16", "speedup_of_value": value / (args.scenes / sec),
                               "note": "the unmodified reference pipeline (its own UNet2DConditionModelMultiview + BEVControlNetModel, "
                                       "oracle/_ref snapshot) on this GPU, CFG on, eager launches, attention = diffusers AttnProcessor2_0 "
                                       "(torch SDPA; the vendored xformers has no sm_100 kernel), wall-clock between synchronised step callbacks"}
        line = {"metric": metric, "value": value, "unit": "scene-steps/s", "n_gpus": n_gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "strong" if by_views else "weak", "vs_baseline": None, "dtype": "bf16",
                "data": "synthetic", "config": config, "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": "scene-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": ms_e2e / args.steps,
                        "note": "per step: latents (pinned host) -> device, 1 denoising step through the denoiser, latents -> host; "
                                "conditioning staged once per call like the reference pipeline"},
                "e2e_full_reencode": {"value": job_scenes / (ms_full * 1e-3), "unit": "scene-steps/s",
                                      "ms_per_step": ms_full, "h2d_bytes_per_step": full_h2d, "d2h_bytes_per_step": d2h,
                                      "note": "every step also re-stages ALL conditioning inputs from the host and re-runs "
                                              "the camera/box/map encoders and the 23 context K/V projections"},
                "gpu_launches": launches_per_step * args.steps, "gpu_launches_per_step": launches_per_step,
                "roofline": roofline, "cpu_baseline": cpu, "gpu_reference": gpu_ref,
                "options": {"cuda_graph": not args.no_graph, "two_stream_overlap": not args.no_overlap,
                            "cfg_streams": bool(args.cfg_streams)}}
        if hires is not None:
            line["configs3_424x800"] = hires
        if vae_decode is not None:
            line["vae_decode"] = vae_decode
        if strong is not None:
            line["strong_scaling"] = strong
        print(json.dumps(line))
        if dumped is not None:
            dump_outputs(args.dump_outputs, dumped)
    if world > 1:
        from magicdrive_b200.dist import shutdown
        sys.stdout.flush()
        shutdown([pipe])
    return 0


if __name__ == "__main__":
    sys.exit(main())
