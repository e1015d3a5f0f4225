#!/usr/bin/env python
"""Device time of the 6-view VAE encode (AutoencoderKL(with_encoder=True).encode_latents: one CUDA-graph replay) at 224x400
and 424x800, its TFLOP/s from the shape-derived FLOP count below, and the reference's own AutoencoderKL.encode in bf16
(diffusers' AttnProcessor2_0 = torch SDPA) on the same GPU when the oracle/_ref snapshot (or the reference tree) is present.
Prints one JSON line with the GPU name and power limit read in the same run.

    python tools/bench_vae_encode.py [--repeats 20] [--warmup 3]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
from dataclasses import asdict

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from magicdrive_b200 import arch  # noqa: E402
from magicdrive_b200.models import AutoencoderKL  # noqa: E402

VIEWS = 6
SIZES = [(224, 400), (424, 800)]


def encode_flops(cfg: arch.VaeConfig, h: int, w: int) -> float:
    """Multiply-adds x 2 of AutoencoderKL.encode for one image, from the layer shapes (GroupNorm / SiLU / softmax not counted)."""
    conv = lambda pix, ci, co, k: 2.0 * pix * co * ci * k * k
    f = conv(h * w, cfg.in_channels, cfg.block_out_channels[0], 3)
    for _, resnets, down in arch.vae_encoder_blocks(cfg):
        for _, ci, co in resnets:
            f += conv(h * w, ci, co, 3) + conv(h * w, co, co, 3) + (conv(h * w, ci, co, 1) if ci != co else 0.0)
        if down:
            h, w = (h - 2) // 2 + 1, (w - 2) // 2 + 1
            f += conv(h * w, resnets[-1][2], resnets[-1][2], 3)
    c, L = cfg.block_out_channels[-1], h * w
    f += 2 * 2 * conv(L, c, c, 3)                  # the mid block's two resnets
    f += 4 * conv(L, c, c, 1) + 2 * 2.0 * L * L * c  # q, k, v, out projections; QK^T and PV
    m = 2 * cfg.latent_channels
    return f + conv(L, c, m, 3) + conv(L, m, m, 1)  # conv_out, quant_conv


def time_ms(fn, warmup: int, repeats: int) -> float:
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts)


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out or "unknown"


def reference_encoder(cfg, sd):
    from oracle import ref_shim
    if not ref_shim.available():
        return None
    R = ref_shim.load()
    vae = R.AutoencoderKL(block_out_channels=list(cfg.block_out_channels), down_block_types=list(cfg.down_block_types),
                          up_block_types=list(cfg.up_block_types), latent_channels=cfg.latent_channels,
                          layers_per_block=cfg.layers_per_block)
    vae.load_state_dict(sd, strict=True)
    return vae.to("cuda", torch.bfloat16).eval()


@torch.no_grad()
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_vae_encode.py measures on a CUDA device; none is available")
    cfg = arch.VaeConfig()
    shapes = dict(arch.vae_encoder_param_shapes(cfg), **arch.vae_decoder_param_shapes(cfg))
    sd = arch.synthetic_state_dict(shapes, 15)
    vae = AutoencoderKL(**asdict(cfg), with_encoder=True)
    vae.load_state_dict(sd)
    vae = vae.to("cuda", torch.bfloat16)
    ref = reference_encoder(cfg, sd)
    name, power = gpu_info()
    res = dict(tool="bench_vae_encode", gpu=name, power_limit=power, views=VIEWS, dtype="bf16",
               timing=f"CUDA events, median of {args.repeats} after {args.warmup} warm-up calls")
    for h, w in SIZES:
        x = (torch.rand(1, VIEWS, 3, h, w, generator=torch.Generator().manual_seed(h)) * 2 - 1).to("cuda")
        flops = VIEWS * encode_flops(cfg, h, w)
        ms = time_ms(lambda: vae.encode_latents(x), args.warmup, args.repeats)
        row = dict(gflop=round(flops / 1e9, 1), ours_ms=round(ms, 3), ours_tflops=round(flops / ms / 1e9, 1))
        if ref is not None:
            xr = x[0].to(torch.bfloat16)
            sf = cfg.scaling_factor
            rms = time_ms(lambda: ref.encode(xr).latent_dist.mean * sf, args.warmup, args.repeats)
            ours, theirs = vae.encode_latents(x)[0].float(), (ref.encode(xr).latent_dist.mean * sf).float()
            row.update(reference_ms=round(rms, 3), reference_tflops=round(flops / rms / 1e9, 1),
                       speedup_vs_reference=round(rms / ms, 2),
                       rel_l2_vs_reference=float((ours - theirs).norm() / theirs.norm()))
        res[f"{h}x{w}"] = row
        del x
        torch.cuda.empty_cache()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
