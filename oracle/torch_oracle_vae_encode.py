"""TEST INFRASTRUCTURE ONLY — plain-torch fp32 restatement of the reference's AutoencoderKL.encode, beside
oracle/torch_oracle.py (whose resnet block and conv helpers it uses).  Pinned to the reference's own output by
tests/golden/vae_encode_80x104.pt (oracle/make_golden_vae_encode.py, checked in tests/test_vae_encode_cpu.py).
Activations are NCHW like the reference; weights are taken by their checkpoint names."""
import torch
import torch.nn.functional as F

from magicdrive_b200 import arch
from oracle.torch_oracle import SD, _conv, _lin, resnet_block


def vae_encode(sd: SD, cfg: "arch.VaeConfig", x):
    """AutoencoderKL.encode up to the moments (autoencoder_kl.py:160-165: Encoder.forward, then quant_conv): conv_in
    (vae.py:53-59), 4 DownEncoderBlock2D (2 resnets each, unet_2d_blocks.py:1030-1087) with a Downsample2D(padding=0) on
    all but the last (resnet.py:213-222: F.pad(x, (0, 1, 0, 1)), then a stride-2 3x3 conv), UNetMidBlock2D (resnet,
    single-head attention with GroupNorm + residual, resnet; unet_2d_blocks.py:395-473), GroupNorm(1e-6), SiLU, conv_out
    to 2 * latent_channels (double_z, vae.py:94-97, 99-133), quant_conv 1x1.  Returns the NCHW moments (mean | logvar)."""
    g, eps = cfg.norm_num_groups, 1e-6
    x = _conv(sd, "encoder.conv_in", x)
    for _, resnets, down in arch.vae_encoder_blocks(cfg):
        for p, _, _ in resnets:
            x = resnet_block(sd, p, x, None, g, eps)
        if down:
            x = _conv(sd, down, F.pad(x, (0, 1, 0, 1)), stride=2, padding=0)
    x = resnet_block(sd, "encoder.mid_block.resnets.0", x, None, g, eps)
    a = "encoder.mid_block.attentions.0"
    b, c, h, w = x.shape
    t = F.group_norm(x.view(b, c, h * w), g, sd[a + ".group_norm.weight"], sd[a + ".group_norm.bias"], eps).transpose(1, 2)
    q, k, v = _lin(sd, a + ".to_q", t), _lin(sd, a + ".to_k", t), _lin(sd, a + ".to_v", t)
    o = torch.softmax(q @ k.transpose(1, 2) * c ** -0.5, dim=-1) @ v
    x = x + _lin(sd, a + ".to_out.0", o).transpose(1, 2).reshape(b, c, h, w)
    x = resnet_block(sd, "encoder.mid_block.resnets.1", x, None, g, eps)
    x = F.silu(F.group_norm(x, g, sd["encoder.conv_norm_out.weight"], sd["encoder.conv_norm_out.bias"], eps))
    x = _conv(sd, "encoder.conv_out", x)
    return _conv(sd, "quant_conv", x, padding=0)


def posterior(moments, noise=None):
    """DiagonalGaussianDistribution (vae.py:397-416): (mean, logvar clamped to [-30, 20], std) of the moments, and with
    `noise` (the randn_tensor draw of .sample) also mean + std * noise."""
    mean, logvar = torch.chunk(moments, 2, dim=1)
    logvar = torch.clamp(logvar, -30.0, 20.0)
    std = torch.exp(0.5 * logvar)
    return dict(mean=mean, logvar=logvar, std=std, sample=None if noise is None else mean + std * noise)
