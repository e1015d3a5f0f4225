"""TEST INFRASTRUCTURE ONLY — tests/golden/vae_encode_80x104.pt: AutoencoderKL.encode of the reference's diffusers
(autoencoder_kl.py:160-171, vae.py:39-133, 397-416) with name-keyed synthetic weights (block_out_channels 32/64/64/64),
via oracle/ref_shim.py.  The file holds the encoder and quant_conv parameter names / shapes, a seeded 2x3x80x104 input in
[-1, 1] (bf16 values), the posterior's mean and (clamped) logvar, and one posterior sample drawn with a seeded generator.
Run in the build container (needs /root/reference):  python -m oracle.make_golden_vae_encode"""
import os
import sys

import torch

from magicdrive_b200 import arch
from oracle import ref_shim
from oracle.make_golden import OUT

SEED, SAMPLE_SEED = 7, 11


@torch.no_grad()
def main():
    R = ref_shim.load()
    cfg = arch.VaeConfig(block_out_channels=(32, 64, 64, 64))
    vae = R.AutoencoderKL(block_out_channels=list(cfg.block_out_channels), down_block_types=["DownEncoderBlock2D"] * 4,
                          up_block_types=["UpDecoderBlock2D"] * 4, latent_channels=4, layers_per_block=2)
    shapes = {k: tuple(v.shape) for k, v in vae.state_dict().items() if k.startswith(("encoder.", "quant_conv."))}
    vae.load_state_dict(arch.synthetic_state_dict(shapes, SEED), strict=False)
    # bf16-representable pixel values, stored as bf16 to halve the file
    x = (torch.rand(2, 3, 80, 104, generator=torch.Generator().manual_seed(3)) * 2 - 1).to(torch.bfloat16)
    post = vae.encode(x.float()).latent_dist
    sample = post.sample(generator=torch.Generator().manual_seed(SAMPLE_SEED))
    path = os.path.join(OUT, "vae_encode_80x104.pt")
    torch.save(dict(block_out_channels=cfg.block_out_channels, seed=SEED, encoder_shapes=shapes, x=x,
                    mean=post.mean.clone(), logvar=post.logvar.clone(), sample_seed=SAMPLE_SEED, sample=sample), path)
    print("vae_encode_80x104.pt", os.path.getsize(path) // 1024, "KiB", tuple(post.mean.shape))


if __name__ == "__main__":
    sys.exit(main())
