"""TEST INFRASTRUCTURE ONLY — tests/golden/vae_decode.pt: AutoencoderKL.decode of the reference's diffusers run on seeded
latents with name-keyed synthetic weights (block_out_channels 32/64/64/64), via oracle/ref_shim.py; and
tests/golden/vae_decode_10x13.pt: the reference decoder's parameter names / shapes and its output on a 10x13 latent grid
(every second output row and column, to keep the file small).
Run in the build container (needs /root/reference):  python -m oracle.make_golden_vae"""
import os
import sys

import torch

from magicdrive_b200 import arch
from oracle import ref_shim
from oracle.make_golden import OUT


@torch.no_grad()
def main():
    R = ref_shim.load()
    cfg = arch.VaeConfig(block_out_channels=(32, 64, 64, 64))
    vae = R.AutoencoderKL(block_out_channels=list(cfg.block_out_channels), down_block_types=["DownEncoderBlock2D"] * 4,
                          up_block_types=["UpDecoderBlock2D"] * 4, latent_channels=4, layers_per_block=2)
    vae.load_state_dict(arch.synthetic_state_dict(arch.vae_decoder_param_shapes(cfg), 5), strict=False)
    decoder_shapes = {k: tuple(v.shape) for k, v in vae.state_dict().items() if k.startswith(("decoder.", "post_quant_conv."))}
    z = torch.randn(2, 4, 6, 7, generator=torch.Generator().manual_seed(1))
    out = vae.decode(z).sample
    torch.save(dict(block_out_channels=cfg.block_out_channels, seed=5, z=z, sample=out), os.path.join(OUT, "vae_decode.pt"))
    z2 = torch.randn(2, 4, 10, 13, generator=torch.Generator().manual_seed(1))
    torch.save(dict(block_out_channels=cfg.block_out_channels, seed=5, decoder_shapes=decoder_shapes, z=z2, step=2,
                    sample=vae.decode(z2).sample[:, :, ::2, ::2].clone()), os.path.join(OUT, "vae_decode_10x13.pt"))
    print("vae_decode.pt", os.path.getsize(os.path.join(OUT, "vae_decode.pt")) // 1024, "KiB", tuple(out.shape))


if __name__ == "__main__":
    sys.exit(main())
