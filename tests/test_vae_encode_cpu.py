"""The VAE encoder without a GPU: the oracle restatement of AutoencoderKL.encode against the reference's own output
(tests/golden/vae_encode_80x104.pt, oracle/make_golden_vae_encode.py), VaeEncoderEngine's host logic (image-patch conv_in,
stride-2 pad-(0, 1, 0, 1) downsamples, quant_conv folded into conv_out, the posterior) through the emulated operators, the
`with_encoder` module interface, and the given-view recipe fed from `encode_latents`."""
import json
from dataclasses import asdict

import pytest
import torch

from magicdrive_b200 import arch, models
from magicdrive_b200.pipeline import BEVControlNetDenoiser
from magicdrive_b200.synthetic import synthetic_inputs
from oracle import torch_oracle_vae_encode as OE
from tests import vae_encode_emulation
from tests.common import golden, rel_l2, tiny_configs


def _bf16_exact(sd):
    return {k: (v.to(torch.bfloat16).float() if v.is_floating_point() else v) for k, v in sd.items()}


def _full_vae(cfg, seed):
    """A with_encoder AutoencoderKL holding a full synthetic checkpoint (bf16-representable weights)."""
    shapes = dict(arch.vae_encoder_param_shapes(cfg), **arch.vae_decoder_param_shapes(cfg))
    sd = _bf16_exact(arch.synthetic_state_dict(shapes, seed))
    vae = models.AutoencoderKL(**asdict(cfg), with_encoder=True)
    vae.load_state_dict(sd)
    return vae, sd


@pytest.fixture
def emulated(monkeypatch):
    vae_encode_emulation.install(monkeypatch)
    from magicdrive_b200 import engine
    monkeypatch.setattr(engine._Weights, "fold_dtype", torch.float32)  # the quant_conv fold is checked apart from its rounding


@torch.no_grad()
def test_oracle_vae_encode_matches_reference_autoencoder():
    """AutoencoderKL.encode of the reference's diffusers (autoencoder_kl.py:160-171) vs the restatement, same weights."""
    g = golden("vae_encode_80x104.pt")
    cfg = arch.VaeConfig(block_out_channels=tuple(g["block_out_channels"]))
    shapes = arch.vae_encoder_param_shapes(cfg)
    assert dict(shapes) == g["encoder_shapes"]
    sd = arch.synthetic_state_dict(shapes, g["seed"])
    mom = OE.vae_encode(sd, cfg, g["x"].float())
    noise = torch.randn(g["mean"].shape, generator=torch.Generator().manual_seed(g["sample_seed"]))
    post = OE.posterior(mom, noise)
    for k in ("mean", "logvar", "sample"):
        torch.testing.assert_close(post[k], g[k], rtol=1e-4, atol=1e-4)
    assert len(arch.vae_encoder_param_shapes(arch.VaeConfig())) == 108  # SD-1.5 VAE: encoder + quant_conv tensors


@torch.no_grad()
@pytest.mark.parametrize("name,cfg,n,h,w", [("small", arch.VaeConfig(block_out_channels=(64, 128, 128, 128)), 3, 48, 64),
                                            ("sd15", arch.VaeConfig(), 1, 32, 40)])
def test_vae_encoder_through_emulated_operators_matches_the_oracle(emulated, name, cfg, n, h, w):
    vae, sd = _full_vae(cfg, 71)
    x = torch.rand(n, 3, h, w, generator=torch.Generator().manual_seed(5)) * 2 - 1
    post = vae.encode(x).latent_dist
    ref = OE.posterior(OE.vae_encode(sd, cfg, x))
    assert post.mean.shape == ref["mean"].shape == (n, 4, h // 8, w // 8)
    assert rel_l2(post.mean, ref["mean"]) < 1e-5 and rel_l2(post.logvar, ref["logvar"]) < 1e-5
    assert rel_l2(post.std, ref["std"]) < 1e-5 and torch.equal(post.var, torch.exp(post.logvar)) and post.mode() is post.mean
    (p2,) = vae.encode(x, return_dict=False)
    assert torch.equal(p2.mean, post.mean)
    # the demo's three lines in one call
    lat = vae.encode_latents(x[None])
    assert lat.shape == (1, n, 4, h // 8, w // 8) and lat.dtype == torch.float32
    assert torch.equal(lat[0], post.mean * vae.config.scaling_factor)


@torch.no_grad()
def test_with_encoder_module_interface(emulated, tmp_path):
    g = golden("vae_encode_80x104.pt")
    cfg = arch.VaeConfig(block_out_channels=tuple(g["block_out_channels"]))
    vae, sd = _full_vae(cfg, 72)
    # the key set is diffusers' full AutoencoderKL: the reference encoder's and decoder's names
    dec = golden("vae_decode_10x13.pt")["decoder_shapes"]
    assert {k: tuple(v.shape) for k, v in vae.state_dict().items()} == {**g["encoder_shapes"], **dec}
    # strict loading needs the encoder keys; pre-0.17 attention names of both mid blocks are mapped
    old = dict(sd)
    for half in ("encoder", "decoder"):
        for new, o in (("to_q", "query"), ("to_k", "key"), ("to_v", "value"), ("to_out.0", "proj_attn")):
            for leaf in ("weight", "bias"):
                old[f"{half}.mid_block.attentions.0.{o}.{leaf}"] = old.pop(f"{half}.mid_block.attentions.0.{new}.{leaf}")
    fresh = models.AutoencoderKL(**asdict(cfg), with_encoder=True)
    fresh.load_state_dict(old)
    assert all(torch.equal(fresh.state_dict()[k], v) for k, v in sd.items())
    with pytest.raises(RuntimeError):
        models.AutoencoderKL(**asdict(cfg), with_encoder=True).load_state_dict(
            {k: v for k, v in sd.items() if not k.startswith("encoder.")})
    # save -> from_pretrained restores with_encoder from config.json; a decoder-only config.json takes it as a keyword
    for sub, conf in (("saved", dict(vae.config)), ("plain", asdict(cfg))):
        d = tmp_path / sub / "vae"
        d.mkdir(parents=True)
        (d / "config.json").write_text(json.dumps({"_class_name": "AutoencoderKL",
                                                  **{k: (list(v) if isinstance(v, tuple) else v) for k, v in conf.items()}}))
        torch.save(sd, d / "diffusion_pytorch_model.bin")
        kw = {} if sub == "saved" else {"with_encoder": True}
        m = models.AutoencoderKL.from_pretrained(str(tmp_path / sub), subfolder="vae", **kw)
        assert m.with_encoder and m.config["with_encoder"] is True and set(m.state_dict()) == set(sd)
    # posterior sample = mean + std * randn of the same seeded generator (DiagonalGaussianDistribution.sample)
    x = g["x"].float()
    post = vae.encode(x).latent_dist
    s = post.sample(torch.Generator().manual_seed(3))
    noise = torch.randn(post.mean.shape, generator=torch.Generator().manual_seed(3))
    assert torch.equal(s, post.mean + post.std * noise)
    z = vae.encode_latents(x[None], sample=True, generator=torch.Generator().manual_seed(3))
    assert rel_l2(z[0], s * vae.config.scaling_factor) < 1e-6
    with pytest.raises(ValueError):
        vae.encode(x[:, :, :76])  # H not divisible by 8
    # the default module is still the decoder only
    dflt = models.AutoencoderKL(**asdict(cfg))
    assert "with_encoder" not in dflt.config and not any(k.startswith(("encoder.", "quant_conv.")) for k in dflt.state_dict())
    with pytest.raises(NotImplementedError):
        dflt.encode(x)
    with pytest.raises(NotImplementedError):
        dflt.encode_latents(x[None])


@torch.no_grad()
def test_given_view_recipe_from_encode_latents(emulated):
    """The demo's recipe with this package alone (demo/run_cond_on_view.py:80-112): encode_latents, pick views into
    conditional_latents, run the given-view denoiser.  Latents staged from where encode_latents left them or from host
    copies give the same result, and match the recipe run on the oracle's latents."""
    ucfg, ccfg = tiny_configs()
    un = models.UNet2DConditionModelMultiview(**asdict(ucfg))
    cn = models.BEVControlNetModel(**asdict(ccfg))
    un.load_state_dict(_bf16_exact(arch.synthetic_state_dict(arch.unet_param_shapes(ucfg), 41)))
    cn.load_state_dict(_bf16_exact(arch.synthetic_state_dict(arch.controlnet_param_shapes(ccfg), 42)))
    vcfg = arch.VaeConfig(block_out_channels=(64, 64, 64, 64))
    vae, vsd = _full_vae(vcfg, 73)
    inp = synthetic_inputs(1, 6, 10, 13, n_box=3, map_hw=52, seed=9)
    pixel_values = torch.rand(1, 6, 3, 80, 104, generator=torch.Generator().manual_seed(8)) * 2 - 1
    lat = vae.encode_latents(pixel_values)
    ref_lat = OE.posterior(OE.vae_encode(vsd, vcfg, pixel_values[0]))["mean"][None] * vcfg.scaling_factor
    assert rel_l2(lat, ref_lat) < 1e-5

    def run(latents):
        cond = [[latents[0, v] if v in (0, 3) else None for v in range(6)]]
        pipe = BEVControlNetDenoiser(un, cn, use_cuda_graph=False, overlap_controlnet=False)
        return pipe(image=inp["bev_map"], camera_param=inp["camera_param"], prompt_embeds=inp["prompt_embeds"],
                    negative_prompt_embeds=inp["negative_prompt_embeds"], latents=inp["latents"], num_inference_steps=2,
                    guidance_scale=2.0, bev_controlnet_kwargs={"bboxes_3d_data": inp["bboxes_3d_data"]},
                    conditional_latents=cond)

    out = run(lat)
    assert torch.equal(out, run(lat.cpu().clone()))
    assert rel_l2(out, run(ref_lat)) < 1e-5
