"""Pins the oracle (oracle/torch_oracle.py): (a) the reference's own known-answer tests for the layers on the path
(hard-coded slices copied from third_party/diffusers/tests/models/test_layers_utils.py and tests/schedulers), rebuilt
here by replaying the reference constructors' RNG order with plain torch.nn layers; (b) fixtures produced by running
the reference itself (tests/golden/*.pt <- oracle/make_golden.py)."""
import pytest
import torch
import torch.nn as nn

from magicdrive_b200 import arch
from oracle import torch_oracle as O
from tests.common import golden, tiny_configs, tiny_state_dicts


def _sd(**mods):
    sd = {}
    for name, m in mods.items():
        for k, v in m.state_dict().items():
            sd[f"{name}.{k}"] = v
    return sd


def test_timestep_embedding_known_answer():
    # test_layers_utils.py:88-114 (EmbeddingsTests.test_sinoid_embeddings_hardcoded)
    ts = torch.arange(128)
    t1 = O.timestep_embedding(ts, 64, flip_sin_to_cos=False, freq_shift=1)
    t2 = O.timestep_embedding(ts, 64, flip_sin_to_cos=True, freq_shift=0)
    assert torch.allclose(t1[23:26, 47:50].flatten(),
                          torch.tensor([0.9646, 0.9804, 0.9892, 0.9615, 0.9787, 0.9882, 0.9582, 0.9769, 0.9872]), 1e-3)
    assert torch.allclose(t2[23:26, 47:50].flatten(),
                          torch.tensor([0.3019, 0.2280, 0.1716, 0.3146, 0.2377, 0.1790, 0.3272, 0.2474, 0.1864]), 1e-3)


@torch.no_grad()
def test_resnet_block_known_answers():
    # test_layers_utils.py:223-251 (ResnetBlock2DTests.test_resnet_default / test_restnet_with_use_in_shortcut)
    for shortcut, expected in ((False, [-1.9010, -0.2974, -0.8245, -1.3533, 0.8742, -0.9645, -2.0584, 1.3387, -0.4746]),
                               (True, [0.2226, -1.0791, -0.1629, 0.3659, -0.2889, -1.2376, 0.0582, 0.9206, 0.0044])):
        torch.manual_seed(0)
        sample, temb = torch.randn(1, 32, 64, 64), torch.randn(1, 128)
        mods = dict(norm1=nn.GroupNorm(32, 32), conv1=nn.Conv2d(32, 32, 3, padding=1), time_emb_proj=nn.Linear(128, 32),
                    norm2=nn.GroupNorm(32, 32), conv2=nn.Conv2d(32, 32, 3, padding=1))
        if shortcut:
            mods["conv_shortcut"] = nn.Conv2d(32, 32, 1)
        sd = {"r." + k: v for k, v in _sd(**mods).items()}
        out = O.resnet_block(sd, "r", sample, temb, groups=32, eps=1e-6)
        assert torch.allclose(out[0, -1, -3:, -3:].flatten(), torch.tensor(expected), atol=1e-3)


@torch.no_grad()
def test_transformer2d_known_answers():
    # test_layers_utils.py:315-363 (Transformer2DModelTests.test_spatial_transformer_default / _cross_attention_dim)
    def build(c, cross):
        inner = c
        m = dict()
        m["proj_in"] = nn.Conv2d(c, inner, 1)
        b = "transformer_blocks.0."
        for a, kv in (("attn1", c),) + ((("attn2", cross),) if cross else ()):
            m[b + a + ".to_q"] = nn.Linear(c, c, bias=False)
            m[b + a + ".to_k"] = nn.Linear(kv, c, bias=False)
            m[b + a + ".to_v"] = nn.Linear(kv, c, bias=False)
            m[b + a + ".to_out.0"] = nn.Linear(c, c)
        m[b + "ff.net.0.proj"] = nn.Linear(c, 8 * c)
        m[b + "ff.net.2"] = nn.Linear(4 * c, c)
        m["proj_out"] = nn.Conv2d(inner, c, 1)
        m["norm"] = nn.GroupNorm(32, c)
        for n in ("norm1", "norm2", "norm3"):
            m[b + n] = nn.LayerNorm(c)
        return {"t." + k: v for k, v in _sd(**m).items()}

    torch.manual_seed(0)
    sample = torch.randn(1, 32, 64, 64)
    sd = build(32, None)
    out = O.transformer_2d(sd, "t", sample, None, heads=1, multiview=False)
    assert torch.allclose(out[0, -1, -3:, -3:].flatten(),
                          torch.tensor([-1.9455, -0.0066, -1.3933, -1.5878, 0.5325, -0.6486, -1.8648, 0.7515, -0.9689]), atol=1e-3)
    torch.manual_seed(0)
    sample = torch.randn(1, 64, 64, 64)
    sd = build(64, 64)
    ctx = torch.randn(1, 4, 64)
    out = O.transformer_2d(sd, "t", sample, ctx, heads=2, multiview=False)
    assert torch.allclose(out[0, -1, -3:, -3:].flatten(),
                          torch.tensor([0.0143, -0.6909, -2.1547, -1.8893, 1.4097, 0.1359, -0.2521, -1.3359, 0.2598]), atol=1e-3)


@torch.no_grad()
def test_resample_known_answers():
    # Downsample2D with conv: test_layers_utils.py:183-196 (test_downsample_with_conv) -- stride-2 3x3, padding 1
    torch.manual_seed(0)
    sample = torch.randn(1, 32, 64, 64)
    conv = nn.Conv2d(32, 32, 3, stride=2, padding=1)
    out = O._conv({"d.weight": conv.weight, "d.bias": conv.bias}, "d", sample, stride=2, padding=1)
    assert torch.allclose(out[0, -1, -3:, -3:].flatten(),
                          torch.tensor([0.9267, 0.5878, 0.3337, 1.2321, -0.1191, -0.3984, -0.7532, -0.0715, -0.3913]), atol=1e-3)
    # Upsample2D without conv: test_layers_utils.py:118-128 (test_upsample_default) -- nearest resize
    torch.manual_seed(0)
    sample = torch.randn(1, 32, 32, 32)
    up = torch.nn.functional.interpolate(sample, size=(64, 64), mode="nearest")
    assert torch.allclose(up[0, -1, -3:, -3:].flatten(),
                          torch.tensor([-0.2173, -1.2079, -1.2079, 0.2952, 1.1254, 1.1254, 0.2952, 1.1254, 1.1254]), atol=1e-3)
    # Upsample2D with conv (:130-142): the slice hard-coded in the reference test is STALE -- the reference's own
    # Upsample2D run in the build container (torch 2.11, via oracle/ref_shim.py) returns the values below, and so
    # does the restatement.  Recorded 2026-09-22.
    torch.manual_seed(0)
    sample = torch.randn(1, 32, 32, 32)
    conv = nn.Conv2d(32, 32, 3, padding=1)
    out = O.upsample({"u.weight": conv.weight, "u.bias": conv.bias}, "u", sample, (64, 64))
    assert torch.allclose(out[0, -1, -3:, -3:].flatten(),
                          torch.tensor([0.7145, 1.3773, 0.3492, 0.8448, 1.0839, -0.3341, 0.5956, 0.1250, -0.4841]), atol=1e-3)


def test_ddim_matches_reference_schedule_and_closed_form():
    # scheduling_ddim.py:287-323,325-445; full_loop-style check of step() == c0*x + c1*eps
    d = O.DDIM()
    ts = d.set_timesteps(50)
    assert ts[:3].tolist() == [981, 961, 941] and ts[-1].item() == 1
    g = torch.Generator().manual_seed(0)
    x, e = torch.randn(4, 4, 8, 8, generator=g), torch.randn(4, 4, 8, 8, generator=g)
    for t in (981, 501, 1):
        c0, c1 = d.coefficients(t)
        assert torch.allclose(d.step(e, t, x), c0 * x + c1 * e, atol=2e-6)
    from magicdrive_b200.pipeline import DDIMSchedule
    s = DDIMSchedule()
    assert s.set_timesteps(50) == ts.tolist()
    for (c0, c1), t in zip(s.coefs, ts.tolist()):
        r0, r1 = d.coefficients(t)
        assert abs(c0 - r0) < 1e-6 and abs(c1 - r1) < 1e-6


@torch.no_grad()
def test_oracle_reproduces_reference_forward_fixture():
    g = golden("tiny_forward.pt")
    ucfg, ccfg = tiny_configs()
    usd, csd = tiny_state_dicts(g["seed"])
    inp = g["inputs"]
    s, n, h, w = g["shape"]
    lat5 = torch.stack([inp["latents"]] * n, 1)
    down, mid, ctx = O.controlnet_forward(csd, ccfg, lat5, torch.tensor([g["t"]]), inp["camera_param"],
                                          inp["bboxes_3d_data"], inp["prompt_embeds"], inp["bev_map"])
    torch.testing.assert_close(ctx, g["ctx"], rtol=1e-4, atol=1e-4)
    for a, b in zip(down, g["down"]):
        torch.testing.assert_close(a, b, rtol=1e-4, atol=1e-5 * b.abs().max().item() + 1e-5)
    torch.testing.assert_close(mid, g["mid"], rtol=1e-4, atol=1e-5 * g["mid"].abs().max().item())
    eps = O.unet_forward(usd, ucfg, lat5.reshape(-1, 4, h, w), torch.tensor(g["t"]), ctx, down, mid)
    torch.testing.assert_close(eps, g["eps"], rtol=1e-3, atol=1e-4)   # the north-star tolerance, met in fp32
    eps2 = O.unet_forward(usd, ucfg, lat5.reshape(-1, 4, h, w), g["t"], ctx)
    torch.testing.assert_close(eps2, g["eps_noctrl"], rtol=1e-3, atol=1e-4)


@torch.no_grad()
def test_oracle_reproduces_reference_sd15_size_fixture():
    """The oracle at the size the benchmark runs (SD-1.5 config: 4 levels, head dims 40 / 80 / 160, 6 views, 20 boxes,
    200x200 BEV map) against the reference's own forward (oracle/make_golden_sd15.py): pins the full-size structure
    (arch.py is shared between oracle and product, so a structural error common to both would otherwise pass)."""
    from magicdrive_b200.synthetic import synthetic_inputs
    g = golden("sd15_forward.pt")
    ucfg, ccfg = arch.UNetConfig(), arch.ControlNetConfig(map_size=(8, g["map_hw"], g["map_hw"]))
    usd = arch.synthetic_state_dict(arch.unet_param_shapes(ucfg), g["seeds"][0])
    csd = arch.synthetic_state_dict(arch.controlnet_param_shapes(ccfg), g["seeds"][1])
    s, n, h, w = g["shape"]
    inp = synthetic_inputs(s, n, h, w, n_box=g["n_box"], map_hw=g["map_hw"], seed=g["input_seed"])
    lat5 = torch.stack([inp["latents"]] * n, 1)
    t = torch.tensor([g["t"]])
    down, mid, ctx = O.controlnet_forward(csd, ccfg, lat5, t, inp["camera_param"], inp["bboxes_3d_data"],
                                          inp["prompt_embeds"], inp["bev_map"])
    eps = O.unet_forward(usd, ucfg, lat5.reshape(-1, 4, h, w), t[0], ctx, down, mid)
    cs, xs = g["ch_step"], g["ctx_step"]
    assert len(down) == g["n_down"]
    for d, nrm in zip(down, g["down_norms"]):
        assert abs(float(d.norm()) - nrm) <= 2e-4 * nrm
    # the north star's literal tolerance (rtol 1e-3 / atol 1e-4), met by the fp32 oracle at every tap
    assert torch.allclose(ctx[:, :, ::xs], g["ctx"], rtol=1e-3, atol=1e-4)
    assert torch.allclose(down[0][:, ::cs], g["down0"], rtol=1e-3, atol=1e-4)
    assert torch.allclose(down[11][:, ::cs], g["down11"], rtol=1e-3, atol=1e-4)
    assert torch.allclose(mid[:, ::cs], g["mid"], rtol=1e-3, atol=1e-4)
    assert torch.allclose(eps, g["eps"], rtol=1e-3, atol=1e-4), (eps - g["eps"]).abs().max()


@torch.no_grad()
def test_oracle_reproduces_reference_pipeline_fixture():
    p = golden("tiny_pipeline.pt")
    ucfg, ccfg = tiny_configs()
    usd, csd = tiny_state_dicts(p["seed"])
    inp = p["inputs"]
    out = O.denoise_loop(usd, csd, ucfg, ccfg, inp["latents"], inp["prompt_embeds"], inp["negative_prompt_embeds"],
                         inp["camera_param"], inp["bboxes_3d_data"], inp["bev_map"], p["steps"], p["guidance"])
    # three chained fp32 steps through O(500)-magnitude activations: allow 3e-4 of the output range
    torch.testing.assert_close(out, p["latents_out"], rtol=1e-3, atol=3e-4 * p["latents_out"].abs().max().item())


@torch.no_grad()
def test_oracle_reproduces_reference_encoders_fixture():
    e = golden("tiny_encoders.pt")
    _, ccfg = tiny_configs()
    _, csd = tiny_state_dicts(e["seed"])
    torch.testing.assert_close(O.embed_camera(e["camera_param"], 4), e["cam_emb"], rtol=0, atol=0)
    torch.testing.assert_close(O.bbox_embed(csd, ccfg, e["boxes"]["bboxes"], e["boxes"]["classes"], e["boxes"]["masks"]),
                               e["box_emb"], rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(O.map_encode(csd, ccfg, e["bev_map"].float()), e["map_emb"], rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(O.uncond_cam_param(csd, ccfg, 2, 6).contiguous(), e["uncond_cam"], rtol=0, atol=0)


def test_oracle_unipc_reproduces_reference_scheduler_fixture():
    """UniPCMultistepScheduler (the reference's default sampler) stepped by the reference itself over seeded tensors
    (oracle/make_golden_unipc.py): the restatement must follow the whole trajectory, incl. warm-up and final lower order."""
    cases = golden("unipc_scheduler.pt")
    for n, c in cases.items():
        s = O.UniPC()
        assert torch.equal(s.set_timesteps(n), c["timesteps"])
        x = c["x"].clone()
        for i, t in enumerate(c["timesteps"].tolist()):
            x = s.step(c["eps"][i], t, x)
            torch.testing.assert_close(x, c["traj"][i], rtol=1e-5, atol=1e-5)


@torch.no_grad()
def test_oracle_reproduces_reference_unipc_pipeline_fixture():
    """The unmodified reference pipeline with its default UniPC sampler, 4 steps, CFG 2.0 (tiny models)."""
    p = golden("tiny_pipeline_unipc.pt")
    inp = golden(p["inputs_from"])["inputs"]
    ucfg, ccfg = tiny_configs()
    usd, csd = tiny_state_dicts(p["seed"])
    out = O.denoise_loop(usd, csd, ucfg, ccfg, inp["latents"], inp["prompt_embeds"], inp["negative_prompt_embeds"],
                         inp["camera_param"], inp["bboxes_3d_data"], inp["bev_map"], p["steps"], p["guidance"],
                         scheduler="unipc")
    torch.testing.assert_close(out, p["latents_out"], rtol=1e-3, atol=3e-4 * p["latents_out"].abs().max().item())


@torch.no_grad()
@pytest.mark.parametrize("case,scheduler,change", [("ddim_change", "ddim", True), ("ddim_once", "ddim", False),
                                                   ("unipc_change", "unipc", True)])
def test_oracle_reproduces_reference_given_view_fixture(case, scheduler, change):
    """StableDiffusionBEVControlNetGivenViewPipeline.__call__ run by the reference (oracle/make_golden_given_view.py):
    views 0 and 3 pinned to clean latents, both re-noising modes."""
    from oracle.make_golden_given_view import pinned_latents
    p = golden("tiny_given_view.pt")
    inp = golden(p["inputs_from"])["inputs"]
    ucfg, ccfg = tiny_configs()
    usd, csd = tiny_state_dicts(p["seed"])
    out = O.denoise_loop(usd, csd, ucfg, ccfg, inp["latents"], inp["prompt_embeds"], inp["negative_prompt_embeds"],
                         inp["camera_param"], inp["bboxes_3d_data"], inp["bev_map"], p["steps"], p["guidance"],
                         scheduler=scheduler, conditional_latents=pinned_latents(p["pinned_seed"]), change_every_input=change)
    ref = p["outputs"][case]
    torch.testing.assert_close(out, ref, rtol=1e-3, atol=3e-4 * ref.abs().max().item())


@torch.no_grad()
def test_oracle_vae_decode_matches_reference_autoencoder():
    """AutoencoderKL.decode of the reference's diffusers (autoencoder_kl.py:177-196) vs the restatement, same weights: the
    reference decoder's parameter names / shapes and its output on a 10x13 latent grid (oracle/make_golden_vae.py)."""
    from magicdrive_b200 import arch
    g = golden("vae_decode_10x13.pt")
    cfg = arch.VaeConfig(block_out_channels=tuple(g["block_out_channels"]))
    shapes = arch.vae_decoder_param_shapes(cfg)
    assert g["decoder_shapes"] == dict(shapes)
    sd = arch.synthetic_state_dict(shapes, g["seed"])
    s = g["step"]
    torch.testing.assert_close(O.vae_decode(sd, cfg, g["z"])[:, :, ::s, ::s], g["sample"], rtol=1e-4, atol=1e-4)
    assert len(arch.vae_decoder_param_shapes(arch.VaeConfig())) == 140  # SD-1.5 VAE: decoder + post_quant tensors


@torch.no_grad()
def test_oracle_vae_decode_reproduces_reference_fixture():
    from magicdrive_b200 import arch
    g = golden("vae_decode.pt")
    cfg = arch.VaeConfig(block_out_channels=tuple(g["block_out_channels"]))
    sd = arch.synthetic_state_dict(arch.vae_decoder_param_shapes(cfg), g["seed"])
    torch.testing.assert_close(O.vae_decode(sd, cfg, g["z"]), g["sample"], rtol=1e-4, atol=1e-4)


@torch.no_grad()
@pytest.mark.parametrize("attn_type", ["concat", "self"])
def test_oracle_reproduces_reference_cross_view_attention_types(attn_type):
    """neighboring_attn_type 'concat' / 'self' (magicdrive/networks/blocks.py:122-138, 209-211) against the reference's own
    forward (oracle/make_golden_attn_types.py)."""
    from dataclasses import replace
    g = golden("tiny_attn_types.pt")
    ucfg = replace(tiny_configs()[0], neighboring_attn_type=attn_type)
    usd = arch.synthetic_state_dict(arch.unet_param_shapes(ucfg), g["seed"])
    eps = O.unet_forward(usd, ucfg, g["sample"], torch.tensor(g["t"]), g["ctx"])
    torch.testing.assert_close(eps, g["eps"][attn_type], rtol=1e-3, atol=1e-4)
    other = "self" if attn_type == "concat" else "concat"
    assert (eps - g["eps"][other]).abs().max() > 1e-2  # the modes do differ on this fixture


@torch.no_grad()
def test_oracle_reproduces_reference_guess_mode_residual_scales():
    """guess_mode: residual i scaled by logspace(-1, 0, 13)[i] * conditioning_scale (unet_addon_rawbox.py:897-905)."""
    g, gf = golden("tiny_attn_types.pt")["guess_mode"], golden("tiny_forward.pt")
    _, ccfg = tiny_configs()
    _, csd = tiny_state_dicts(gf["seed"])
    inp = gf["inputs"]
    lat5 = torch.stack([inp["latents"]] * 6, 1)
    down, mid, _ = O.controlnet_forward(csd, ccfg, lat5, torch.tensor([gf["t"]]), inp["camera_param"], inp["bboxes_3d_data"],
                                        inp["prompt_embeds"], inp["bev_map"], conditioning_scale=g["conditioning_scale"],
                                        guess_mode=True)
    for a, b in zip(down + [mid], g["down"] + [g["mid"]]):
        torch.testing.assert_close(a, b, rtol=1e-3, atol=1e-4 * max(1.0, b.abs().max().item()))


def _map_plus_case():
    from dataclasses import replace
    g, gf = golden("tiny_attn_types.pt")["map_plus"], golden("tiny_forward.pt")
    _, ccfg = tiny_configs()
    ccfg = replace(ccfg, map_size=(8, 52, 60), map_embedding_size=(10, 13))
    csd = arch.synthetic_state_dict(arch.controlnet_param_shapes(ccfg), g["seed"])
    return g, gf, ccfg, csd


@torch.no_grad()
def test_oracle_reproduces_reference_map_embedder_plus():
    """BEVControlNetConditioningEmbeddingPlus (map_embedder.py:79-126, the 272x736 experiment's map encoder): embedding and the
    ControlNet residuals computed with it, against the reference's own outputs."""
    g, gf, ccfg, csd = _map_plus_case()
    torch.testing.assert_close(O.map_encode(csd, ccfg, g["bev_map"]), g["embedding"], rtol=1e-3, atol=1e-4)
    inp = gf["inputs"]
    lat5 = torch.stack([inp["latents"]] * 6, 1)[:1]
    down, mid, _ = O.controlnet_forward(csd, ccfg, lat5, torch.tensor([gf["t"]]), inp["camera_param"][:1], None,
                                        inp["prompt_embeds"][:1], g["bev_map"])
    torch.testing.assert_close(mid, g["mid"], rtol=1e-3, atol=1e-4)
    torch.testing.assert_close(down[0], g["down0"], rtol=1e-3, atol=1e-4)
