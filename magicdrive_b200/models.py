"""Drop-in modules for the two networks of the hot path.

`UNet2DConditionModelMultiview` and `BEVControlNetModel` keep the reference's constructor kwargs, parameter names
(so `load_state_dict(reference.state_dict())` and the diffusers `save_pretrained` directories load unchanged),
`forward` signatures and return types (magicdrive/networks/unet_2d_condition_multiview.py:327-339,524-527;
magicdrive/networks/unet_addon_rawbox.py:707-724,921-932), plus the helper methods the pipeline calls
(`uncond_cam_param`, `add_uncond_to_kwargs`, `prepare`).  Their arithmetic runs in `engine.py` on the sm_100a
kernels; inputs must be CUDA tensors — there is no CPU path (ops raise).
"""
import json
import logging
import os
from collections import OrderedDict
from dataclasses import asdict, dataclass, fields
from typing import Any, Dict, List, Optional, Tuple, Union

import torch
import torch.nn as nn

from . import arch, ops
from .engine import ControlNetEngine, UNetEngine, VaeDecoderEngine, VaeEncoderEngine

BF16, F32 = torch.bfloat16, torch.float32


@dataclass
class UNet2DConditionOutput:
    sample: torch.Tensor

    def __getitem__(self, i):
        return (self.sample,)[i]


@dataclass
class BEVControlNetOutput:  # magicdrive/networks/output_cls.py:8-13
    down_block_res_samples: Tuple[torch.Tensor]
    mid_block_res_sample: torch.Tensor
    encoder_hidden_states_with_cam: torch.Tensor


class _Config(dict):
    """dict with attribute access, like diffusers' FrozenDict config."""
    __getattr__ = dict.__getitem__


def _register_tree(root: nn.Module, shapes: "OrderedDict[str, tuple]", dtype=F32):
    """Create nested nn.Modules so that parameter names equal the reference checkpoint keys."""
    for key, shape in shapes.items():
        parts = key.split(".")
        mod = root
        for name in parts[:-1]:
            if name not in mod._modules:
                mod.add_module(name, nn.Module())
            mod = mod._modules[name]
        t = torch.empty(shape, dtype=dtype)
        if key in arch.BUFFER_KEYS:
            mod.register_buffer(parts[-1], t)
        else:
            mod.register_parameter(parts[-1], nn.Parameter(t, requires_grad=False))


class _B200Module(nn.Module):
    config_name = "config.json"
    _cfg_cls = None

    def _init_common(self, cfg, shapes, extra_config: Dict[str, Any]):
        self.arch_cfg = cfg
        cd = {k: (list(v) if isinstance(v, tuple) else v) for k, v in asdict(cfg).items()}
        cd.update(extra_config)
        self.config = _Config(cd)
        _register_tree(self, shapes)
        self._engine = None
        self._engine_key = None
        self._ctx_cache = {}
        self._view_shard = None  # re-applied to every engine this module builds (engines are rebuilt when weights change)

    # -- nn.Module conveniences the pipeline relies on (pipeline_utils.py:624, 664-685)
    @property
    def dtype(self):
        return next(self.parameters()).dtype

    @property
    def device(self):
        return next(self.parameters()).device

    def set_use_memory_efficient_attention_xformers(self, *a, **k):  # attention is always our fused kernel
        return None

    enable_xformers_memory_efficient_attention = set_use_memory_efficient_attention_xformers

    def load_state_dict(self, state_dict, strict=True, **kw):
        r = super().load_state_dict(state_dict, strict=strict, **kw)
        self._engine = None
        self._ctx_cache = {}
        return r

    def _apply(self, fn, *a, **k):
        r = super()._apply(fn, *a, **k)
        self._engine = None
        self._ctx_cache = {}
        return r

    def reset_parameters_synthetic(self, seed=0):
        """Deterministic non-zero weights (no checkpoint ships with the reference: pretrained/.gitkeep)."""
        shapes = OrderedDict((k, tuple(v.shape)) for k, v in self.state_dict().items())
        self.load_state_dict(arch.synthetic_state_dict(shapes, seed))
        return self

    @classmethod
    def from_pretrained(cls, path, torch_dtype=None, subfolder=None, **kw):
        """Load a diffusers `save_pretrained` directory: config.json + diffusion_pytorch_model.{safetensors,bin}
        (multiview_runner.py:233-242; utils/constants.py:22-26)."""
        if subfolder:
            path = os.path.join(path, subfolder)
        with open(os.path.join(path, cls.config_name)) as f:
            raw = json.load(f)
        # keyword arguments override / extend config.json, as in diffusers (e.g. AutoencoderKL's with_encoder=True)
        model = cls(**{**{k: v for k, v in raw.items() if not k.startswith("_")}, **kw})
        st = os.path.join(path, "diffusion_pytorch_model.safetensors")
        if os.path.exists(st):
            from safetensors.torch import load_file
            sd = load_file(st)
        else:
            sd = torch.load(os.path.join(path, "diffusion_pytorch_model.bin"), map_location="cpu", weights_only=True)
        model.load_state_dict(sd, strict=True)
        if torch_dtype is not None:
            model = model.to(torch_dtype)
        return model

    def _get_engine(self, cls_):
        dev = self.device
        if dev.type != "cuda":
            raise ops._lib.MdbError(f"{type(self).__name__} runs only on a CUDA (sm_100a) device; parameters are on {dev}")
        if self._engine is None:
            self._engine = cls_(self.arch_cfg, dict(self.state_dict()), dev)
            if self._view_shard is not None and hasattr(self._engine, "set_view_shard"):
                self._engine.set_view_shard(self._view_shard)
        return self._engine

    def set_view_shard(self, shard) -> None:
        """Split the cameras across ranks (dist.ViewShard) or None; survives engine rebuilds (load_state_dict / .to())."""
        self._view_shard = shard
        if self._engine is not None and hasattr(self._engine, "set_view_shard"):
            self._engine.set_view_shard(shard)


def _timesteps_f32(timestep, n, device):
    """unet_2d_condition_multiview.py:386-402: python number, 0-dim or (V,) tensor -> fp32 [n] on device."""
    if not torch.is_tensor(timestep):
        t = torch.tensor([timestep], dtype=F32, device=device)
    else:
        t = timestep.reshape(-1).to(device=device, dtype=F32)
    if t.numel() == 1 and n > 1:
        t = t.expand(n)
    return t.contiguous()


def _pick(cfg_cls, kwargs):
    names = {f.name for f in fields(cfg_cls)}
    known = {k: (tuple(v) if isinstance(v, list) else v) for k, v in kwargs.items() if k in names}
    extra = {k: v for k, v in kwargs.items() if k not in names}
    return known, extra


class UNet2DConditionModelMultiview(_B200Module):
    """B200-native stand-in for magicdrive.networks.unet_2d_condition_multiview.UNet2DConditionModelMultiview."""

    def __init__(self, **kwargs):
        super().__init__()
        known, extra = _pick(arch.UNetConfig, kwargs)
        if "neighboring_view_pair" in known and known["neighboring_view_pair"] is not None:
            known["neighboring_view_pair"] = {int(k): [int(x) for x in v] for k, v in known["neighboring_view_pair"].items()}
        elif "neighboring_view_pair" in known:
            known.pop("neighboring_view_pair")
        cfg = arch.UNetConfig(**known)
        for k, want in (("use_linear_projection", False), ("class_embed_type", None), ("addition_embed_type", None),
                        ("resnet_time_scale_shift", "default"), ("dual_cross_attention", False),
                        ("upcast_attention", False), ("center_input_sample", False), ("encoder_hid_dim", None),
                        ("crossview_attn_type", "basic"), ("only_cross_attention", False), ("act_fn", "silu")):
            if extra.get(k, want) != want:
                raise ValueError(f"UNet2DConditionModelMultiview (B200): unsupported config {k}={extra[k]!r}")
        self._init_common(cfg, arch.unet_param_shapes(cfg), extra)

    @classmethod
    def stock_unet(cls, **kwargs):
        """The plain diffusers UNet2DConditionModel (unet_2d_condition.py:161-505) on the same engine: no cross-view attention,
        any batch size (BASELINE.json configs[0]: 1-view SD-1.5 UNet, text-only conditioning)."""
        return cls(neighboring_view_pair={}, **kwargs)

    def engine(self) -> UNetEngine:
        return self._get_engine(UNetEngine)

    def prepare_context(self, encoder_hidden_states: torch.Tensor):
        """Project the conditioning tokens to K/V for all 16 transformer blocks (cached while the tensor is unchanged)."""
        eng = self._get_engine(UNetEngine)
        key = (encoder_hidden_states.data_ptr(), encoder_hidden_states._version, tuple(encoder_hidden_states.shape),
               encoder_hidden_states.dtype)
        hit = self._ctx_cache.get("kv")
        if hit is None or hit[0] != key:
            v, lc, cdim = encoder_hidden_states.shape
            ctx = encoder_hidden_states.reshape(v * lc, cdim)
            ctx = ops.f32_to_bf16(ctx.float().contiguous()) if ctx.dtype != BF16 else ctx.contiguous()
            hit = (key, eng.context_kv(ctx), lc, encoder_hidden_states)  # keep a ref so data_ptr is not recycled
            self._ctx_cache["kv"] = hit
        return hit[1], hit[2]

    @torch.no_grad()
    def forward(self, sample, timestep, encoder_hidden_states, class_labels=None, timestep_cond=None,
                attention_mask=None, cross_attention_kwargs=None, down_block_additional_residuals=None,
                mid_block_additional_residual=None, return_dict: bool = True):
        if attention_mask is not None or class_labels is not None or timestep_cond is not None:
            raise ValueError("attention_mask / class_labels / timestep_cond are not used by the MagicDrive path")
        eng = self._get_engine(UNetEngine)
        n, c, h, w = sample.shape
        if self.arch_cfg.multiview and n % self.arch_cfg.n_cam:
            raise ValueError(f"batch {n} is not a multiple of the {self.arch_cfg.n_cam} camera views")
        ctx_kv, lc = self.prepare_context(encoder_hidden_states)
        x = ops.pack_latents(ops.nchw_to_nhwc(sample), UNetEngine.CIN_PAD)
        t = _timesteps_f32(timestep, n, sample.device)
        down = mid = None
        if down_block_additional_residuals is not None:
            down = [ops.nchw_to_nhwc(r) for r in down_block_additional_residuals]
        if mid_block_additional_residual is not None:
            mid = ops.nchw_to_nhwc(mid_block_additional_residual)
        eps = eng.forward(x, n, h, w, t, ctx_kv, lc, down, mid)  # fp32 [n*h*w, 8], first out_channels valid
        co = self.arch_cfg.out_channels
        out = eps[:, :co].reshape(n, h, w, co).permute(0, 3, 1, 2).contiguous().to(sample.dtype)
        if not return_dict:
            return (out,)
        return UNet2DConditionOutput(sample=out)


class BEVControlNetModel(_B200Module):
    """B200-native stand-in for magicdrive.networks.unet_addon_rawbox.BEVControlNetModel (inference path)."""

    def __init__(self, **kwargs):
        super().__init__()
        kw = dict(kwargs)
        cep = kw.pop("cam_embedder_param", None) or {}
        bep = kw.pop("bbox_embedder_param", None) or {}
        known, extra = _pick(arch.ControlNetConfig, kw)
        if cep:
            known["cam_num_freqs"] = cep.get("num_freqs", 4)
        if bep:
            if bep.get("mode", "all-xyz") != "all-xyz" or bep.get("minmax_normalize", False):
                raise ValueError("only bbox mode 'all-xyz' without minmax_normalize (SDv1.5mv_rawbox.yaml) is implemented")
            known.update(bbox_n_classes=bep.get("n_classes", 10), bbox_class_token_dim=bep.get("class_token_dim", 768),
                         bbox_num_freqs=bep.get("embedder_num_freq", 4),
                         bbox_proj_dims=tuple(bep.get("proj_dims", (768, 512, 512, 768))))
        if known.get("conditioning_embedding_out_channels") is None:
            known.pop("conditioning_embedding_out_channels", None)
        # map embedder class (unet_addon_rawbox.py:172-181): the default BEVControlNetConditioningEmbedding built from map_size,
        # or BEVControlNetConditioningEmbeddingPlus built from map_embedder_param (configs/exp/272x736.yaml:16-22)
        mcls, mpar = extra.get("map_embedder_cls"), dict(extra.get("map_embedder_param") or {})
        if mcls is not None:
            if str(mcls).rsplit(".", 1)[-1] != "BEVControlNetConditioningEmbeddingPlus":
                raise ValueError(f"map_embedder_cls {mcls!r} is not implemented (BEVControlNetConditioningEmbedding[Plus] only)")
            if "conditioning_embedding_size" not in mpar:
                raise ValueError("BEVControlNetConditioningEmbeddingPlus needs map_embedder_param.conditioning_embedding_size")
            known["map_embedding_size"] = tuple(int(v) for v in mpar["conditioning_embedding_size"])
            known["map_size"] = tuple(mpar.get("conditioning_size", (25, 200, 200)))
            known["conditioning_embedding_out_channels"] = tuple(mpar.get("block_out_channels", (16, 32, 96, 256)))
            if mpar.get("conditioning_embedding_channels", known.get("block_out_channels", (320,))[0]) != \
                    known.get("block_out_channels", (320,))[0]:
                raise ValueError("conditioning_embedding_channels must equal block_out_channels[0]")
        if known.get("map_size") is None:
            known.pop("map_size", None)
        cfg = arch.ControlNetConfig(**known)
        extra.update(cam_embedder_param=cep, bbox_embedder_param=bep,
                     controlnet_conditioning_channel_order=extra.get("controlnet_conditioning_channel_order", "rgb"),
                     global_pool_conditions=extra.get("global_pool_conditions", False))
        self._init_common(cfg, arch.controlnet_param_shapes(cfg), extra)
        # unconditional BEV map (unet_addon_rawbox.py:188-202): present (and a checkpoint key) only when configured
        um = extra.get("use_uncond_map")
        if um is not None and extra.get("drop_cond_ratio", 0.0) > 0:
            if um not in ("negative1", "random", "learnable"):
                raise TypeError(f"Unknown map type: {um}.")
            t = -torch.ones(tuple(cfg.map_size)) if um == "negative1" else torch.randn(tuple(cfg.map_size))
            if um == "learnable":
                self.register_parameter("uncond_map", nn.Parameter(t, requires_grad=False))
            else:
                self.register_buffer("uncond_map", t)
        else:
            self.uncond_map = None
        self.training = False

    def engine(self) -> ControlNetEngine:
        return self._get_engine(ControlNetEngine)

    # ---------------------------------------------------------------- helpers the pipeline calls
    def uncond_cam_param(self, repeat_size: Union[List[int], int] = 1):
        """unet_addon_rawbox.py:307-315."""
        if isinstance(repeat_size, int):
            repeat_size = [1, repeat_size]
        w = self.uncond_cam.weight[0]
        n = 1
        for r in repeat_size:
            n *= int(r)
        return w[None].expand(n, -1).reshape(*repeat_size, -1, self.arch_cfg.uncond_cam_in_dim[1])

    def add_uncond_to_kwargs(self, camera_param, bboxes_3d_data, image, max_len=None, **kwargs):
        """unet_addon_rawbox.py:625-682: uncond (null camera, zero boxes + masks) in front, cond in the tail."""
        batch_size, n_cam = camera_param.shape[:2]
        ret = dict()
        ret["camera_param"] = torch.cat([self.uncond_cam_param([batch_size, n_cam]).to(camera_param), camera_param])
        if bboxes_3d_data is None:
            if not getattr(self, "_warned_no_boxes", False):  # the reference logs this on every call; once is enough
                logging.warning("Your 'bboxes_3d_data' should not be None. If this warning keeps popping, please check your code.")
                self._warned_no_boxes = True
            if max_len is not None:
                dev = camera_param.device
                ret["bboxes_3d_data"] = {
                    "bboxes": torch.zeros([batch_size * 2, n_cam, max_len, 8, 3], device=dev),
                    "classes": torch.zeros([batch_size * 2, n_cam, max_len], device=dev, dtype=torch.long),
                    "masks": torch.zeros([batch_size * 2, n_cam, max_len], device=dev, dtype=torch.bool)}
            else:
                ret["bboxes_3d_data"] = None
        else:
            ret["bboxes_3d_data"] = dict()
            for key in ["bboxes", "classes", "masks"]:
                v = torch.cat([torch.zeros_like(bboxes_3d_data[key]), bboxes_3d_data[key]])
                if max_len is not None:
                    token_num = max_len - v.shape[2]
                    assert token_num >= 0
                    pad = torch.zeros_like(v[:, :, :1]).expand(-1, -1, token_num, *v.shape[3:])
                    v = torch.cat([v, pad], dim=2)
                ret["bboxes_3d_data"][key] = v
        # the unconditional half sees the configured uncond map instead of the scene's (substitute_with_uncond_map, :378-395)
        ret["image"] = image if self.uncond_map is None else self.uncond_map[None].expand_as(image).to(image).clone()
        for k, v in kwargs.items():
            ret[k] = v
        return ret

    @torch.no_grad()
    def prepare(self, cfg, **kwargs):
        """BEVControlNetModel.prepare -> ContinuousBBoxWithTextEmbedding.prepare / set_category_token
        (unet_addon_rawbox.py:704-705, bbox_embedder.py:117-136): with `use_text_encoder_init` the class tokens are the
        pooled CLIP embeddings of the dataset's class names (done once before training; checkpoints already carry them)."""
        if not self.config["bbox_embedder_param"].get("use_text_encoder_init", False):
            return
        tokenizer, text_encoder = kwargs["tokenizer"], kwargs["text_encoder"]
        tokens = self.bbox_embedder._class_tokens
        for idx, name in enumerate(cfg.dataset.object_classes):
            ids = tokenizer([name], padding="do_not_pad", return_tensors="pt").input_ids.to(tokens.device)
            tokens[idx].copy_(text_encoder(ids).pooler_output[0])
        self._engine = None  # weights changed: repack on the next use
        self._ctx_cache = {}

    # ---------------------------------------------------------------- step-invariant conditioning (cached)
    def _key(self, *ts):
        k = []
        for t in ts:
            if t is None:
                k.append(None)
            elif isinstance(t, dict):
                k.append(tuple((n, v.data_ptr(), v._version, tuple(v.shape)) for n, v in sorted(t.items())))
            else:
                k.append((t.data_ptr(), t._version, tuple(t.shape), t.dtype))
        return tuple(k)

    def prepare_conditions(self, camera_param, bboxes_3d_data, encoder_hidden_states, controlnet_cond):
        """Camera / box / text tokens, their K/V projections for the 7 ControlNet transformers and the BEV-map
        embedding: all independent of the latents and of the timestep, so computed once and reused across steps."""
        eng = self._get_engine(ControlNetEngine)
        key = self._key(camera_param, bboxes_3d_data, encoder_hidden_states, controlnet_cond)
        hit = self._ctx_cache.get("cond")
        if hit is None or hit[0] != key:
            n_cam = camera_param.shape[1]
            ctx = eng.context(camera_param, bboxes_3d_data, encoder_hidden_states)  # fp32 (V, Lc, 768)
            ctx_bf = ops.f32_to_bf16(ctx.reshape(-1, ctx.shape[-1]))
            kv = eng.context_kv(ctx_bf)
            memb = eng.map_embedding(controlnet_cond)  # [b, h, w, 320]
            memb = memb.repeat_interleave(n_cam, dim=0).contiguous()  # 'b ... -> (b repeat) ...' (:842-843)
            hit = (key, dict(ctx=ctx, kv=kv, lc=ctx.shape[1], map=memb),
                   (camera_param, bboxes_3d_data, encoder_hidden_states, controlnet_cond))
            self._ctx_cache["cond"] = hit
        return hit[1]

    @torch.no_grad()
    def forward(self, sample, timestep, camera_param, bboxes_3d_data, encoder_hidden_states, controlnet_cond,
                encoder_hidden_states_uncond=None, conditioning_scale: float = 1.0, class_labels=None,
                timestep_cond=None, attention_mask=None, cross_attention_kwargs=None, guess_mode: bool = False,
                return_dict: bool = True, **kwargs):
        # guess_mode: the 12 + 1 residuals are scaled by torch.logspace(-1, 0, 13) * conditioning_scale instead of one factor
        # (unet_addon_rawbox.py:897-905).  Only the MODULE-level switch exists here: the reference pipeline's guess_mode + CFG
        # branch calls add_uncond_to_emb, which has a latent bug (:684-702), so the denoiser does not offer it.
        if self.config.get("controlnet_conditioning_channel_order", "rgb") != "rgb":
            raise ValueError("only 'rgb' controlnet_conditioning_channel_order is supported")
        eng = self._get_engine(ControlNetEngine)
        b, n_cam, c, h, w = sample.shape
        cond = self.prepare_conditions(camera_param, bboxes_3d_data, encoder_hidden_states, controlnet_cond)
        x = ops.pack_latents(ops.nchw_to_nhwc(sample.reshape(b * n_cam, c, h, w)), ControlNetEngine.CIN_PAD)
        t = _timesteps_f32(timestep, b, sample.device)
        if t.numel() == b and n_cam > 1:
            t = t.repeat_interleave(n_cam)  # 'b ... -> (b repeat) ...' (:840-841)
        n_res = len(arch.controlnet_residual_channels(self.arch_cfg)) + 1  # 12 down residuals + mid
        scale = ([float(v) * float(conditioning_scale) for v in torch.logspace(-1, 0, n_res)] if guess_mode
                 else float(conditioning_scale))
        down, mid, skips, xm = eng.forward(x, b * n_cam, h, w, t, cond["kv"], cond["lc"], cond["map"], scale)
        dt = sample.dtype
        down_nchw = [ops.nhwc_to_nchw(d, s.n, s.c, s.h, s.w, F32).to(dt) for d, s in zip(down, skips)]
        mid_nchw = ops.nhwc_to_nchw(mid, xm.n, xm.c, xm.h, xm.w, F32).to(dt)
        ctx = cond["ctx"].to(dt)
        if not return_dict:
            return (down_nchw, mid_nchw, ctx)
        return BEVControlNetOutput(down_block_res_samples=down_nchw, mid_block_res_sample=mid_nchw,
                                   encoder_hidden_states_with_cam=ctx)

    @classmethod
    def from_unet(cls, unet, **kwargs):
        """unet_addon_rawbox.py:414-475: copy the encoder configuration (and weights) of a UNet."""
        u = unet.arch_cfg
        model = cls(in_channels=u.in_channels, block_out_channels=u.block_out_channels,
                    down_block_types=u.down_block_types, layers_per_block=u.layers_per_block,
                    attention_head_dim=u.attention_head_dim, cross_attention_dim=u.cross_attention_dim,
                    norm_num_groups=u.norm_num_groups, norm_eps=u.norm_eps, **kwargs)
        own = model.state_dict()
        src = {k: v for k, v in unet.state_dict().items() if k in own and own[k].shape == v.shape}
        model.load_state_dict(src, strict=False)
        return model


class DecoderOutput:  # diffusers/models/vae.py:27-36
    def __init__(self, sample):
        self.sample = sample

    def __getitem__(self, i):
        return (self.sample,)[i]


class DiagonalGaussianDistribution:
    """diffusers/models/vae.py:397-416 over NCHW `parameters` (mean | logvar along the channels): `.mean`, `.logvar`
    (clamped to [-30, 20]), `.std`, `.var`, `.sample(generator)` = mean + std * randn_tensor(mean.shape), `.mode()`."""

    def __init__(self, parameters: torch.Tensor, deterministic: bool = False):
        self.parameters = parameters
        self.mean, self.logvar = torch.chunk(parameters, 2, dim=1)
        self.logvar = torch.clamp(self.logvar, -30.0, 20.0)
        self.deterministic = deterministic
        self.std = torch.exp(0.5 * self.logvar)
        self.var = torch.exp(self.logvar)
        if deterministic:
            self.var = self.std = torch.zeros_like(self.mean)

    def sample(self, generator: Optional[torch.Generator] = None) -> torch.Tensor:
        noise = randn_tensor(self.mean.shape, generator, self.parameters.device, self.parameters.dtype)
        return self.mean + self.std * noise

    def mode(self) -> torch.Tensor:
        return self.mean


def randn_tensor(shape, generator: Optional[torch.Generator], device, dtype=F32) -> torch.Tensor:
    """diffusers.utils.torch_utils.randn_tensor for one generator: drawn on the generator's device (a CPU generator
    feeding a CUDA tensor draws on the host and copies), so a seeded generator gives diffusers' draw."""
    device = torch.device(device)
    gen_dev = generator.device if generator is not None else device
    x = torch.randn(tuple(shape), generator=generator, device=gen_dev, dtype=dtype)
    return x.to(device)


@dataclass
class AutoencoderKLOutput:  # diffusers/models/autoencoder_kl.py:28-37
    latent_dist: DiagonalGaussianDistribution

    def __getitem__(self, i):
        return (self.latent_dist,)[i]


class AutoencoderKL(_B200Module):
    """diffusers' AutoencoderKL (models/autoencoder_kl.py) for the pipeline's `decode_latents` (pipeline_bev_controlnet.py:
    100-112) and, with `with_encoder=True`, for `encode` (the given-view demo's latents, demo/run_cond_on_view.py:80-86):
    same constructor kwargs and checkpoint key names, `.config.scaling_factor` and `.config.block_out_channels` as the
    pipeline reads them (pipeline_controlnet.py:130-179), `decode(z).sample`, `encode(x).latent_dist`.
    By default the module is the decoder half only (`decoder.*`, `post_quant_conv.*`; `encoder.*` / `quant_conv.*` of a
    full checkpoint are accepted and ignored) and `encode` raises.  `with_encoder=True` (kept in `.config`, so a saved
    config.json restores it) holds the full key set, loads it strictly and runs the encoder on the GPU too."""

    def __init__(self, with_encoder: bool = False, **kwargs):
        super().__init__()
        known, extra = _pick(arch.VaeConfig, dict(kwargs))
        cfg = arch.VaeConfig(**{k: (tuple(v) if isinstance(v, list) else v) for k, v in known.items()})
        if cfg.act_fn != "silu" or any(t != "UpDecoderBlock2D" for t in cfg.up_block_types):
            raise ValueError("only the SD-1.5 AutoencoderKL layout (UpDecoderBlock2D, silu) is implemented")
        self.with_encoder = bool(with_encoder)
        shapes = arch.vae_decoder_param_shapes(cfg)
        if self.with_encoder:
            if any(t != "DownEncoderBlock2D" for t in cfg.down_block_types):
                raise ValueError("only the SD-1.5 AutoencoderKL encoder layout (DownEncoderBlock2D, silu) is implemented")
            extra["with_encoder"] = True
            shapes = OrderedDict(list(arch.vae_encoder_param_shapes(cfg).items()) + list(shapes.items()))
        self._init_common(cfg, shapes, extra)
        self.training = False

    _OLD_ATTN = {"query": "to_q", "key": "to_k", "value": "to_v", "proj_attn": "to_out.0"}  # pre-0.17 checkpoint names

    def load_state_dict(self, state_dict, strict=True, **kw):
        sd = {}
        for k, v in state_dict.items():
            if not self.with_encoder and k.startswith(("encoder.", "quant_conv.")):
                continue
            parts = k.split(".")
            if "attentions" in parts and parts[-2] in self._OLD_ATTN:  # attention_processor.py:_from_deprecated_attn_block
                k = ".".join(parts[:-2] + [self._OLD_ATTN[parts[-2]], parts[-1]])
            sd[k] = v
        return super().load_state_dict(sd, strict=strict, **kw)

    use_cuda_graph = True  # decode_latents / encode_latents replay one captured graph per shape
    _decode_graphs: dict = {}
    _encode_graphs: dict = {}

    def engine(self) -> VaeDecoderEngine:
        """The decoder engine, or with_encoder the VaeEncoderEngine that also decodes (one packed-weight cache)."""
        eng = self._get_engine(VaeEncoderEngine if self.with_encoder else VaeDecoderEngine)
        if getattr(self, "_graphs_for", None) is not eng:  # weights changed -> engine rebuilt -> graphs stale
            self._decode_graphs, self._encode_graphs, self._graphs_for = {}, {}, eng
        return eng

    def _encoder_engine(self, x: torch.Tensor) -> VaeEncoderEngine:
        if not self.with_encoder:
            raise NotImplementedError("this AutoencoderKL holds the decoder only; build it with with_encoder=True "
                                      "(AutoencoderKL(..., with_encoder=True) or from_pretrained(..., with_encoder=True)) to encode")
        if x.shape[-3] != self.arch_cfg.in_channels or x.shape[-2] % 8 or x.shape[-1] % 8:
            raise ValueError(f"encode expects (..., {self.arch_cfg.in_channels}, H, W) images with H and W divisible by 8, "
                             f"got {tuple(x.shape)}")
        return self.engine()

    @torch.no_grad()
    def encode(self, x: torch.Tensor, return_dict: bool = True):
        """AutoencoderKL.encode (autoencoder_kl.py:160-171): NCHW images in [-1, 1] -> the posterior over the latents
        (DiagonalGaussianDistribution of fp32 NCHW (n, 2 * latent_channels, H/8, W/8) moments)."""
        eng = self._encoder_engine(x)
        n, _, h, w = x.shape
        c = self.arch_cfg.latent_channels
        mom = eng.encode(x.to(self.device))
        params = mom.view(n, h // 8, w // 8, -1)[..., : 2 * c].permute(0, 3, 1, 2).contiguous()
        posterior = DiagonalGaussianDistribution(params)
        return AutoencoderKLOutput(latent_dist=posterior) if return_dict else (posterior,)

    @torch.no_grad()
    def encode_latents(self, pixel_values: torch.Tensor, sample: bool = False,
                       generator: Optional[torch.Generator] = None) -> torch.Tensor:
        """The given-view demo's latents (demo/run_cond_on_view.py:80-86): (b, n_cam, 3, H, W) images in [-1, 1] ->
        fp32 (b, n_cam, latent_channels, H/8, W/8) = scaling_factor * posterior mean (or, with `sample`, a posterior
        sample drawn with `generator` like DiagonalGaussianDistribution.sample), on the module's device.  Each shape is
        one CUDA-graph replay; the sample's noise is drawn outside the graph into a resident buffer."""
        b, n_cam = pixel_values.shape[:2]
        x = pixel_values.reshape(b * n_cam, *pixel_values.shape[2:])
        eng = self._encoder_engine(x)
        n, _, hh, ww = x.shape
        h, w, c = hh // 8, ww // 8, self.arch_cfg.latent_channels
        scale = float(self.config["scaling_factor"])
        noise = randn_tensor((n, c, h, w), generator, self.device) if sample else None

        def run(xx, nz):
            return ops.latent_dist(eng.encode(xx), n, h, w, c, noise=nz, scale=scale)

        x = x.to(self.device)
        if not (self.use_cuda_graph and x.is_cuda):
            z = run(x, noise)
        else:
            key = (id(eng), n, hh, ww, x.dtype, sample)
            g = self._encode_graphs.get(key)
            if g is None:
                xin, nin = x.clone(), (noise.clone() if sample else None)
                run(xin, nin)  # eager once: sizes the scratch and the split-K workspace
                torch.cuda.synchronize()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    out = run(xin, nin)
                g = self._encode_graphs[key] = (graph, xin, nin, out)
            graph, xin, nin, out = g
            xin.copy_(x)
            if sample:
                nin.copy_(noise)
            graph.replay()
            z = out.clone()
        return z.reshape(b, n_cam, c, h, w)
    @torch.no_grad()
    def decode(self, z: torch.Tensor, return_dict: bool = True):
        """z: (n, 4, h, w) latents already divided by scaling_factor, as the pipeline passes them -> (n, 3, 8h, 8w)."""
        n, c, h, w = z.shape
        z_nhwc = z.to(F32).permute(0, 2, 3, 1).contiguous().view(-1, c)
        img = self.engine().decode(z_nhwc, n, h, w).permute(0, 3, 1, 2).to(z.dtype)
        return DecoderOutput(img) if return_dict else (img,)

    @torch.no_grad()
    def decode_latents(self, latents: torch.Tensor) -> torch.Tensor:
        """StableDiffusionBEVControlNetPipeline.decode_latents (:100-112) on (b, n_cam, 4, h, w) latents, with the
        1/scaling_factor, image/2+0.5 and clamp folded into the first and last convolution: (b, n_cam, 8h, 8w, 3) fp32."""
        b, n_cam, c, h, w = latents.shape
        z = latents.to(self.device, F32).permute(0, 1, 3, 4, 2).contiguous().view(-1, c)
        eng = self.engine()
        run = lambda zz: eng.decode(zz, b * n_cam, h, w, scale=1.0 / self.config["scaling_factor"], to_unit_range=True)
        if not (self.use_cuda_graph and z.is_cuda):
            img = run(z)
        else:
            # the decode of a given shape is one CUDA graph on resident input / output buffers (eager once to size scratch)
            key = (id(eng), b * n_cam, h, w)
            g = self._decode_graphs.get(key)
            if g is None:
                zin = z.clone()
                run(zin)
                torch.cuda.synchronize()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    out = run(zin)
                g = self._decode_graphs[key] = (graph, zin, out)
            graph, zin, out = g
            zin.copy_(z)
            graph.replay()
            img = out.clone()
        return img.reshape(b, n_cam, *img.shape[1:])
