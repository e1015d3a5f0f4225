"""Layer enumeration of the two networks on the hot path, derived from their config alone.

Produces (a) the exact parameter names + shapes of the reference checkpoints, so our modules load
`UNet2DConditionModelMultiview` / `BEVControlNetModel` state dicts unchanged, and (b) a structural "program"
(list of resnet / transformer / sampler steps) that both the CUDA engine and the CPU oracle walk.

Reference structure: diffusers/models/unet_2d_condition.py:161-505 (constructor), unet_2d_blocks.py:794-941,
944-1027, 478-584, 1886-2030, 2033-2111; magicdrive/networks/unet_2d_condition_multiview.py:123-235;
magicdrive/networks/unet_addon_rawbox.py:33-286; bbox_embedder.py:32-108; map_embedder.py:20-64.
"""
from collections import OrderedDict
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

DEFAULT_NEIGHBORS = {0: [5, 1], 1: [0, 2], 2: [1, 3], 3: [2, 4], 4: [3, 5], 5: [4, 0]}


@dataclass
class UNetConfig:
    in_channels: int = 4
    out_channels: int = 4
    block_out_channels: Tuple[int, ...] = (320, 640, 1280, 1280)
    down_block_types: Tuple[str, ...] = ("CrossAttnDownBlock2D", "CrossAttnDownBlock2D", "CrossAttnDownBlock2D",
                                         "DownBlock2D")
    up_block_types: Tuple[str, ...] = ("UpBlock2D", "CrossAttnUpBlock2D", "CrossAttnUpBlock2D", "CrossAttnUpBlock2D")
    layers_per_block: int = 2
    attention_head_dim: int = 8  # diffusers 0.17.1 passes this as the NUMBER of heads (unet_2d_blocks.py:842-845)
    cross_attention_dim: int = 768
    norm_num_groups: int = 32
    norm_eps: float = 1e-5
    flip_sin_to_cos: bool = True
    freq_shift: int = 0
    neighboring_view_pair: Dict[int, List[int]] = field(default_factory=lambda: dict(DEFAULT_NEIGHBORS))
    neighboring_attn_type: str = "add"
    zero_module_type: str = "zero_linear"
    sample_size: Optional[int] = 64

    @property
    def time_embed_dim(self):
        return self.block_out_channels[0] * 4

    @property
    def n_cam(self):
        return len(self.neighboring_view_pair)

    @property
    def multiview(self) -> bool:
        """False (no neighbouring_view_pair) = the stock diffusers UNet2DConditionModel: BasicTransformerBlock without the
        cross-view attention (BASELINE.json configs[0]: 1-view SD-1.5 UNet, text-only conditioning)."""
        return len(self.neighboring_view_pair) > 0


@dataclass
class ControlNetConfig:
    in_channels: int = 4
    block_out_channels: Tuple[int, ...] = (320, 640, 1280, 1280)
    down_block_types: Tuple[str, ...] = ("CrossAttnDownBlock2D", "CrossAttnDownBlock2D", "CrossAttnDownBlock2D",
                                         "DownBlock2D")
    layers_per_block: int = 2
    attention_head_dim: int = 8
    cross_attention_dim: int = 768
    norm_num_groups: int = 32
    norm_eps: float = 1e-5
    flip_sin_to_cos: bool = True
    freq_shift: int = 0
    # BEV specifics (configs/model/SDv1.5mv_rawbox.yaml)
    uncond_cam_in_dim: Tuple[int, int] = (3, 7)
    camera_in_dim: int = 189
    camera_out_dim: int = 768
    map_size: Tuple[int, int, int] = (8, 200, 200)
    conditioning_embedding_out_channels: Tuple[int, ...] = (16, 32, 96, 256)
    # map_embedder_cls BEVControlNetConditioningEmbeddingPlus (configs/exp/272x736.yaml:16-22): (h, w) of its AdaptiveAvgPool2d,
    # i.e. the latent grid the BEV-map embedding is pooled to; None = the plain BEVControlNetConditioningEmbedding
    map_embedding_size: Optional[Tuple[int, int]] = None
    cam_num_freqs: int = 4
    # bbox embedder (ContinuousBBoxWithTextEmbedding, mode all-xyz, minmax_normalize False)
    bbox_n_classes: int = 10
    bbox_class_token_dim: int = 768
    bbox_num_freqs: int = 4
    bbox_proj_dims: Tuple[int, ...] = (768, 512, 512, 768)
    bbox_points: int = 8

    @property
    def time_embed_dim(self):
        return self.block_out_channels[0] * 4


# ------------------------------------------------------------------------------------------ structural program
@dataclass
class ResnetSpec:
    prefix: str
    cin: int
    cout: int
    skip_c: int = 0  # channels taken from the skip connection (concatenated AFTER the running tensor)

    @property
    def shortcut(self):
        return self.cin != self.cout


@dataclass
class TransformerSpec:
    prefix: str
    c: int
    heads: int
    multiview: bool


@dataclass
class SamplerSpec:
    prefix: str
    c: int
    kind: str  # "down" (3x3 stride 2 pad 1) or "up" (nearest resize + 3x3)


@dataclass
class BlockSpec:
    name: str
    layers: List[Tuple[ResnetSpec, Optional[TransformerSpec]]]
    sampler: Optional[SamplerSpec]


def _heads(cfg, i):
    a = cfg.attention_head_dim
    return a[i] if isinstance(a, (tuple, list)) else a


def down_blocks(cfg, multiview: bool) -> List[BlockSpec]:
    blocks = []
    out_c = cfg.block_out_channels[0]
    for i, typ in enumerate(cfg.down_block_types):
        in_c, out_c = out_c, cfg.block_out_channels[i]
        final = i == len(cfg.block_out_channels) - 1
        layers = []
        for j in range(cfg.layers_per_block):
            rs = ResnetSpec(f"down_blocks.{i}.resnets.{j}", in_c if j == 0 else out_c, out_c)
            tr = None
            if typ == "CrossAttnDownBlock2D":
                tr = TransformerSpec(f"down_blocks.{i}.attentions.{j}", out_c, _heads(cfg, i), multiview)
            layers.append((rs, tr))
        samp = None if final else SamplerSpec(f"down_blocks.{i}.downsamplers.0.conv", out_c, "down")
        blocks.append(BlockSpec(f"down_blocks.{i}", layers, samp))
    return blocks


def mid_block(cfg, multiview: bool):
    c = cfg.block_out_channels[-1]
    return (ResnetSpec("mid_block.resnets.0", c, c),
            TransformerSpec("mid_block.attentions.0", c, _heads(cfg, len(cfg.block_out_channels) - 1), multiview),
            ResnetSpec("mid_block.resnets.1", c, c))


def up_blocks(cfg: UNetConfig) -> List[BlockSpec]:
    blocks = []
    rev = list(reversed(cfg.block_out_channels))
    a = cfg.attention_head_dim
    rev_heads = list(reversed(a)) if isinstance(a, (tuple, list)) else [a] * len(rev)
    out_c = rev[0]
    n = len(cfg.up_block_types)
    for i, typ in enumerate(cfg.up_block_types):
        prev_out = out_c
        out_c = rev[i]
        in_c = rev[min(i + 1, len(rev) - 1)]
        final = i == n - 1
        layers = []
        for j in range(cfg.layers_per_block + 1):
            skip_c = in_c if j == cfg.layers_per_block else out_c
            run_c = prev_out if j == 0 else out_c
            rs = ResnetSpec(f"up_blocks.{i}.resnets.{j}", run_c + skip_c, out_c, skip_c=skip_c)
            tr = None
            if typ == "CrossAttnUpBlock2D":
                tr = TransformerSpec(f"up_blocks.{i}.attentions.{j}", out_c, rev_heads[i], cfg.multiview)
            layers.append((rs, tr))
        samp = None if final else SamplerSpec(f"up_blocks.{i}.upsamplers.0.conv", out_c, "up")
        blocks.append(BlockSpec(f"up_blocks.{i}", layers, samp))
    return blocks


# ------------------------------------------------------------------------------------------ parameter shapes
def _conv(sh, p, co, ci, k, bias=True):
    sh[p + ".weight"] = (co, ci, k, k)
    if bias:
        sh[p + ".bias"] = (co,)


def _lin(sh, p, co, ci, bias=True):
    sh[p + ".weight"] = (co, ci)
    if bias:
        sh[p + ".bias"] = (co,)


def _norm(sh, p, c):
    sh[p + ".weight"] = (c,)
    sh[p + ".bias"] = (c,)


def _resnet_shapes(sh, rs: ResnetSpec, temb):
    _norm(sh, rs.prefix + ".norm1", rs.cin)
    _conv(sh, rs.prefix + ".conv1", rs.cout, rs.cin, 3)
    _lin(sh, rs.prefix + ".time_emb_proj", rs.cout, temb)
    _norm(sh, rs.prefix + ".norm2", rs.cout)
    _conv(sh, rs.prefix + ".conv2", rs.cout, rs.cout, 3)
    if rs.shortcut:
        _conv(sh, rs.prefix + ".conv_shortcut", rs.cout, rs.cin, 1)


def _attn_shapes(sh, p, c, kv):
    _lin(sh, p + ".to_q", c, c, bias=False)
    _lin(sh, p + ".to_k", c, kv, bias=False)
    _lin(sh, p + ".to_v", c, kv, bias=False)
    _lin(sh, p + ".to_out.0", c, c)


def _transformer_shapes(sh, tr: TransformerSpec, cross):
    p = tr.prefix
    _norm(sh, p + ".norm", tr.c)
    _conv(sh, p + ".proj_in", tr.c, tr.c, 1)
    b = p + ".transformer_blocks.0"
    _norm(sh, b + ".norm1", tr.c)
    _attn_shapes(sh, b + ".attn1", tr.c, tr.c)
    _norm(sh, b + ".norm2", tr.c)
    _attn_shapes(sh, b + ".attn2", tr.c, cross)
    _norm(sh, b + ".norm3", tr.c)
    _lin(sh, b + ".ff.net.0.proj", 8 * tr.c, tr.c)
    _lin(sh, b + ".ff.net.2", tr.c, 4 * tr.c)
    if tr.multiview:
        _norm(sh, b + ".norm4", tr.c)
        _attn_shapes(sh, b + ".attn4", tr.c, tr.c)
        _lin(sh, b + ".connector", tr.c, tr.c)
    _conv(sh, p + ".proj_out", tr.c, tr.c, 1)


def _encoder_shapes(sh, cfg, multiview):
    c0 = cfg.block_out_channels[0]
    temb = cfg.time_embed_dim
    _conv(sh, "conv_in", c0, cfg.in_channels, 3)
    _lin(sh, "time_embedding.linear_1", temb, c0)
    _lin(sh, "time_embedding.linear_2", temb, temb)
    for blk in down_blocks(cfg, multiview):
        for rs, tr in blk.layers:
            _resnet_shapes(sh, rs, temb)
            if tr is not None:
                _transformer_shapes(sh, tr, cfg.cross_attention_dim)
        if blk.sampler is not None:
            _conv(sh, blk.sampler.prefix, blk.sampler.c, blk.sampler.c, 3)
    r0, tr, r1 = mid_block(cfg, multiview)
    _resnet_shapes(sh, r0, temb)
    _transformer_shapes(sh, tr, cfg.cross_attention_dim)
    _resnet_shapes(sh, r1, temb)


def unet_param_shapes(cfg: UNetConfig) -> "OrderedDict[str, tuple]":
    sh = OrderedDict()
    _encoder_shapes(sh, cfg, cfg.multiview)
    temb = cfg.time_embed_dim
    for blk in up_blocks(cfg):
        for rs, tr in blk.layers:
            _resnet_shapes(sh, rs, temb)
            if tr is not None:
                _transformer_shapes(sh, tr, cfg.cross_attention_dim)
        if blk.sampler is not None:
            _conv(sh, blk.sampler.prefix, blk.sampler.c, blk.sampler.c, 3)
    _norm(sh, "conv_norm_out", cfg.block_out_channels[0])
    _conv(sh, "conv_out", cfg.out_channels, cfg.block_out_channels[0], 3)
    return sh


def map_encoder_layers(cfg: ControlNetConfig):
    """(name, cin, cout, stride(h,w), pad(h,w)) of BEVControlNetConditioningEmbedding (map_embedder.py:28-64) or, with
    cfg.map_embedding_size set, of BEVControlNetConditioningEmbeddingPlus (:79-126: all pads 1, first strided block stride 1,
    and an AdaptiveAvgPool2d(cfg.map_embedding_size) as `blocks.{last}` ahead of conv_out -- it has no parameters and is
    not listed here; engine / oracle insert it)."""
    ch = cfg.conditioning_embedding_out_channels
    plus = cfg.map_embedding_size is not None
    layers = [("controlnet_cond_embedding.conv_in", cfg.map_size[0], ch[0], (1, 1), (1, 1))]
    bi = 0
    for i in range(len(ch) - 2):
        layers.append((f"controlnet_cond_embedding.blocks.{bi}", ch[i], ch[i], (1, 1), (1, 1)))
        if plus:
            st = (1, 1) if i == 0 else (2, 2)
            layers.append((f"controlnet_cond_embedding.blocks.{bi + 1}", ch[i], ch[i + 1], st, (1, 1)))
        else:
            layers.append((f"controlnet_cond_embedding.blocks.{bi + 1}", ch[i], ch[i + 1], (2, 2), (2, 1)))
        bi += 2
    layers.append((f"controlnet_cond_embedding.blocks.{bi}", ch[-2], ch[-2], (1, 1), (1, 1) if plus else (2, 1)))
    layers.append((f"controlnet_cond_embedding.blocks.{bi + 1}", ch[-2], ch[-1], (2, 1), (1, 1) if plus else (2, 1)))
    layers.append(("controlnet_cond_embedding.conv_out", ch[-1], cfg.block_out_channels[0], (1, 1), (1, 1)))
    return layers


def controlnet_residual_channels(cfg) -> List[int]:
    """Channels of the 1 + sum(layers + sampler) skip tensors (unet_addon_rawbox.py:221-259)."""
    chans = [cfg.block_out_channels[0]]
    for i, _ in enumerate(cfg.down_block_types):
        c = cfg.block_out_channels[i]
        chans += [c] * cfg.layers_per_block
        if i != len(cfg.block_out_channels) - 1:
            chans.append(c)
    return chans


def controlnet_param_shapes(cfg: ControlNetConfig) -> "OrderedDict[str, tuple]":
    sh = OrderedDict()
    _lin(sh, "cam2token", cfg.camera_out_dim, cfg.camera_in_dim)
    sh["uncond_cam.weight"] = (1, cfg.uncond_cam_in_dim[0] * cfg.uncond_cam_in_dim[1])
    _encoder_shapes(sh, cfg, False)
    for name, ci, co, _, _ in map_encoder_layers(cfg):
        _conv(sh, name, co, ci, 3)
    fdim = 3 * (1 + 2 * cfg.bbox_num_freqs) * cfg.bbox_points
    pd = cfg.bbox_proj_dims
    _lin(sh, "bbox_embedder.bbox_proj", pd[0], fdim)
    _lin(sh, "bbox_embedder.second_linear.0", pd[1], pd[0] + cfg.bbox_class_token_dim)
    _lin(sh, "bbox_embedder.second_linear.2", pd[2], pd[1])
    _lin(sh, "bbox_embedder.second_linear.4", pd[3], pd[2])
    sh["bbox_embedder._class_tokens"] = (cfg.bbox_n_classes, cfg.bbox_class_token_dim)  # buffer
    sh["bbox_embedder.null_class_feature"] = (cfg.bbox_class_token_dim,)
    sh["bbox_embedder.null_pos_feature"] = (fdim,)
    for i, c in enumerate(controlnet_residual_channels(cfg)):
        _conv(sh, f"controlnet_down_blocks.{i}", c, c, 1)
    _conv(sh, "controlnet_mid_block", cfg.block_out_channels[-1], cfg.block_out_channels[-1], 1)
    return sh


# ------------------------------------------------------------------------------------------ VAE decoder (SURVEY §8 f2)
@dataclass
class VaeConfig:
    """AutoencoderKL config of SD-1.5 (third_party/diffusers/src/diffusers/models/autoencoder_kl.py:66-82); only the
    decoder half is on the path (pipeline_bev_controlnet.py:100-112)."""
    in_channels: int = 3
    out_channels: int = 3
    down_block_types: Tuple[str, ...] = ("DownEncoderBlock2D",) * 4
    up_block_types: Tuple[str, ...] = ("UpDecoderBlock2D",) * 4
    block_out_channels: Tuple[int, ...] = (128, 256, 512, 512)
    layers_per_block: int = 2
    act_fn: str = "silu"
    latent_channels: int = 4
    norm_num_groups: int = 32
    sample_size: int = 512
    scaling_factor: float = 0.18215


def vae_decoder_blocks(cfg: VaeConfig):
    """[(prefix, [(resnet prefix, cin, cout)], upsampler prefix or None)] of Decoder.up_blocks (vae.py:193-219)."""
    rev = list(reversed(cfg.block_out_channels))
    blocks, out_c = [], rev[0]
    for i in range(len(rev)):
        prev, out_c = out_c, rev[i]
        res = [(f"decoder.up_blocks.{i}.resnets.{j}", prev if j == 0 else out_c, out_c) for j in range(cfg.layers_per_block + 1)]
        up = None if i == len(rev) - 1 else f"decoder.up_blocks.{i}.upsamplers.0.conv"
        blocks.append((f"decoder.up_blocks.{i}", res, up))
    return blocks


def _vae_resnet(sh, p, ci, co):
    """ResnetBlock2D without a time embedding (resnet.py:525-589, temb_channels=None)."""
    _norm(sh, p + ".norm1", ci)
    _conv(sh, p + ".conv1", co, ci, 3)
    _norm(sh, p + ".norm2", co)
    _conv(sh, p + ".conv2", co, co, 3)
    if ci != co:
        _conv(sh, p + ".conv_shortcut", co, ci, 1)


def _vae_mid_block(sh, p, c):
    """UNetMidBlock2D of the VAE: single-head attention, then its two resnets (unet_2d_blocks.py:395-473)."""
    a = p + ".attentions.0"
    _norm(sh, a + ".group_norm", c)
    for n in ("to_q", "to_k", "to_v", "to_out.0"):
        _lin(sh, f"{a}.{n}", c, c)
    _vae_resnet(sh, p + ".resnets.0", c, c)
    _vae_resnet(sh, p + ".resnets.1", c, c)


def vae_decoder_param_shapes(cfg: VaeConfig) -> "OrderedDict[str, tuple]":
    """Decoder + post_quant_conv keys of AutoencoderKL.state_dict() (vae.py:152-225, autoencoder_kl.py:107-108)."""
    sh: "OrderedDict[str, tuple]" = OrderedDict()
    c_mid = cfg.block_out_channels[-1]
    _conv(sh, "decoder.conv_in", c_mid, cfg.latent_channels, 3)
    for _, resnets, up in vae_decoder_blocks(cfg):
        for p, ci, co in resnets:
            _vae_resnet(sh, p, ci, co)
        if up:
            _conv(sh, up, resnets[-1][2], resnets[-1][2], 3)
    _vae_mid_block(sh, "decoder.mid_block", c_mid)
    _norm(sh, "decoder.conv_norm_out", cfg.block_out_channels[0])
    _conv(sh, "decoder.conv_out", cfg.out_channels, cfg.block_out_channels[0], 3)
    _conv(sh, "post_quant_conv", cfg.latent_channels, cfg.latent_channels, 1)
    return sh


def vae_encoder_blocks(cfg: VaeConfig):
    """[(prefix, [(resnet prefix, cin, cout)], downsampler conv prefix or None)] of Encoder.down_blocks: one
    DownEncoderBlock2D per level with a padding-0 Downsample2D on every level but the last (vae.py:62-82,
    unet_2d_blocks.py:1030-1087)."""
    blocks, out_c = [], cfg.block_out_channels[0]
    for i, c in enumerate(cfg.block_out_channels):
        prev, out_c = out_c, c
        res = [(f"encoder.down_blocks.{i}.resnets.{j}", prev if j == 0 else out_c, out_c) for j in range(cfg.layers_per_block)]
        down = None if i == len(cfg.block_out_channels) - 1 else f"encoder.down_blocks.{i}.downsamplers.0.conv"
        blocks.append((f"encoder.down_blocks.{i}", res, down))
    return blocks


def vae_encoder_param_shapes(cfg: VaeConfig) -> "OrderedDict[str, tuple]":
    """Encoder + quant_conv keys of AutoencoderKL.state_dict() (vae.py:39-97 with double_z, autoencoder_kl.py:95-106)."""
    sh: "OrderedDict[str, tuple]" = OrderedDict()
    c_mid = cfg.block_out_channels[-1]
    _conv(sh, "encoder.conv_in", cfg.block_out_channels[0], cfg.in_channels, 3)
    for _, resnets, down in vae_encoder_blocks(cfg):
        for p, ci, co in resnets:
            _vae_resnet(sh, p, ci, co)
        if down:
            _conv(sh, down, resnets[-1][2], resnets[-1][2], 3)
    _vae_mid_block(sh, "encoder.mid_block", c_mid)
    _norm(sh, "encoder.conv_norm_out", c_mid)
    _conv(sh, "encoder.conv_out", 2 * cfg.latent_channels, c_mid, 3)
    _conv(sh, "quant_conv", 2 * cfg.latent_channels, 2 * cfg.latent_channels, 1)
    return sh


BUFFER_KEYS = {"bbox_embedder._class_tokens"}


# ------------------------------------------------------------------------------------------ deterministic weights
def synthetic_state_dict(shapes, seed: int = 0, scale: float = 1.0):
    """Name-keyed deterministic weights (numpy Philox per tensor name) so that the reference model built in the
    oracle container and our model on the GPU box hold bit-identical fp32 parameters without shipping them.
    Every tensor is non-zero: the reference zero-initialises `connector`, the ControlNet 1x1 convs and the map
    encoder's conv_out (controlnet.py:585-588), which would hide cross-view / ControlNet bugs."""
    import zlib

    import numpy as np
    import torch

    def make(item):
        name, shape = item
        rng = np.random.Generator(np.random.Philox(key=(seed << 32) + zlib.crc32(name.encode())))
        if name.endswith(".weight") and len(shape) >= 2:
            fan_in = int(np.prod(shape[1:]))
            # the camera / box encoders see raw metric inputs (fx ~ 1.27e3 px, box corners +-50 m); a trained
            # checkpoint keeps their tokens O(1-10) like the CLIP tokens beside them, so do the synthetic weights
            # (otherwise one token saturates every conditioning softmax and bf16 parity becomes a coin flip)
            gain = {"cam2token.weight": 0.02, "bbox_embedder.bbox_proj.weight": 0.1}.get(name, 1.0)
            a = rng.standard_normal(shape, dtype=np.float32) * (gain * scale / np.sqrt(fan_in))
        elif name.endswith(".weight"):  # norm gains
            a = 1.0 + 0.1 * rng.standard_normal(shape, dtype=np.float32)
        elif "_class_tokens" in name:
            a = rng.standard_normal(shape, dtype=np.float32)
        else:  # biases, null features
            a = 0.05 * rng.standard_normal(shape, dtype=np.float32)
        return name, torch.from_numpy(np.ascontiguousarray(a.astype(np.float32)))

    # one independent Philox stream per tensor name: order- and thread-count-independent, so the tensors are generated
    # in parallel (numpy releases the GIL while filling)
    import os
    from concurrent.futures import ThreadPoolExecutor
    items = list(shapes.items())
    with ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 1)) as ex:
        sd = OrderedDict(ex.map(make, items))
    return sd
