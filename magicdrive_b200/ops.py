"""torch.Tensor-facing wrappers of the C-ABI operators.

torch is plumbing only: it owns device memory and the CUDA stream; every function here forwards raw pointers to
`libmagicdrive_b200.so` and raises if the library / a CUDA device is unavailable (no CPU or eager fallback).
Feature maps are NHWC bf16 ("channels innermost") everywhere; a token matrix [tokens, C] is the same layout.

One process drives ONE device (the launch contract: one process per GPU): the module-level workspace slot / launch counter and the
library's cached device attributes (SM count, per-kernel shared-memory opt-ins) are per process, not per device, and not thread-safe.
"""
import ctypes as C
import contextlib
import os
from typing import Optional

import torch

from . import _lib
from ._lib import GemmDesc, check

BF16 = torch.bfloat16
F32 = torch.float32

GEMM_VARIANT = int(os.environ.get('MDB_GEMM_VARIANT', '0'))  # A/B hook: mdb_gemm_desc.kernel_variant (2 = single-CTA kernel, 3 = CTA pairs)
_launches = 0  # kernels launched through this module (bench.py reports it as gpu_launches)
_profile = None  # when a list: (kind, algorithmic flops, start event, end event) per tensor-core launch


def start_profile():
    """Bracket every tensor-core launch with CUDA events on the launching stream (eager mode only)."""
    global _profile
    _profile = []


def stop_profile(with_info: bool = False):
    global _profile
    rec, _profile = _profile, None
    torch.cuda.synchronize()
    if with_info:
        return [(k, f, a.elapsed_time(b) * 1e-3, info) for k, f, a, b, info in rec]
    return [(k, f, a.elapsed_time(b) * 1e-3) for k, f, a, b, _ in rec]


def _prof_begin():
    if _profile is None:
        return None
    e = torch.cuda.Event(enable_timing=True)
    e.record()
    return e


def _prof_end(kind, flops, e0, info=""):
    if e0 is not None:
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record()
        _profile.append((kind, flops, e0, e1, info))


def launch_count() -> int:
    return _launches


def reset_launch_count():
    global _launches
    _launches = 0


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.MdbError("magicdrive_b200 operators need CUDA tensors; there is no CPU fallback")


_ws = {}
_ws_slot = 0


class workspace_slot:
    """Select which split-K scratch buffer the enclosed launches use (slot 1 = the concurrent ControlNet stream)."""

    def __init__(self, slot):
        self.slot = slot

    def __enter__(self):
        global _ws_slot
        self.prev, _ws_slot = _ws_slot, self.slot

    def __exit__(self, *a):
        global _ws_slot
        _ws_slot = self.prev


def workspace(nbytes: int, device) -> torch.Tensor:
    """Per-device scratch (split-K partials); grown on demand outside CUDA-graph capture."""
    # one scratch per (device, slot): split-K GEMMs may run concurrently on the ControlNet / UNet streams
    key = (device.index if device.index is not None else torch.cuda.current_device(), _ws_slot)
    buf = _ws.get(key)
    if buf is None or buf.numel() < nbytes:
        if torch.cuda.is_current_stream_capturing():
            raise _lib.MdbError("workspace must be sized before CUDA-graph capture (run one eager step first)")
        buf = torch.empty(max(nbytes, 64 << 20), dtype=torch.uint8, device=device)
        _ws[key] = buf
    return buf


class RowStats:
    """Per-row partial (sum, sum of squares) of a bf16 [rows, C] tensor, fp32 [rows, parts, 2], written by the epilogue of
    the GEMM that produced the tensor and consumed by a GEMM with a folded LayerNorm."""

    def __init__(self, data: torch.Tensor, parts: int):
        self.data, self.parts = data, parts


def gemm_conv(a0: torch.Tensor, w: torch.Tensor, *, n_img: int, h_in: int, w_in: int, c0: int, lda0: int,
              n_out: int, taps: int = 1, stride: int = 1, pad: int = 0, h_out: Optional[int] = None,
              w_out: Optional[int] = None, a1: Optional[torch.Tensor] = None, c1: int = 0, lda1: int = 0,
              bias: Optional[torch.Tensor] = None, rowbias: Optional[torch.Tensor] = None,
              residual: Optional[torch.Tensor] = None, ldr: int = 0, out: Optional[torch.Tensor] = None,
              ldo: Optional[int] = None, out_f32: bool = False, out_scale: float = 1.0, geglu: bool = False,
              force_block_n: int = 0, force_splits: int = 0, allow_split_k: bool = True,
              kernel_variant: int = 0, trace: Optional[torch.Tensor] = None, debug_flags: int = 0,
              ln: Optional["RowStats"] = None, ln_colsum: Optional[torch.Tensor] = None, ln_eps: float = 1e-5,
              emit_stats: bool = False):
    """tcgen05 GEMM / implicit-GEMM conv (mdb_gemm_conv).  `a0` (and `a1`) are NHWC bf16 buffers whose pixel
    stride is lda* elements; `w` is bf16 [n_out, taps*taps*(c0+c1)].
    ln / ln_colsum: fold a LayerNorm of the rows of `a0` into this GEMM (`ln` = the RowStats the producer of `a0`
    emitted, `w` pre-multiplied by gamma, `bias` = beta-term + bias).  emit_stats: also return the RowStats of the
    output rows -> (out, RowStats)."""
    global _launches
    _need_cuda(a0, w)
    if h_out is None:
        h_out = (h_in + 2 * pad - taps) // stride + 1
    if w_out is None:
        w_out = (w_in + 2 * pad - taps) // stride + 1
    pixels = n_img * h_out * w_out
    width = n_out // 2 if geglu else n_out
    if out is None:
        out = torch.empty((pixels, width), dtype=F32 if out_f32 else BF16, device=a0.device)
        ldo = width
    elif ldo is None:
        ldo = out.stride(0) if out.dim() == 2 else out.shape[-1]
    d = GemmDesc()
    d.a0, d.a1 = _ptr(a0), _ptr(a1)
    d.c0, d.lda0, d.c1, d.lda1 = c0, lda0, c1, lda1
    d.n_img, d.h_in, d.w_in = n_img, h_in, w_in
    d.w, d.n_out = _ptr(w), n_out
    d.taps_h = d.taps_w = taps
    d.stride, d.pad_h, d.pad_w = stride, pad, pad
    d.h_out, d.w_out = h_out, w_out
    d.bias = _ptr(bias)
    d.rowbias = _ptr(rowbias)
    d.rowbias_ld = (rowbias.stride(0) if rowbias.shape[0] > 1 else 0) if rowbias is not None else 0  # 1 row = shared by all images
    d.residual, d.ldr = _ptr(residual), ldr
    d.out, d.ldo, d.out_is_f32, d.out_scale = _ptr(out), ldo, int(out_f32), float(out_scale)
    d.epi_mode = 1 if geglu else 0
    if allow_split_k and not geglu:
        ws = workspace(64 << 20, a0.device)
        d.workspace, d.workspace_bytes = ws.data_ptr(), ws.numel()
    else:
        d.workspace, d.workspace_bytes = None, 0
    d.force_block_n, d.force_splits = force_block_n, force_splits
    d.kernel_variant = kernel_variant or GEMM_VARIANT
    d.trace = _ptr(trace)
    d.debug_flags = debug_flags
    L = _lib.lib()
    if ln is not None:
        d.ln_stats, d.ln_parts, d.ln_eps, d.ln_colsum = ln.data.data_ptr(), ln.parts, float(ln_eps), _ptr(ln_colsum)
    stats = None
    if emit_stats:
        d.stats_out = 1  # any non-null value: the planner only asks whether statistics are wanted
        parts = L.mdb_gemm_conv_stats_parts(C.byref(d))
        if parts <= 0:
            check(parts, "mdb_gemm_conv_stats_parts")
        stats = RowStats(torch.empty((pixels, parts, 2), dtype=F32, device=a0.device), parts)
        d.stats_out = stats.data.data_ptr()
    e0 = _prof_begin()
    check(L.mdb_gemm_conv(C.byref(d), _stream()), "mdb_gemm_conv")
    _prof_end("gemm_conv", 2.0 * pixels * n_out * taps * taps * (c0 + c1), e0,
              f"M={pixels} N={n_out} K={taps * taps * (c0 + c1)} img={n_img}x{h_out}x{w_out} taps={taps} s={stride} "
              f"geglu={int(geglu)} res={int(residual is not None)}")
    _launches += L.mdb_gemm_conv_launches(C.byref(d))
    return (out, stats) if emit_stats else out


@contextlib.contextmanager
def pdl_region(enabled: bool = True):
    """Launch the kernels issued inside with programmatic dependent launch (mdb_set_pdl): use around single-stream
    stretches only -- with two concurrent branches the early-scheduled dependents take SMs from the other branch."""
    lib = _lib.lib()
    old = lib.mdb_set_pdl(int(enabled))
    try:
        yield
    finally:
        lib.mdb_set_pdl(old)


def linear(x: torch.Tensor, w: torch.Tensor, bias=None, residual=None, out=None, ldo=None, geglu=False,
           out_f32=False, out_scale=1.0, **kw):
    """Token GEMM: x [M, K] bf16 (row stride may exceed K), w [N, K] bf16."""
    m, k = x.shape
    return gemm_conv(x, w, n_img=1, h_in=1, w_in=m, c0=k, lda0=x.stride(0), n_out=w.shape[0], bias=bias,
                     residual=residual, ldr=(residual.stride(0) if residual is not None else 0), out=out, ldo=ldo,
                     geglu=geglu, out_f32=out_f32, out_scale=out_scale, **kw)


def conv_direct(x, wgt, bias, *, n, h, w, cin, cout, k, stride=(1, 1), pad=(1, 1), silu=False, residual=None,
                out_f32=False):
    global _launches
    _need_cuda(x, wgt)
    ho = (h + 2 * pad[0] - k) // stride[0] + 1
    wo = (w + 2 * pad[1] - k) // stride[1] + 1
    out = torch.empty((n, ho, wo, cout), dtype=F32 if out_f32 else BF16, device=x.device)
    check(_lib.lib().mdb_conv_direct(_ptr(x), int(x.dtype == F32), n, h, w, cin, _ptr(wgt), _ptr(bias), cout, k, k,
                                     stride[0], stride[1], pad[0], pad[1], ho, wo, int(silu), _ptr(residual),
                                     _ptr(out), int(out_f32), _stream()), "mdb_conv_direct")
    _launches += 1
    return out


def groupnorm(x0, c0, ld0, n_img, hw, gamma, beta, eps, silu, x1=None, c1=0, ld1=0, groups=32):
    global _launches
    _need_cuda(x0)
    out = torch.empty((n_img * hw, c0 + c1), dtype=BF16, device=x0.device)
    stats = torch.empty((max(n_img, 160) * groups * 2,), dtype=F32, device=x0.device)  # scratch: per-(image | CTA run) group partials
    check(_lib.lib().mdb_groupnorm(_ptr(x0), c0, ld0, _ptr(x1), c1, ld1, n_img, hw, groups, float(eps), _ptr(gamma),
                                   _ptr(beta), int(silu), _ptr(out), c0 + c1, _ptr(stats), _stream()), "mdb_groupnorm")
    _launches += 2 if os.environ.get("MDB_GN_TWO_KERNEL") else 1  # one fused kernel (A/B: stats + apply)
    return out


def layernorm(x, gamma, beta, eps=1e-5):
    global _launches
    _need_cuda(x)
    rows, c = x.shape
    out = torch.empty((rows, c), dtype=BF16, device=x.device)
    check(_lib.lib().mdb_layernorm(_ptr(x), rows, c, x.stride(0), _ptr(gamma), _ptr(beta), float(eps), _ptr(out), c,
                                   _stream()), "mdb_layernorm")
    _launches += 1
    return out


def softmax_rows(s, cols: int, cols_out: int):
    """fp32 scores [rows, >=cols] -> bf16 probabilities [rows, cols_out], columns >= cols zero."""
    global _launches
    _need_cuda(s)
    out = torch.empty((s.shape[0], cols_out), dtype=BF16, device=s.device)
    check(_lib.lib().mdb_softmax_rows(_ptr(s), s.stride(0), s.shape[0], cols, _ptr(out), cols_out, cols_out, _stream()),
          "mdb_softmax_rows")
    _launches += 1
    return out


def attention(q, k, v, *, b, heads, lq, lk, d, ldq, ldk, ldv, scale, kv_index=None, n_sets=1, out=None, b_kv=None):
    """q: [b*lq, >=heads*d] view with row stride ldq, k/v [b_kv*lk, ...] likewise; returns [b*lq, heads*d] bf16."""
    b_kv = b if b_kv is None else b_kv
    global _launches
    _need_cuda(q, k, v)
    if out is None:
        out = torch.empty((b * lq, heads * d), dtype=BF16, device=q.device)
    e0 = _prof_begin()
    check(_lib.lib().mdb_attention(_ptr(q), ldq, _ptr(k), ldk, _ptr(v), ldv, _ptr(out), out.stride(0), b, b_kv, heads, lq,
                                   lk, d, _ptr(kv_index), n_sets, float(scale), _stream()), "mdb_attention")
    _prof_end("attention", 4.0 * b * heads * lq * lk * d * n_sets, e0, f"B={b} H={heads} Lq={lq} Lk={lk} D={d} sets={n_sets}")
    _launches += 1
    return out


def attention_multi(q, sources, *, b, heads, lq, lk, d, ldq, scale, kv_index, n_sets=1, out=None):
    """Fused attention whose K/V batches live in up to three buffers (mdb_attention_multi).  `sources` = list of (k, v, ld, b_kv):
    k / v are [b_kv * lk, >= heads*d] views with row stride ld (a peer GPU's buffer mapped through NVLink works like a local
    one); kv_index entries are (source << 24) | batch index."""
    global _launches
    _need_cuda(q, *[t for s_ in sources for t in s_[:2]])
    n = len(sources)
    if out is None:
        out = torch.empty((b * lq, heads * d), dtype=BF16, device=q.device)
    ks = (C.c_void_p * n)(*[s_[0].data_ptr() for s_ in sources])
    vs = (C.c_void_p * n)(*[s_[1].data_ptr() for s_ in sources])
    ldk = (C.c_int * n)(*[int(s_[2]) for s_ in sources])
    bkv = (C.c_int * n)(*[int(s_[3]) for s_ in sources])
    e0 = _prof_begin()
    check(_lib.lib().mdb_attention_multi(_ptr(q), ldq, n, ks, ldk, vs, ldk, bkv, _ptr(out), out.stride(0), b, heads, lq, lk, d,
                                         _ptr(kv_index), n_sets, float(scale), _stream()), "mdb_attention_multi")
    _prof_end("attention", 4.0 * b * heads * lq * lk * d * n_sets, e0, f"B={b} H={heads} Lq={lq} Lk={lk} D={d} sets={n_sets} src={n}")
    _launches += 1
    return out


def peer_barrier(flag_ptrs_dev: int, rank: int, world: int, channel: int, n_channels: int, epoch, timed_out,
                 timeout_s: float = 5.0):
    """Device-side barrier over NVLink peer memory (mdb_peer_barrier); one warp on the current stream."""
    global _launches
    cycles = int(timeout_s * 1.9e9)
    check(_lib.lib().mdb_peer_barrier(flag_ptrs_dev, rank, world, channel, n_channels, _ptr(epoch), cycles, _ptr(timed_out),
                                      _stream()), "mdb_peer_barrier")
    _launches += 1


def add(a, b):
    global _launches
    _need_cuda(a, b)
    out = torch.empty_like(a)
    check(_lib.lib().mdb_add(_ptr(a), _ptr(b), _ptr(out), a.numel(), _stream()), "mdb_add")
    _launches += 1
    return out


def upsample_nearest(x, n, h, w, c, ho, wo):
    global _launches
    _need_cuda(x)
    out = torch.empty((n * ho * wo, c), dtype=BF16, device=x.device)
    check(_lib.lib().mdb_upsample_nearest(_ptr(x), n, h, w, c, _ptr(out), ho, wo, _stream()), "mdb_upsample_nearest")
    _launches += 1
    return out


def adaptive_avgpool(x, n, h, w, c, ho, wo, silu=False):
    """nn.AdaptiveAvgPool2d((ho, wo)) (+ SiLU) over an NHWC fp32 map [n, h, w, c] -> fp32 [n, ho, wo, c]."""
    global _launches
    _need_cuda(x)
    assert x.dtype == F32 and x.is_contiguous()
    out = torch.empty((n, ho, wo, c), dtype=F32, device=x.device)
    check(_lib.lib().mdb_adaptive_avgpool(_ptr(x), n, h, w, c, _ptr(out), ho, wo, int(silu), _stream()), "mdb_adaptive_avgpool")
    _launches += 1
    return out


def linear_small(x, w, bias=None, pre_silu=False, post_silu=False):
    """x fp32 [m, k]; w bf16 [n, k]; returns fp32 [m, n]."""
    global _launches
    _need_cuda(x, w)
    m, k = x.shape
    n = w.shape[0]
    out = torch.empty((m, n), dtype=F32, device=x.device)
    check(_lib.lib().mdb_linear_small(_ptr(x), m, k, x.stride(0), _ptr(w), w.stride(0), _ptr(bias), n, int(pre_silu),
                                      int(post_silu), _ptr(out), n, _stream()), "mdb_linear_small")
    _launches += 1
    return out


def timestep_embedding(t, dim, flip_sin_to_cos=True, freq_shift=0.0):
    global _launches
    _need_cuda(t)
    out = torch.empty((t.numel(), dim), dtype=F32, device=t.device)
    check(_lib.lib().mdb_timestep_embedding(_ptr(t), t.numel(), dim, int(flip_sin_to_cos), float(freq_shift), _ptr(out),
                                            _stream()), "mdb_timestep_embedding")
    _launches += 1
    return out


def fourier_embed(x, num_freqs):
    global _launches
    _need_cuda(x)
    rows, d = x.shape
    out = torch.empty((rows, d * (1 + 2 * num_freqs)), dtype=F32, device=x.device)
    check(_lib.lib().mdb_fourier_embed(_ptr(x), rows, d, num_freqs, _ptr(out), _stream()), "mdb_fourier_embed")
    _launches += 1
    return out


def nchw_to_nhwc(x):
    global _launches
    _need_cuda(x)
    n, c, h, w = x.shape
    x = x.contiguous()
    if x.dtype not in (F32, BF16):
        x = x.float()
    out = torch.empty((n * h * w, c), dtype=BF16, device=x.device)
    check(_lib.lib().mdb_nchw_to_nhwc(_ptr(x), int(x.dtype == F32), n, c, h, w, _ptr(out), _stream()), "mdb_nchw_to_nhwc")
    _launches += 1
    return out


def nhwc_to_nchw(x, n, c, h, w, dtype=F32):
    global _launches
    _need_cuda(x)
    out = torch.empty((n, c, h, w), dtype=dtype, device=x.device)
    check(_lib.lib().mdb_nhwc_to_nchw(_ptr(x), n, c, h, w, _ptr(out), int(dtype == F32), _stream()), "mdb_nhwc_to_nchw")
    _launches += 1
    return out


def f32_to_bf16(x):
    global _launches
    out = torch.empty(x.shape, dtype=BF16, device=x.device)
    check(_lib.lib().mdb_f32_to_bf16(_ptr(x), _ptr(out), x.numel(), _stream()), "mdb_f32_to_bf16")
    _launches += 1
    return out


def cfg_ddim_step(eps, latents, coef, cfg: bool, guidance: float, c: int = 4):
    """eps fp32 [(2|1)*pixels, ld>=c]; latents fp32 [pixels, c] updated in place."""
    global _launches
    _need_cuda(eps, latents, coef)
    check(_lib.lib().mdb_cfg_ddim_step(_ptr(eps), eps.stride(0), c, int(cfg), float(guidance), _ptr(coef), _ptr(latents),
                                       latents.numel(), _stream()), "mdb_cfg_ddim_step")
    _launches += 1
    return latents


def cfg_unipc_step(eps, latents, last_sample, m0, m1, coef, cfg: bool, guidance: float, c: int = 4):
    """Guidance + one UniPC step; latents / last_sample / m0 / m1 fp32 [pixels, c] updated in place, coef fp32[12]."""
    global _launches
    _need_cuda(eps, latents, last_sample, m0, m1, coef)
    check(_lib.lib().mdb_cfg_unipc_step(_ptr(eps), eps.stride(0), c, int(cfg), float(guidance), _ptr(coef), _ptr(latents),
                                        _ptr(last_sample), _ptr(m0), _ptr(m1), latents.numel(), _stream()),
          "mdb_cfg_unipc_step")
    _launches += 1
    return latents


def pin_views(dst, a, b, coef, view_mask, rows_per_view: int, c: int = 4):
    """dst[rows of flagged views, :c] = coef[0]*a + coef[1]*b  (a may be None); dst fp32 [n_views*rows_per_view, ld>=c]."""
    global _launches
    _need_cuda(dst, b, coef, view_mask)
    assert view_mask.dtype == torch.int32 and dst.shape[0] == view_mask.numel() * rows_per_view
    check(_lib.lib().mdb_pin_views(_ptr(dst), dst.stride(0), _ptr(a), _ptr(b), c, _ptr(coef), _ptr(view_mask),
                                   rows_per_view, view_mask.numel(), _stream()), "mdb_pin_views")
    _launches += 1
    return dst


def pack_image_patches(x):
    """NCHW images [n, cin, h, w] fp32/bf16 -> bf16 [n*h*w, 64]: the zero-padded 3x3 neighbourhood of every pixel in
    column order (tap, channel), columns >= 9*cin zero (the A operand of the VAE encoder's conv_in as a K = 64 GEMM)."""
    global _launches
    _need_cuda(x)
    n, cin, h, w = x.shape
    x = x.contiguous()
    if x.dtype not in (F32, BF16):
        x = x.float()
    out = torch.empty((n * h * w, 64), dtype=BF16, device=x.device)
    check(_lib.lib().mdb_pack_image_patches(_ptr(x), int(x.dtype == F32), n, cin, h, w, _ptr(out), _stream()),
          "mdb_pack_image_patches")
    _launches += 1
    return out


def latent_dist(moments, n: int, h: int, w: int, c: int = 4, noise=None, scale: float = 1.0):
    """fp32 NHWC moments [n*h*w, >= 2c] (mean | logvar) -> fp32 NCHW [n, c, h, w] =
    scale * (mean + exp(0.5 * clamp(logvar, -30, 20)) * noise); noise fp32 NCHW or None (scale * mean)."""
    global _launches
    _need_cuda(moments, noise)
    assert moments.dtype == F32 and moments.shape[0] == n * h * w
    if noise is not None:
        assert noise.dtype == F32 and noise.is_contiguous() and noise.numel() == n * c * h * w
    out = torch.empty((n, c, h, w), dtype=F32, device=moments.device)
    check(_lib.lib().mdb_latent_dist(_ptr(moments), moments.stride(0), n, c, h, w, _ptr(noise), float(scale), _ptr(out),
                                     _stream()), "mdb_latent_dist")
    _launches += 1
    return out


def pack_latents(x, cpad: int = 64, repeat: int = 1):
    """[pix, cin] fp32/bf16 -> bf16 [repeat*pix, cpad] zero-padded channels."""
    global _launches
    _need_cuda(x)
    pix, cin = x.shape
    out = torch.empty((repeat * pix, cpad), dtype=BF16, device=x.device)
    check(_lib.lib().mdb_pack_latents(_ptr(x), int(x.dtype == F32), pix, cin, cpad, repeat, _ptr(out), _stream()),
          "mdb_pack_latents")
    _launches += 1
    return out
