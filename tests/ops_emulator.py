"""TEST INFRASTRUCTURE ONLY — a torch restatement of every operator in magicdrive_b200/ops.py, following the semantics the C
header documents (include/magicdrive_b200.h), so that the HOST side of the product (weight packing in engine._Weights /
params.py, layer sequencing in engine.py, the module wrappers, the denoiser) can be executed and checked against the
oracle in the build container, which has no GPU.  It is never imported by the package; `install(monkeypatch)` swaps it in
for the duration of one test.  What it cannot check is the CUDA code itself: that is tests/test_*_gpu.py.

Arithmetic is fp32 from the (bf16-rounded) packed weights; activations are NOT rounded to bf16 (`ROUND_ACTIVATIONS`
switches that on), so a host-logic mistake shows up at 1e-5, not inside bf16 noise.  `COMPUTE_DTYPE` = float64 turns the
same restatements into a high-precision reference of the device kernels (tests/launch_check.py); every operator computes
on the device of its inputs."""
import math

import torch
import torch.nn.functional as F

from magicdrive_b200 import ops

ROUND_ACTIVATIONS = False
COMPUTE_DTYPE = torch.float32  # float64: the reference of tests/launch_check.py


def _f(x):
    """An operand in the compute dtype."""
    return x.to(COMPUTE_DTYPE)


def _act(x):
    """Output of a device operator: a fresh contiguous buffer (optionally with the device's bf16 rounding)."""
    return (_f(x.to(torch.bfloat16)) if ROUND_ACTIVATIONS else _f(x)).contiguous()


def gemm_conv(a0, w, *, n_img, h_in, w_in, c0, lda0, n_out, taps=1, stride=1, pad=0, h_out=None, w_out=None, a1=None,
              c1=0, lda1=0, bias=None, rowbias=None, residual=None, ldr=0, out=None, ldo=None, out_f32=False,
              out_scale=1.0, geglu=False, ln=None, ln_colsum=None, ln_eps=1e-5, emit_stats=False, **_):
    if h_out is None:
        h_out = (h_in + 2 * pad - taps) // stride + 1
    if w_out is None:
        w_out = (w_in + 2 * pad - taps) // stride + 1
    pix_in = n_img * h_in * w_in
    assert a0.shape[0] == pix_in and a0.stride(0) == lda0, (a0.shape, a0.stride(), lda0)
    x = _f(a0[:, :c0])
    if c1:
        assert a1.shape[0] == pix_in and a1.stride(0) == lda1
        x = torch.cat([x, _f(a1[:, :c1])], 1)
    cin = c0 + c1
    assert w.shape == (n_out, taps * taps * cin), (w.shape, n_out, taps, cin)
    x = x.reshape(n_img, h_in, w_in, cin).permute(0, 3, 1, 2)
    w4 = _f(w).reshape(n_out, taps, taps, cin).permute(0, 3, 1, 2)  # K ordered (tap, channel)
    acc = F.conv2d(x, w4, stride=stride, padding=pad)
    assert acc.shape[2:] == (h_out, w_out)
    acc = acc.permute(0, 2, 3, 1).reshape(n_img * h_out * w_out, n_out)
    if ln is not None:  # folded LayerNorm: rstd * (acc - mean * colsum) with the producer's row statistics
        assert taps == 1 and ln.data.shape[0] == acc.shape[0]
        tot = _f(ln.data).sum(1)
        mean = tot[:, 0:1] / cin
        var = (tot[:, 1:2] / cin - mean * mean).clamp_min(0)
        acc = torch.rsqrt(var + ln_eps) * (acc - mean * _f(ln_colsum)[None, :])
    if bias is not None:
        acc = acc + _f(bias)
    if rowbias is not None:
        rb = _f(rowbias)
        rb = rb.expand(n_img, -1) if rb.shape[0] == 1 else rb
        acc = acc + rb[:, :n_out].repeat_interleave(h_out * w_out, 0)
    acc = acc * out_scale
    if geglu:  # 256-column tiles of [128 value | 128 gate]
        t = acc.reshape(acc.shape[0], n_out // 256, 2, 128)
        res = (t[:, :, 0] * F.gelu(t[:, :, 1])).reshape(acc.shape[0], n_out // 2)
    else:
        res = acc
    if residual is not None:
        r2 = residual.reshape(-1, residual.shape[-1])  # the device reads it as [pixels, ldr] through a raw pointer
        assert r2.shape[0] == res.shape[0] and r2.stride(0) == ldr, (residual.shape, ldr)
        res = res + r2[:, :res.shape[1]].float()
    res = res.contiguous() if out_f32 else _act(res)
    stats = None
    if emit_stats:  # two partial slots per row, like a one-tile launch of the device kernel
        rr = _f(res)  # the device accumulates the values it stores (already bf16-rounded when ROUND_ACTIVATIONS)
        half = res.shape[1] // 2
        parts = torch.stack([torch.stack([rr[:, :half].sum(1), (rr[:, :half] ** 2).sum(1)], -1),
                             torch.stack([rr[:, half:].sum(1), (rr[:, half:] ** 2).sum(1)], -1)], 1)
        stats = ops.RowStats(parts.contiguous(), 2)
    if out is not None:
        out[:, :res.shape[1]] = res
        return (out, stats) if emit_stats else out
    return (res, stats) if emit_stats else res


def linear(x, w, bias=None, residual=None, out=None, ldo=None, geglu=False, out_f32=False, out_scale=1.0, **kw):
    m, k = x.shape
    return gemm_conv(x, w, n_img=1, h_in=1, w_in=m, c0=k, lda0=x.stride(0), n_out=w.shape[0], bias=bias,
                     residual=residual, ldr=(residual.stride(0) if residual is not None else 0), out=out, ldo=ldo,
                     geglu=geglu, out_f32=out_f32, out_scale=out_scale, **kw)


def conv_direct(x, wgt, bias, *, n, h, w, cin, cout, k, stride=(1, 1), pad=(1, 1), silu=False, residual=None, out_f32=False):
    assert wgt.shape == (k, k, cin, cout)
    y = F.conv2d(_f(x).reshape(n, h, w, cin).permute(0, 3, 1, 2), _f(wgt).permute(3, 2, 0, 1), _f(bias),
                 stride=stride, padding=pad)
    if silu:
        y = F.silu(y)
    y = y.permute(0, 2, 3, 1)
    if residual is not None:
        y = y + _f(residual).reshape(y.shape)
    return (y if out_f32 else _act(y)).contiguous()


def groupnorm(x0, c0, ld0, n_img, hw, gamma, beta, eps, silu, x1=None, c1=0, ld1=0, groups=32):
    assert x0.stride(0) == ld0
    x = _f(x0[:, :c0])
    if c1:
        assert x1.stride(0) == ld1
        x = torch.cat([x, _f(x1[:, :c1])], 1)
    c = c0 + c1
    y = F.group_norm(x.reshape(n_img, hw, c).permute(0, 2, 1), groups, _f(gamma), _f(beta), eps)
    if silu:
        y = F.silu(y)
    return _act(y.permute(0, 2, 1).reshape(n_img * hw, c))


def layernorm(x, gamma, beta, eps=1e-5):
    return _act(F.layer_norm(_f(x), (x.shape[1],), _f(gamma), _f(beta), eps))


def attention(q, k, v, *, b, heads, lq, lk, d, ldq, ldk, ldv, scale, kv_index=None, n_sets=1, out=None, b_kv=None):
    b_kv = b if b_kv is None else b_kv
    c = heads * d
    assert q.stride(0) == ldq and k.stride(0) == ldk and v.stride(0) == ldv
    qh = _f(q[:, :c]).reshape(b, lq, heads, d).transpose(1, 2)
    kh = _f(k[:, :c]).reshape(b_kv, lk, heads, d).transpose(1, 2)
    vh = _f(v[:, :c]).reshape(b_kv, lk, heads, d).transpose(1, 2)
    if kv_index is None:
        assert n_sets == 1 and b_kv == b
        sels = [torch.arange(b)]
    else:
        idx = kv_index.reshape(b, n_sets).long().cpu()
        sels = [idx[:, s] for s in range(n_sets)]
    parts = []
    nb = max(1, (1 << 28) // (heads * lq * lk))  # images per chunk: bounds the score tensor of long sequences
    for b0 in range(0, b, nb):
        rows, part = slice(b0, b0 + nb), 0
        for sel in sels:
            o = torch.softmax(qh[rows] @ kh[sel[rows]].transpose(-1, -2) * scale, -1) @ vh[sel[rows]]
            part = part + _act(o)  # each branch is rounded to bf16 before the sum on the device
        parts.append(part)
    res = parts[0] if len(parts) == 1 else torch.cat(parts)
    res = _act(res.transpose(1, 2).reshape(b * lq, c))
    if out is not None:
        out[:, :c] = res
        return out
    return res


def softmax_rows(s, cols, cols_out):
    p = torch.softmax(_f(s[:, :cols]), -1)
    return _act(F.pad(p, (0, cols_out - cols)))


def add(a, b):
    return _act(_f(a) + _f(b))


def upsample_nearest(x, n, h, w, c, ho, wo):
    xi = _f(x).reshape(n, h, w, c)
    iy = torch.div(torch.arange(ho, device=x.device) * h, ho, rounding_mode="floor")
    ix = torch.div(torch.arange(wo, device=x.device) * w, wo, rounding_mode="floor")
    return xi[:, iy][:, :, ix].reshape(n * ho * wo, c).contiguous()


def adaptive_avgpool(x, n, h, w, c, ho, wo, silu=False):
    y = F.adaptive_avg_pool2d(_f(x).reshape(n, h, w, c).permute(0, 3, 1, 2), (ho, wo))
    y = F.silu(y) if silu else y
    return y.permute(0, 2, 3, 1).contiguous()


def linear_small(x, w, bias=None, pre_silu=False, post_silu=False):
    h = F.silu(_f(x)) if pre_silu else _f(x)
    y = h @ _f(w).t()
    if bias is not None:
        y = y + _f(bias)
    return F.silu(y) if post_silu else y


def timestep_embedding(t, dim, flip_sin_to_cos=True, freq_shift=0.0):
    half = dim // 2
    freqs = torch.exp(-math.log(10000.0) * torch.arange(half, dtype=COMPUTE_DTYPE, device=t.device) / (half - freq_shift))
    arg = _f(t)[:, None] * freqs[None]
    emb = torch.cat([torch.sin(arg), torch.cos(arg)], -1)
    return torch.cat([emb[:, half:], emb[:, :half]], -1) if flip_sin_to_cos else emb


def fourier_embed(x, num_freqs):
    outs = [_f(x)]
    for k in range(num_freqs):
        outs += [torch.sin(_f(x) * 2.0 ** k), torch.cos(_f(x) * 2.0 ** k)]
    return torch.cat(outs, -1)


def nchw_to_nhwc(x):
    n, c, h, w = x.shape
    return _act(_f(x).permute(0, 2, 3, 1).reshape(n * h * w, c))


def nhwc_to_nchw(x, n, c, h, w, dtype=torch.float32):
    return _f(x).reshape(n, h, w, -1)[..., :c].permute(0, 3, 1, 2).contiguous().to(dtype)


def f32_to_bf16(x):
    return _act(x)


def bf16_to_f32(x):
    return x.float()


def pack_latents(x, cpad=64, repeat=1):
    return _act(F.pad(_f(x), (0, cpad - x.shape[1]))).repeat(repeat, 1)


def cfg_combine(eps, cfg, guidance, c, npix):
    e = _f(eps[:, :c])
    return e[:npix] + guidance * (e[npix:] - e[:npix]) if cfg else e


def cfg_ddim_step(eps, latents, coef, cfg, guidance, c=4):
    latents.copy_(_f(coef[0]) * _f(latents) + _f(coef[1]) * cfg_combine(eps, cfg, guidance, c, latents.shape[0]))
    return latents


def cfg_unipc_step(eps, latents, last, m0, m1, coef, cfg, guidance, c=4):
    e, x, coef = cfg_combine(eps, cfg, guidance, c, latents.shape[0]), _f(latents).clone(), _f(coef)
    x0 = coef[0] * x + coef[1] * e
    xc = coef[2] * _f(last) + coef[3] * _f(m0) + coef[4] * _f(m1) + coef[5] * x0 if coef[9] != 0 else x
    latents.copy_(coef[6] * xc + coef[7] * x0 + coef[8] * _f(m0))
    last.copy_(xc)
    m1.copy_(m0)
    m0.copy_(x0)
    return latents


def pin_views(dst, a, b, coef, view_mask, rows_per_view, c=4):
    sel = view_mask.bool().repeat_interleave(rows_per_view)
    coef = _f(coef)
    dst[sel, :c] = ((coef[0] * _f(a[sel]) if a is not None else 0) + coef[1] * _f(b[sel])).to(dst.dtype)
    return dst


class workspace_slot:
    def __init__(self, slot):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


EMULATED = ["softmax_rows", "gemm_conv", "linear", "conv_direct", "groupnorm", "layernorm", "attention", "add", "upsample_nearest", "adaptive_avgpool",
            "linear_small", "timestep_embedding", "fourier_embed", "nchw_to_nhwc", "nhwc_to_nchw", "f32_to_bf16",
            "pack_latents", "cfg_ddim_step", "cfg_unipc_step", "pin_views", "workspace_slot"]


def install(monkeypatch):
    """Swap every operator of magicdrive_b200.ops for its torch restatement and let the modules build engines on CPU."""
    from magicdrive_b200 import models
    for name in EMULATED:
        assert hasattr(ops, name), name
        monkeypatch.setattr(ops, name, globals()[name])
    monkeypatch.setattr(models._B200Module, "_get_engine",
                        lambda self, cls_: self.__dict__.setdefault("_eng", cls_(self.arch_cfg, dict(self.state_dict()), self.device)))
