"""GPU parity of each C-ABI operator against plain torch fp32 on the same (bf16-rounded) inputs."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from magicdrive_b200 import ops  # noqa: E402


def _bf(x):
    return x.to(torch.bfloat16)


def _rel(a, b):
    return ((a.float() - b.float()).abs().max() / (b.float().abs().max() + 1e-6)).item()


def _nhwc(x):  # NCHW -> [n*h*w, c]
    n, c, h, w = x.shape
    return x.permute(0, 2, 3, 1).reshape(n * h * w, c).contiguous()


def _conv_weight(wt):  # [co, ci, kh, kw] -> [co, kh*kw*ci] (tap-major, channel-minor)
    co, ci, kh, kw = wt.shape
    return wt.permute(0, 2, 3, 1).reshape(co, kh * kw * ci).contiguous()


@pytest.mark.parametrize("variant", [0, 2])  # 0 = planner's choice (CTA-pair kernel where it applies), 2 = single-CTA persistent kernel
@pytest.mark.parametrize("bn", [0, 64, 128, 160, 256])
@pytest.mark.parametrize("m,k,n", [(1000, 320, 320), (128, 64, 640), (336, 1280, 1280), (16800, 320, 960)])
def test_gemm_plain(cuda_lib, bn, m, k, n, variant):
    g = torch.Generator(device="cuda").manual_seed(1)
    x = _bf(torch.randn(m, k, device="cuda", generator=g))
    w = _bf(torch.randn(n, k, device="cuda", generator=g) / math.sqrt(k))
    b = torch.randn(n, device="cuda", generator=g)
    r = _bf(torch.randn(m, n, device="cuda", generator=g))
    ref = x.float() @ w.float().t() + b + r.float()
    out = ops.linear(x, w, bias=b, residual=r, out_f32=True, force_block_n=bn, allow_split_k=False, kernel_variant=variant)
    torch.cuda.synchronize()
    assert _rel(out, ref) < 2e-5, _rel(out, ref)
    out16 = ops.linear(x, w, bias=b, residual=r, force_block_n=bn, allow_split_k=False, kernel_variant=variant)
    assert _rel(out16, ref) < 6e-3


@pytest.mark.parametrize("splits", [2, 5])
def test_gemm_split_k(cuda_lib, splits):
    g = torch.Generator(device="cuda").manual_seed(2)
    m, k, n = 336, 2560, 1280
    x = _bf(torch.randn(m, k, device="cuda", generator=g))
    w = _bf(torch.randn(n, k, device="cuda", generator=g) / math.sqrt(k))
    b = torch.randn(n, device="cuda", generator=g)
    ref = (x.float() @ w.float().t() + b) * 0.5
    out = ops.linear(x, w, bias=b, out_f32=True, out_scale=0.5, force_splits=splits)
    assert _rel(out, ref) < 2e-5, _rel(out, ref)


@pytest.mark.parametrize("case", ["zero_conv", "conv3x3_shift"])
def test_gemm_split_k_bf16_residual(cuda_lib, case):
    """The planner's own split-K route (nothing forced) at the 4 x 7 level of the benchmark (V = 12, M = 336), bf16 output:
    a ControlNet zero convolution onto the UNet skip (residual, out_scale) and a ResNet conv1 with its per-image time shift
    (four images per M tile, which the pair kernel refuses) plus residual.  Every element within one bf16 rounding step."""
    g = torch.Generator(device="cuda").manual_seed(15)
    n, h, w, c = 12, 4, 7, 1280
    x = _bf(torch.randn(n * h * w, c, device="cuda", generator=g))
    r = _bf(torch.randn(n * h * w, c, device="cuda", generator=g))
    b = torch.randn(c, device="cuda", generator=g)
    n0 = ops.launch_count()
    if case == "zero_conv":
        wt = _bf(torch.randn(c, c, device="cuda", generator=g) / math.sqrt(c))
        out = ops.linear(x, wt, bias=b, residual=r, out_scale=0.7)
        ref = 0.7 * (x.float() @ wt.float().t() + b) + r.float()
    else:
        wt = _bf(torch.randn(c, c, 3, 3, device="cuda", generator=g) / math.sqrt(9 * c))
        temb = torch.randn(n, c, device="cuda", generator=g)
        out = ops.gemm_conv(x, _conv_weight(wt), n_img=n, h_in=h, w_in=w, c0=c, lda0=c, n_out=c, taps=3, pad=1, bias=b,
                            rowbias=temb, residual=r, ldr=c)
        xi = x.float().reshape(n, h, w, c).permute(0, 3, 1, 2)
        ref = _nhwc(F.conv2d(xi, wt.float(), b, padding=1) + temb[:, :, None, None]) + r.float()
    assert ops.launch_count() - n0 == 2  # split-K partials + finalize
    err = (out.float() - ref).abs()
    bad = (err > ref.abs() * 2.0 ** -7 + 2e-3 * ref.abs().max()).sum().item()
    assert bad == 0, (bad, err.max().item())


def test_gemm_strided_views(cuda_lib):
    """A read from a column slice of a wider buffer, output written into a column slice (fused-QKV style)."""
    g = torch.Generator(device="cuda").manual_seed(3)
    m, k, n = 700, 320, 320
    big = _bf(torch.randn(m, 3 * k, device="cuda", generator=g))
    x = big[:, k:2 * k]
    w = _bf(torch.randn(n, k, device="cuda", generator=g) / math.sqrt(k))
    outbuf = torch.zeros(m, 2 * n, dtype=torch.bfloat16, device="cuda")
    ops.linear(x, w, out=outbuf[:, n:], ldo=2 * n)
    ref = x.float() @ w.float().t()
    assert _rel(outbuf[:, n:], ref) < 6e-3
    assert outbuf[:, :n].abs().max().item() == 0


@pytest.mark.parametrize("n,h,w,ci,co,stride", [
    (3, 28, 50, 320, 320, 1), (2, 14, 25, 640, 1280, 1), (5, 4, 7, 1280, 1280, 1), (3, 7, 13, 1280, 640, 1),
    (2, 28, 50, 320, 320, 2), (3, 14, 25, 640, 640, 2), (5, 7, 13, 1280, 1280, 2), (1, 53, 100, 320, 320, 1),
    (12, 28, 50, 320, 320, 1),
])
@pytest.mark.parametrize("variant", [0, 2])
def test_conv3x3(cuda_lib, n, h, w, ci, co, stride, variant):
    g = torch.Generator(device="cuda").manual_seed(4)
    x = _bf(torch.randn(n, ci, h, w, device="cuda", generator=g))
    wt = _bf(torch.randn(co, ci, 3, 3, device="cuda", generator=g) / math.sqrt(9 * ci))
    b = torch.randn(co, device="cuda", generator=g)
    temb = torch.randn(n, co, device="cuda", generator=g)
    ref = F.conv2d(x.float(), wt.float(), b, stride=stride, padding=1) + temb[:, :, None, None]
    ho, wo = ref.shape[-2:]
    out = ops.gemm_conv(_nhwc(x), _conv_weight(wt), n_img=n, h_in=h, w_in=w, c0=ci, lda0=ci, n_out=co, taps=3,
                        stride=stride, pad=1, bias=b, rowbias=temb, out_f32=True, kernel_variant=variant)
    assert out.shape == (n * ho * wo, co)
    assert _rel(out, _nhwc(ref)) < 3e-5, _rel(out, _nhwc(ref))


def test_conv3x3_two_sources_residual(cuda_lib):
    g = torch.Generator(device="cuda").manual_seed(5)
    n, h, w, c0, c1, co = 2, 14, 25, 640, 320, 640
    xa = _bf(torch.randn(n, c0, h, w, device="cuda", generator=g))
    xb = _bf(torch.randn(n, c1, h, w, device="cuda", generator=g))
    wt = _bf(torch.randn(co, c0 + c1, 3, 3, device="cuda", generator=g) / math.sqrt(9 * (c0 + c1)))
    res = _bf(torch.randn(n, co, h, w, device="cuda", generator=g))
    ref = F.conv2d(torch.cat([xa, xb], 1).float(), wt.float(), None, padding=1) + res.float()
    out = ops.gemm_conv(_nhwc(xa), _conv_weight(wt), n_img=n, h_in=h, w_in=w, c0=c0, lda0=c0, a1=_nhwc(xb), c1=c1,
                        lda1=c1, n_out=co, taps=3, pad=1, residual=_nhwc(res), ldr=co, out_f32=True)
    assert _rel(out, _nhwc(ref)) < 3e-5
    # 1x1 shortcut over the same concat
    w1 = _bf(torch.randn(co, c0 + c1, 1, 1, device="cuda", generator=g) / math.sqrt(c0 + c1))
    ref1 = F.conv2d(torch.cat([xa, xb], 1).float(), w1.float())
    out1 = ops.gemm_conv(_nhwc(xa), _conv_weight(w1), n_img=n, h_in=h, w_in=w, c0=c0, lda0=c0, a1=_nhwc(xb), c1=c1,
                         lda1=c1, n_out=co, out_f32=True)
    assert _rel(out1, _nhwc(ref1)) < 3e-5


def test_geglu(cuda_lib):
    from magicdrive_b200.params import pack_geglu
    g = torch.Generator(device="cuda").manual_seed(6)
    m, c = 777, 320
    x = _bf(torch.randn(m, c, device="cuda", generator=g))
    w = _bf(torch.randn(8 * c, c, device="cuda", generator=g) / math.sqrt(c))
    b = torch.randn(8 * c, device="cuda", generator=g)
    h = x.float() @ w.float().t() + b
    val, gate = h.chunk(2, dim=-1)
    ref = val * F.gelu(gate)
    wp, bp = pack_geglu(w, b)
    out = ops.linear(x, wp, bias=bp, geglu=True)
    assert out.shape == (m, 4 * c)
    assert _rel(out, ref) < 8e-3, _rel(out, ref)


@pytest.mark.parametrize("c0,c1,hw,n", [(320, 0, 1400, 3), (640, 320, 350, 2), (1280, 1280, 91, 5), (64, 0, 1400, 2)])
@pytest.mark.parametrize("silu", [False, True])
def test_groupnorm(cuda_lib, c0, c1, hw, n, silu):
    g = torch.Generator(device="cuda").manual_seed(7)
    xa = _bf(torch.randn(n * hw, c0, device="cuda", generator=g) * 2 + 0.5)
    xb = _bf(torch.randn(n * hw, c1, device="cuda", generator=g)) if c1 else None
    c = c0 + c1
    gamma = torch.randn(c, device="cuda", generator=g)
    beta = torch.randn(c, device="cuda", generator=g)
    full = xa if xb is None else torch.cat([xa, xb], 1)
    ref = F.group_norm(full.float().reshape(n, hw, c).permute(0, 2, 1), 32, gamma, beta, 1e-5)
    if silu:
        ref = F.silu(ref)
    ref = ref.permute(0, 2, 1).reshape(n * hw, c)
    out = ops.groupnorm(xa, c0, c0, n, hw, gamma, beta, 1e-5, silu, x1=xb, c1=c1, ld1=c1)
    assert (out.float() - ref).abs().max().item() < 0.06  # bf16 output rounding on O(5) values
    assert _rel(out, ref) < 8e-3


@pytest.mark.parametrize("c0,c1,hw,n,pad", [(320, 0, 1400, 12, 0), (640, 0, 350, 12, 64), (320, 320, 1400, 3, 0), (640, 320, 350, 2, 8),
                                             (1280, 1280, 91, 5, 0), (1280, 0, 28, 12, 0), (64, 0, 1400, 2, 0), (320, 0, 37, 3, 0),
                                             (1280, 640, 350, 2, 0)])
@pytest.mark.parametrize("silu", [False, True])
def test_groupnorm_cluster_rows(cuda_lib, monkeypatch, c0, c1, hw, n, pad, silu):
    """pixel-major cluster kernel (forced): same fp32 reference, and agreement with the (image, group) kernel; `pad` =
    extra row stride of the first source (a channel slice of a wider buffer)."""
    g = torch.Generator(device="cuda").manual_seed(17)
    wide = _bf(torch.randn(n * hw, c0 + pad, device="cuda", generator=g) * 2 + 0.5)
    xa = wide[:, :c0]
    xb = _bf(torch.randn(n * hw, c1, device="cuda", generator=g)) if c1 else None
    c = c0 + c1
    gamma = torch.randn(c, device="cuda", generator=g)
    beta = torch.randn(c, device="cuda", generator=g)
    full = xa if xb is None else torch.cat([xa, xb], 1)
    ref = F.group_norm(full.float().reshape(n, hw, c).permute(0, 2, 1), 32, gamma, beta, 1e-5)
    if silu:
        ref = F.silu(ref)
    ref = ref.permute(0, 2, 1).reshape(n * hw, c)
    monkeypatch.setenv("MDB_GN_ROWS", "0")
    base = ops.groupnorm(xa, c0, c0 + pad, n, hw, gamma, beta, 1e-5, silu, x1=xb, c1=c1, ld1=c1)
    monkeypatch.setenv("MDB_GN_ROWS", "1")
    out = ops.groupnorm(xa, c0, c0 + pad, n, hw, gamma, beta, 1e-5, silu, x1=xb, c1=c1, ld1=c1)
    torch.cuda.synchronize()
    assert (out.float() - ref).abs().max().item() < 0.06
    assert _rel(out, ref) < 8e-3
    assert _rel(out, ref) <= _rel(base, ref) * 1.05 + 1e-5
    # both kernels round the same fp32 values up to the last bits of mean / rstd: a handful of one-ulp flips at most
    assert (out != base).float().mean().item() < 2e-3


@pytest.mark.parametrize("c", [64, 320, 640, 1280])
def test_layernorm(cuda_lib, c):
    g = torch.Generator(device="cuda").manual_seed(8)
    x = _bf(torch.randn(1003, c, device="cuda", generator=g) * 3 + 1)
    gamma = torch.randn(c, device="cuda", generator=g)
    beta = torch.randn(c, device="cuda", generator=g)
    ref = F.layer_norm(x.float(), (c,), gamma, beta, 1e-5)
    out = ops.layernorm(x, gamma, beta)
    assert _rel(out, ref) < 8e-3


ATTN_KERNELS = ["tc2", "tc2d", "tc"]  # tcgen05 v2 (2 CTAs/SM | double-buffered S; d = 160 falls to tc), tcgen05 v1


def _pick_attention_kernel(monkeypatch, kernel):
    monkeypatch.delenv("MDB_ATTN_LEGACY", raising=False)
    monkeypatch.setenv("MDB_ATTN_KERNEL", kernel)


@pytest.mark.parametrize("kernel", ATTN_KERNELS)
@pytest.mark.parametrize("d,heads", [(40, 8), (80, 8), (160, 8), (32, 2), (64, 2)])
@pytest.mark.parametrize("lq,lk", [(1400, 1400), (350, 98), (91, 91), (28, 28), (70, 130), (130, 257), (200, 40), (129, 600)])
def test_attention(cuda_lib, monkeypatch, d, heads, lq, lk, kernel):
    _pick_attention_kernel(monkeypatch, kernel)
    g = torch.Generator(device="cuda").manual_seed(9)
    b = 3
    c = heads * d
    q = _bf(torch.randn(b * lq, c, device="cuda", generator=g))
    k = _bf(torch.randn(b * lk, c, device="cuda", generator=g))
    v = _bf(torch.randn(b * lk, c, device="cuda", generator=g))
    scale = d ** -0.5
    out = ops.attention(q, k, v, b=b, heads=heads, lq=lq, lk=lk, d=d, ldq=c, ldk=c, ldv=c, scale=scale)
    qh = q.float().reshape(b, lq, heads, d).transpose(1, 2)
    kh = k.float().reshape(b, lk, heads, d).transpose(1, 2)
    vh = v.float().reshape(b, lk, heads, d).transpose(1, 2)
    ref = torch.softmax(qh @ kh.transpose(-1, -2) * scale, -1) @ vh
    ref = ref.transpose(1, 2).reshape(b * lq, c)
    # the xformers bf16 tolerance the reference's own kernel tests use (fmha/common.py:209-219): atol 2e-2 rtol 5e-3
    torch.testing.assert_close(out.float(), ref, atol=2e-2, rtol=5e-3)


@pytest.mark.parametrize("b,heads,d,lq,lk", [(12, 8, 40, 1400, 98), (12, 8, 40, 1337, 128), (12, 8, 40, 1400, 40), (30, 2, 32, 1400, 77),
                                             (30, 2, 64, 700, 98), (40, 8, 40, 300, 1)])
def test_attention_multi_q_tiles_per_cta(cuda_lib, monkeypatch, b, heads, d, lq, lk):
    """One K/V tile (lk <= 128) and more query tiles than CTA slots: the single-S kernel's multi-Q instantiation (a CTA keeps the
    K/V tile and walks several query tiles) against fp32 torch and, bit for bit, against the one-tile-per-CTA kernel."""
    monkeypatch.delenv("MDB_ATTN_KERNEL", raising=False)
    g = torch.Generator(device="cuda").manual_seed(29)
    c = heads * d
    q = _bf(torch.randn(b * lq, c, device="cuda", generator=g))
    k = _bf(torch.randn(b * lk, c, device="cuda", generator=g))
    v = _bf(torch.randn(b * lk, c, device="cuda", generator=g))
    scale = d ** -0.5
    monkeypatch.setenv("MDB_ATTN_MULTIQ", "1")
    out = ops.attention(q, k, v, b=b, heads=heads, lq=lq, lk=lk, d=d, ldq=c, ldk=c, ldv=c, scale=scale)
    monkeypatch.setenv("MDB_ATTN_MULTIQ", "0")
    one = ops.attention(q, k, v, b=b, heads=heads, lq=lq, lk=lk, d=d, ldq=c, ldk=c, ldv=c, scale=scale)
    qh = q.float().reshape(b, lq, heads, d).transpose(1, 2)
    kh = k.float().reshape(b, lk, heads, d).transpose(1, 2)
    vh = v.float().reshape(b, lk, heads, d).transpose(1, 2)
    ref = (torch.softmax(qh @ kh.transpose(-1, -2) * scale, -1) @ vh).transpose(1, 2).reshape(b * lq, c)
    torch.testing.assert_close(out.float(), ref, atol=2e-2, rtol=5e-3)
    assert torch.equal(out, one)


@pytest.mark.parametrize("kernel", ATTN_KERNELS)
@pytest.mark.parametrize("d,heads", [(40, 8), (80, 4)])
@pytest.mark.parametrize("lq,lk", [(300, 700), (1400, 1400)])
def test_attention_growing_scores(cuda_lib, monkeypatch, d, heads, lq, lk, kernel):
    """Scores that grow along the key axis (later key tiles dominate by far more than 2^8): exercises the running-max
    update of the online softmax, incl. the in-TMEM accumulator rescale of the tc2 kernel."""
    _pick_attention_kernel(monkeypatch, kernel)
    g = torch.Generator(device="cuda").manual_seed(19)
    b = 2
    c = heads * d
    q = _bf(torch.randn(b * lq, c, device="cuda", generator=g))
    ramp = (1.0 + 9.0 * torch.arange(lk, device="cuda") / lk).repeat(b)[:, None]  # |k| x1 .. x10 along the keys
    k = _bf(torch.randn(b * lk, c, device="cuda", generator=g) * ramp)
    v = _bf(torch.randn(b * lk, c, device="cuda", generator=g))
    scale = d ** -0.5
    out = ops.attention(q, k, v, b=b, heads=heads, lq=lq, lk=lk, d=d, ldq=c, ldk=c, ldv=c, scale=scale)
    qh = q.float().reshape(b, lq, heads, d).transpose(1, 2)
    kh = k.float().reshape(b, lk, heads, d).transpose(1, 2)
    vh = v.float().reshape(b, lk, heads, d).transpose(1, 2)
    ref = (torch.softmax(qh @ kh.transpose(-1, -2) * scale, -1) @ vh).transpose(1, 2).reshape(b * lq, c)
    torch.testing.assert_close(out.float(), ref, atol=2e-2, rtol=5e-3)


@pytest.mark.parametrize("kernel", ATTN_KERNELS)
@pytest.mark.parametrize("l,heads,d", [(350, 8, 80), (1400, 8, 40), (91, 8, 160), (130, 2, 32), (130, 2, 64), (35, 2, 64)])
def test_attention_two_sets_cross_view(cuda_lib, monkeypatch, kernel, l, heads, d):
    """attn4 'add' mode: out[view i] = attn(q_i, kv_left(i)) + attn(q_i, kv_right(i)) (blocks.py:112-121,213-217)."""
    _pick_attention_kernel(monkeypatch, kernel)
    g = torch.Generator(device="cuda").manual_seed(10)
    scenes, ncam = 2, 6
    c = heads * d
    b = scenes * ncam
    qkv = _bf(torch.randn(b * l, 3 * c, device="cuda", generator=g))
    q, k, v = qkv[:, :c], qkv[:, c:2 * c], qkv[:, 2 * c:]
    nbr = {0: [5, 1], 1: [0, 2], 2: [1, 3], 3: [2, 4], 4: [3, 5], 5: [4, 0]}
    idx = torch.tensor([[s * ncam + nbr[i][0], s * ncam + nbr[i][1]] for s in range(scenes) for i in range(ncam)],
                       dtype=torch.int32, device="cuda")
    out = ops.attention(q, k, v, b=b, heads=heads, lq=l, lk=l, d=d, ldq=3 * c, ldk=3 * c, ldv=3 * c, scale=d ** -0.5,
                        kv_index=idx, n_sets=2)
    qh = q.float().reshape(b, l, heads, d).transpose(1, 2)
    kh = k.float().reshape(b, l, heads, d).transpose(1, 2)
    vh = v.float().reshape(b, l, heads, d).transpose(1, 2)
    ref = 0
    for s in range(2):
        sel = idx[:, s].long()
        ref = ref + torch.softmax(qh @ kh[sel].transpose(-1, -2) * d ** -0.5, -1) @ vh[sel]
    ref = ref.transpose(1, 2).reshape(b * l, c)
    torch.testing.assert_close(out.float(), ref, atol=3e-2, rtol=5e-3)


def test_pointwise_and_embeddings(cuda_lib):
    g = torch.Generator(device="cuda").manual_seed(11)
    a = _bf(torch.randn(1000, 320, device="cuda", generator=g))
    b = _bf(torch.randn(1000, 320, device="cuda", generator=g))
    assert torch.equal(ops.add(a, b), (a.float() + b.float()).to(torch.bfloat16))
    # nearest resize with explicit non-integer-ratio sizes (4x7 -> 7x13 etc.)
    for (h, w, ho, wo) in [(4, 7, 7, 13), (7, 13, 14, 25), (14, 25, 28, 50), (27, 50, 53, 100)]:
        x = _bf(torch.randn(3, 64, h, w, device="cuda", generator=g))
        ref = F.interpolate(x.float(), size=(ho, wo), mode="nearest")
        out = ops.upsample_nearest(_nhwc(x), 3, h, w, 64, ho, wo)
        assert torch.equal(out, _nhwc(ref).to(torch.bfloat16))
    # layout round trip
    x = torch.randn(3, 4, 28, 50, device="cuda", generator=g)
    nh = ops.nchw_to_nhwc(x)
    assert torch.equal(nh, _nhwc(x).to(torch.bfloat16))
    back = ops.nhwc_to_nchw(nh, 3, 4, 28, 50)
    assert torch.equal(back, x.to(torch.bfloat16).float())
    # timestep embedding (embeddings.py:24-64)
    t = torch.tensor([981.0, 500.0, 1.0], device="cuda")
    half = 160
    expo = -math.log(10000) * torch.arange(half, dtype=torch.float32, device="cuda") / half
    emb = t[:, None] * torch.exp(expo)[None]
    ref = torch.cat([torch.cos(emb), torch.sin(emb)], -1)
    torch.testing.assert_close(ops.timestep_embedding(t, 320), ref, atol=2e-4, rtol=0)
    # fourier (embedder.py:15-40)
    x = torch.randn(50, 3, device="cuda", generator=g) * 10
    parts = [x]
    for f in [1.0, 2.0, 4.0, 8.0]:
        parts += [torch.sin(x * f), torch.cos(x * f)]
    torch.testing.assert_close(ops.fourier_embed(x, 4), torch.cat(parts, -1), atol=1e-5, rtol=0)


@pytest.mark.parametrize("m,k,n", [(12, 1280, 1280), (12, 320, 1280), (37, 189, 768), (240, 1536, 512)])
def test_linear_small(cuda_lib, m, k, n):
    g = torch.Generator(device="cuda").manual_seed(12)
    x = torch.randn(m, k, device="cuda", generator=g)
    w = _bf(torch.randn(n, k, device="cuda", generator=g) / math.sqrt(k))
    b = torch.randn(n, device="cuda", generator=g)
    ref = F.silu(F.silu(x) @ w.float().t() + b)
    out = ops.linear_small(x, w, b, pre_silu=True, post_silu=True)
    torch.testing.assert_close(out, ref, atol=1e-4, rtol=1e-4)


def test_conv_direct(cuda_lib):
    g = torch.Generator(device="cuda").manual_seed(13)
    x = torch.randn(2, 8, 40, 40, device="cuda", generator=g)
    wt = torch.randn(16, 8, 3, 3, device="cuda", generator=g) / 8
    b = torch.randn(16, device="cuda", generator=g)
    ref = F.silu(F.conv2d(x, wt, b, stride=(2, 1), padding=(2, 1)))
    xh = x.permute(0, 2, 3, 1).contiguous()
    out = ops.conv_direct(xh, wt.permute(2, 3, 1, 0).contiguous(), b, n=2, h=40, w=40, cin=8, cout=16, k=3, stride=(2, 1),
                          pad=(2, 1), silu=True, out_f32=True)
    torch.testing.assert_close(out.permute(0, 3, 1, 2), ref, atol=1e-4, rtol=1e-4)


def test_cfg_ddim(cuda_lib):
    g = torch.Generator(device="cuda").manual_seed(14)
    n = 6 * 4 * 28 * 50
    eps = torch.randn(2, n, device="cuda", generator=g)
    lat = torch.randn(n, device="cuda", generator=g)
    coef = torch.tensor([1.01, -0.05], device="cuda")
    ref = 1.01 * lat + (-0.05) * (eps[0] + 2.0 * (eps[1] - eps[0]))
    # eps rows are [pixel, 8] with 4 valid channels (the padded conv_out output)
    eps8 = torch.zeros(2 * (n // 4), 8, device="cuda")
    eps8[:, :4] = eps.view(-1, 4)
    out = ops.cfg_ddim_step(eps8, lat.clone().view(-1, 4), coef, True, 2.0, c=4)
    torch.testing.assert_close(out.view(-1), ref, atol=1e-6, rtol=1e-6)
    # latent packing: fp32 [pix, 4] -> bf16 [2*pix, 64]
    x = torch.randn(100, 4, device="cuda", generator=g)
    pk = ops.pack_latents(x, 64, repeat=2)
    assert pk.shape == (200, 64) and torch.equal(pk[:100, :4], x.to(torch.bfloat16)) and torch.equal(pk[100:], pk[:100])
    assert pk[:, 4:].abs().max().item() == 0
