"""GPU parity of the VAE encoder (AutoencoderKL(with_encoder=True)): the image-patch pack and latent-distribution kernels,
the stride-2 convolution with Downsample2D(padding=0)'s far-edge zero row and column on both GEMM kernels, encode against
the fp32 oracle restatement of AutoencoderKL.encode (pinned to the reference in tests/test_vae_encode_cpu.py) with the
decoder's criterion err(ours) <= 1.5 x err(reference arithmetic in bf16) + 2e-3, the CUDA-graph replay of encode_latents,
and every launch of a 6-view 224x400 encode against float64."""
from dataclasses import asdict

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from magicdrive_b200 import arch, ops  # noqa: E402
from magicdrive_b200.models import AutoencoderKL  # noqa: E402
from oracle import torch_oracle_vae_encode as OE  # noqa: E402  (checker only)
from tests import vae_encode_emulation  # noqa: E402
from tests.common import max_rel, record, rel_l2  # noqa: E402
from tests.launch_check import SCHED, LaunchChecker, err_over_tol  # noqa: E402

DEV = "cuda"
BF16 = torch.bfloat16


@pytest.fixture(autouse=True)
def _no_tf32():
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


@pytest.mark.parametrize("dtype", [torch.float32, BF16])
@pytest.mark.parametrize("n,h,w", [(2, 80, 104), (6, 224, 400), (1, 37, 45)])
def test_pack_image_patches_bit_exact(cuda_lib, dtype, n, h, w):
    x = (torch.rand(n, 3, h, w, generator=torch.Generator().manual_seed(h)) * 2 - 1).to(DEV, dtype)
    got = ops.pack_image_patches(x)
    cols = F.unfold(x.float(), 3, padding=1).reshape(n, 3, 9, h * w).permute(0, 3, 2, 1).reshape(n * h * w, 27)
    ref = F.pad(cols, (0, 37)).to(BF16)
    assert got.shape == (n * h * w, 64) and torch.equal(got, ref)


@pytest.mark.parametrize("with_noise", [False, True])
def test_latent_dist_vs_float64(cuda_lib, with_noise):
    n, h, w = 6, 28, 50
    g = torch.Generator().manual_seed(4)
    mom = torch.randn(n * h * w, 8, generator=g)
    mom[:, 4:] = mom[:, 4:] * 15  # logvar beyond both clamp bounds too
    noise = torch.randn(n, 4, h, w, generator=g) if with_noise else None
    scale = 0.18215
    got = ops.latent_dist(mom.to(DEV), n, h, w, 4, noise=None if noise is None else noise.to(DEV), scale=scale)
    m = mom.double().reshape(n, h, w, 8).permute(0, 3, 1, 2)
    ref = m[:, :4] if noise is None else m[:, :4] + torch.exp(0.5 * m[:, 4:].clamp(-30, 20)) * noise.double()
    ref = scale * ref
    assert got.shape == (n, 4, h, w) and got.dtype == torch.float32
    assert err_over_tol(got.cpu(), ref, SCHED) <= 1.0
    if noise is None:  # scale * mean is one fp32 product
        assert torch.equal(got.cpu(), scale * m[:, :4].float())


@pytest.mark.parametrize("variant", [0, 2, 3])
@pytest.mark.parametrize("h,w", [(224, 400), (112, 200), (56, 100), (53, 100)])
@pytest.mark.parametrize("c", [128, 256, 512])
def test_gemm_conv_stride2_far_edge_pad(cuda_lib, c, h, w, variant):
    """Downsample2D(padding=0): F.pad(x, (0, 1, 0, 1)) + 3x3 stride-2 conv == mdb_gemm_conv with pad 0 and
    h_out = (h - 2) // 2 + 1; two images, so a tap past the bottom edge of image 0 must read zeros, not image 1."""
    n = 2
    g = torch.Generator().manual_seed(c + h + variant)
    x = torch.randn(n, c, h, w, generator=g).to(BF16)
    wt = (torch.randn(c, c, 3, 3, generator=g) / (3 * c ** 0.5)).to(BF16)
    b = torch.randn(c, generator=g) * 0.1
    ref = F.conv2d(F.pad(x.float().to(DEV), (0, 1, 0, 1)), wt.float().to(DEV), b.to(DEV), stride=2)
    ho, wo = (h - 2) // 2 + 1, (w - 2) // 2 + 1
    assert ref.shape[2:] == (ho, wo)
    xn = x.permute(0, 2, 3, 1).reshape(-1, c).contiguous().to(DEV)
    wp = wt.permute(0, 2, 3, 1).reshape(c, 9 * c).contiguous().to(DEV)
    out = ops.gemm_conv(xn, wp, n_img=n, h_in=h, w_in=w, c0=c, lda0=c, n_out=c, taps=3, stride=2, pad=0, h_out=ho, w_out=wo,
                        bias=b.to(DEV), kernel_variant=variant)
    out = out.reshape(n, ho, wo, c).permute(0, 3, 1, 2).float()
    err = (out - ref).abs()
    tol = ref.abs() * 2.0 ** -7 + 2e-3 * ref.abs().max()  # test_gemm_pair_gpu._close_bf16
    assert (err > tol).sum().item() == 0, f"max err {err.max().item():.3e}, rel-L2 {rel_l2(out, ref):.3e}"


def _vae(cfg, seed):
    shapes = dict(arch.vae_encoder_param_shapes(cfg), **arch.vae_decoder_param_shapes(cfg))
    sd = arch.synthetic_state_dict(shapes, seed)
    vae = AutoencoderKL(**asdict(cfg), with_encoder=True)
    vae.load_state_dict(sd)
    return vae.to(DEV, BF16), sd


@torch.no_grad()
@pytest.mark.parametrize("name,cfg,n,h,w", [("small", arch.VaeConfig(block_out_channels=(64, 128, 128, 128)), 3, 80, 104),
                                            ("sd15", arch.VaeConfig(), 2, 224, 400),
                                            ("sd15", arch.VaeConfig(), 1, 424, 800)])
def test_vae_encode_vs_oracle(cuda_lib, name, cfg, n, h, w):
    vae, sd = _vae(cfg, 81)
    x = torch.rand(n, 3, h, w, generator=torch.Generator().manual_seed(h)) * 2 - 1
    post = vae.encode(x.to(DEV, BF16)).latent_dist
    truth = OE.posterior(OE.vae_encode({k: v.to(DEV) for k, v in sd.items()}, cfg, x.to(DEV)))
    yard = OE.posterior(OE.vae_encode({k: v.to(DEV, BF16) for k, v in sd.items()}, cfg, x.to(DEV, BF16)))
    assert post.mean.shape == truth["mean"].shape == (n, 4, h // 8, w // 8)
    for k in ("mean", "logvar"):
        e, ey = rel_l2(getattr(post, k), truth[k]), rel_l2(yard[k], truth[k])
        record(f"[parity] vae encode {name} {n}x{h}x{w} {k}: rel-L2 ours {e:.3e} reference-bf16 {ey:.3e} "
               f"max-rel ours {max_rel(getattr(post, k), truth[k]):.3e}")
        assert e <= 1.5 * ey + 2e-3, (k, e, ey)


@torch.no_grad()
def test_encode_latents_graph_replay_is_bit_identical(cuda_lib):
    vae, _ = _vae(arch.VaeConfig(), 82)
    px = (torch.rand(1, 3, 3, 224, 400, generator=torch.Generator().manual_seed(2)) * 2 - 1).to(DEV)
    eager = vae.encode(px[0]).latent_dist.mean * vae.config.scaling_factor
    for _ in range(2):  # capture, then a plain replay
        z = vae.encode_latents(px)
        assert z.shape == (1, 3, 4, 28, 50) and z.is_cuda and torch.equal(z[0], eager)
    # sampling: the noise is drawn outside the graph; replay == an eager run with the same generator seed
    zs = vae.encode_latents(px, sample=True, generator=torch.Generator().manual_seed(5))
    vae.use_cuda_graph = False
    ze = vae.encode_latents(px, sample=True, generator=torch.Generator().manual_seed(5))
    assert torch.equal(zs, ze) and not torch.equal(zs, z)


def test_vae_encode_every_launch(cuda_lib, monkeypatch):
    """An eager encode_latents of six 224 x 400 views: GroupNorms over full-resolution maps, the K = 64 conv_in, the
    stride-2 pad-(0, 1, 0, 1) downsamples, the 1400-token single-head attention, the folded fp32 conv_out."""
    vae = AutoencoderKL(**asdict(arch.VaeConfig()), with_encoder=True).reset_parameters_synthetic(14).to(DEV, BF16)
    vae.use_cuda_graph = False
    vae_encode_emulation.checker(monkeypatch)
    px = (torch.rand(1, 6, 3, 224, 400, generator=torch.Generator().manual_seed(0)) * 2 - 1).to(DEV)
    with torch.no_grad(), LaunchChecker("VAE encode 6 x 224x400") as chk, chk.phase("encode"):
        vae.encode_latents(px)
    chk.assert_all_close()
    cnt = chk.counts()
    assert cnt[("pack_image_patches", "")] == 1 and cnt[("latent_dist", "")] == 1 and cnt[("softmax_rows", "")] == 6
