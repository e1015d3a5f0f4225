"""Every kernel launch of a real denoising step, checked element by element against a float64 restatement of that launch
(tests/launch_check.py), for each shipped configuration: the shapes, planner routes (CTA-pair kernel, single-CTA kernel,
split-K + finalize) and activation statistics are the production ones.  Plus the sharded mode's multi-source attention
(mdb_attention_multi) on one GPU.  Each configuration appends a summary line to profiles/parity_gpu_latest.txt."""
from collections import Counter
from dataclasses import asdict

import pytest
import torch

pytestmark = pytest.mark.gpu

from magicdrive_b200 import arch, ops  # noqa: E402
from magicdrive_b200.models import AutoencoderKL, BEVControlNetModel, UNet2DConditionModelMultiview  # noqa: E402
from magicdrive_b200.synthetic import synthetic_inputs  # noqa: E402
from tests import ops_emulator as emu  # noqa: E402
from tests.common import record, tiny_configs, tiny_state_dicts, to_dev  # noqa: E402
from tests.launch_check import ATTN2, LaunchChecker, _compute_dtype, denoise_step, err_over_tol  # noqa: E402

DEV = "cuda"
BF16 = torch.bfloat16


@pytest.fixture(scope="module")
def sd15(cuda_lib):
    """The benchmark's networks (bench.py): SD-1.5-size UNet + BEVControlNet, synthetic weights 11 / 12, bf16."""
    un = UNet2DConditionModelMultiview(**asdict(arch.UNetConfig())).reset_parameters_synthetic(11).to(DEV, BF16)
    cn = BEVControlNetModel(**asdict(arch.ControlNetConfig(map_size=(8, 200, 200)))).reset_parameters_synthetic(12).to(DEV, BF16)
    return un, cn


def _per_op(counts):
    c = Counter()
    for (op, _), n in counts.items():
        c[op] += n
    return c


def _check_step(name, un, cn, h, w, map_hw, scenes=1):
    inp = to_dev(synthetic_inputs(scenes, 6, h, w, n_box=20, map_hw=map_hw, seed=0), DEV)
    with torch.no_grad(), LaunchChecker(name) as chk:
        launches = denoise_step(chk, un, cn, inp)
    chk.assert_all_close()
    return chk, launches


def test_configs2_224x400_every_launch(sd15):
    """The benchmark workload: 6 views, 28 x 50 latents, 20 boxes, 200 x 200 map, CFG 2.0 (V = 12)."""
    un, cn = sd15
    chk, launches = _check_step("configs[2] 224x400 V=12", un, cn, 28, 50, 200)
    step = chk.counts("step")
    # The launch mix of the step in profiles/launches_step_r2_final.summary.txt (the captured CUDA graph of the overlapped
    # two-stream step): the single-stream eager step issues the same kernels, the ControlNet residual additions riding the
    # zero convolutions' epilogues in both.
    assert _per_op(step) == {"gemm_conv": 321, "attention": 62, "groupnorm": 88, "upsample_nearest": 3, "pack_latents": 1,
                             "cfg_ddim_step": 1}, _per_op(step)
    # the M = 336 GEMMs of the 4 x 7 level: ResNet convolutions and 1x1 shortcuts (per-image shift, four images per tile),
    # the zero convolutions with the UNet skip as residual and out_scale, the mid block's token GEMMs
    assert step[("gemm_conv", "splitk")] == 37, step
    assert launches == 513


def test_configs3_424x800_every_launch(sd15):
    """53 x 100 latents (5300-token attention), 400 x 400 map: the same networks, as bench.py's configs[3] sub-record."""
    un, cn = sd15
    chk, _ = _check_step("configs[3] 424x800 V=12", un, cn, 53, 100, 400)
    # No split-K at this size: the deepest level is 7 x 13 (91 pixels, one image per M tile), where the 1280-wide GEMMs
    # already have 90 to 120 CTAs (9 to 12 M tiles x 10 N tiles), more than half the 148 SMs (capi_gemm.cu make_plan).
    assert chk.counts("step")[("gemm_conv", "splitk")] == 0


def test_272x736_every_launch(sd15):
    """configs/exp/272x736.yaml: 34 x 92 latents (odd pyramid 17 x 46, 9 x 23, 5 x 12) with 12 view-samples, and the ...Plus map
    encoder pooling the 200 x 200 map to the latent grid (adaptive_avgpool)."""
    un, _ = sd15
    ccfg = arch.ControlNetConfig(map_size=(8, 200, 200), map_embedding_size=(34, 92))
    cn = BEVControlNetModel(**asdict(ccfg)).reset_parameters_synthetic(12).to(DEV, BF16)
    chk, _ = _check_step("272x736 V=12", un, cn, 34, 92, 200)
    assert chk.counts("step")[("gemm_conv", "splitk")] > 0
    assert chk.counts("prepare")[("adaptive_avgpool", "")] == 1


def test_configs0_stock_unet_every_launch(cuda_lib):
    """BASELINE.json configs[0]: the stock single-view SD-1.5 UNet2DConditionModel call (no ControlNet, text only), 28 x 50."""
    un = UNet2DConditionModelMultiview.stock_unet().reset_parameters_synthetic(11).to(DEV, BF16)
    g = torch.Generator().manual_seed(6)
    x, text = torch.randn(1, 4, 28, 50, generator=g).to(DEV), torch.randn(1, 77, 768, generator=g).to(DEV)
    with torch.no_grad(), LaunchChecker("configs[0] stock UNet 1 view") as chk, chk.phase("step"):
        un(x, torch.tensor(981.0, device=DEV), encoder_hidden_states=text)
    chk.assert_all_close()
    assert chk.counts()[("attention", "")] == 32  # 16 transformers: self and text cross-attention, no cross-view attention


def test_vae_decode_every_launch(cuda_lib):
    """AutoencoderKL.decode_latents of configs[2]'s six 28 x 50 latents (eager: the checker cannot run inside a graph
    capture): GroupNorms over 224 x 400 maps, the fp32 scores of the single-head attention (ldo = padded key count),
    softmax_rows, the narrow fp32 conv_out."""
    vae = AutoencoderKL(**asdict(arch.VaeConfig())).reset_parameters_synthetic(13).to(DEV, BF16)
    vae.use_cuda_graph = False
    lat = synthetic_inputs(1, 6, 28, 50, n_box=0, map_hw=8, seed=0)["latents"]
    lat5 = torch.stack([lat] * 6, 1).to(DEV) * 0.18215
    with torch.no_grad(), LaunchChecker("VAE decode 6 x 224x400") as chk, chk.phase("decode"):
        vae.decode_latents(lat5)
    chk.assert_all_close()
    assert chk.counts()[("softmax_rows", "")] == 6


def test_tiny_config_every_launch(cuda_lib):
    """64 / 128 channels, head dims 32 / 64: the block_n = 64 and K = 64 corners of the GEMM, two scenes (V = 24)."""
    ucfg, ccfg = tiny_configs()
    usd, csd = tiny_state_dicts(7)
    un, cn = UNet2DConditionModelMultiview(**asdict(ucfg)), BEVControlNetModel(**asdict(ccfg))
    un.load_state_dict(usd)
    cn.load_state_dict(csd)
    _check_step("tiny 10x13 V=24", un.to(DEV, BF16), cn.to(DEV, BF16), 10, 13, 52, scenes=2)


# ---------------------------------------------------------------------------- sharded mode's attention on one GPU
NEIGHBOURS = {0: [5, 1], 1: [0, 2], 2: [1, 3], 3: [2, 4], 4: [3, 5], 5: [4, 0]}  # ring of the 6 cameras (Nuscenes.yaml)
OWNER = {0: [0, 3, 6, 9, 11], 1: [1, 4, 7], 2: [2, 5, 8, 10]}  # buffer holding each view-sample's K/V: b_kv 5 / 3 / 4


@pytest.mark.parametrize("layout", ["engine", "wide_ld"])
@pytest.mark.parametrize("d,L", [(40, 1400), (80, 350), (160, 91)])
def test_attention_multi_three_sources(cuda_lib, d, L, layout):
    """mdb_attention_multi with the neighbour K/V of 2 scenes x 6 cameras spread over three [K | V] buffers laid out as
    engine.py's sharded branch does (row stride 2C, unequal b_kv; `wide_ld`: one buffer with 64 spare columns per row,
    filled with garbage).  It must equal, bit for bit, ops.attention on one buffer holding the same view-samples with the
    indices rebased (same arithmetic: any difference is an addressing error), and agree with the float64 reference."""
    heads, scenes, ncam = 8, 2, 6
    c, b = heads * d, scenes * ncam
    g = torch.Generator(device=DEV).manual_seed(d)
    q = torch.randn(b * L, c, device=DEV, generator=g).to(BF16)
    kv = torch.randn(b * L, 2 * c, device=DEV, generator=g).to(BF16)  # [K | V] of every view-sample, view-sample major
    srcs, where = [], {}
    for s, views in OWNER.items():
        ld = 2 * c + (64 if layout == "wide_ld" and s == 1 else 0)
        buf = torch.randn(len(views) * L, ld, device=DEV, generator=g).to(BF16) * 100
        for j, v in enumerate(views):
            buf[j * L:(j + 1) * L, :2 * c] = kv[v * L:(v + 1) * L]
            where[v] = (s, j)
        srcs.append((buf, buf[:, c:], ld, len(views)))
    glob = [[sc * ncam + NEIGHBOURS[i][0], sc * ncam + NEIGHBOURS[i][1]] for sc in range(scenes) for i in range(ncam)]
    idx_multi = torch.tensor([[(where[v][0] << 24) | where[v][1] for v in row] for row in glob], dtype=torch.int32, device=DEV)
    idx_one = torch.tensor(glob, dtype=torch.int32, device=DEV)
    assert {int(x) >> 24 for x in idx_multi.flatten()} == {0, 1, 2}
    kw = dict(b=b, heads=heads, lq=L, lk=L, d=d, scale=d ** -0.5, n_sets=2)
    out = ops.attention_multi(q, srcs, ldq=c, kv_index=idx_multi, **kw)
    one = ops.attention(q, kv, kv[:, c:], ldq=c, ldk=2 * c, ldv=2 * c, kv_index=idx_one, **kw)
    with _compute_dtype(torch.float64):
        ref = emu.attention(q, kv, kv[:, c:], ldq=c, ldk=2 * c, ldv=2 * c, kv_index=idx_one, **kw)
    torch.cuda.synchronize()
    e = err_over_tol(out, ref, ATTN2)
    record(f"[launch-parity] attention_multi 3 sources d={d} L={L} {layout}: err/tol {e:.3f} vs float64, "
           f"bit-identical to the one-buffer launch: {torch.equal(out, one)}")
    assert torch.equal(out, one), (out.float() - one.float()).abs().max().item()
    assert e <= 1.0, e
