"""The launch checker's own test, without a GPU: the fp32 operator restatements play the device at the tiny configuration.
Against their float64 selves every launch must pass; a device whose gemm_conv is wrong in one small way in one launch
must be reported at exactly that launch.  This shows the criteria of tests/launch_check.py are sharp before a B200 runs
tests/test_zz_launch_parity_gpu.py."""
from dataclasses import asdict

import pytest
import torch

from magicdrive_b200 import models, ops
from magicdrive_b200.synthetic import synthetic_inputs
from tests import ops_emulator
from tests.common import tiny_configs, tiny_state_dicts
from tests.launch_check import LaunchChecker, denoise_step


@pytest.fixture
def tiny(monkeypatch):
    ops_emulator.install(monkeypatch)
    ucfg, ccfg = tiny_configs()
    usd, csd = tiny_state_dicts(7)
    un, cn = models.UNet2DConditionModelMultiview(**asdict(ucfg)), models.BEVControlNetModel(**asdict(ccfg))
    un.load_state_dict(usd)
    cn.load_state_dict(csd)
    return un, cn, synthetic_inputs(1, 6, 10, 13, n_box=3, map_hw=52, seed=9)


def _run(tiny, name):
    un, cn, inp = tiny
    with torch.no_grad(), LaunchChecker(name) as chk:
        denoise_step(chk, un, cn, inp)
    return chk


def test_emulated_device_passes_every_launch_and_counts_repeat(tiny):
    a = _run(tiny, "tiny (fp32 emulator as device)")
    a.assert_all_close(log=False)
    b = _run(tiny, "tiny (fp32 emulator as device, again)")
    b.assert_all_close(log=False)
    assert a.counts() == b.counts() and [r[4] for r in a.rows] == [r[4] for r in b.rows]
    step = a.counts("step")
    ops_in_step = {op for op, _ in step}
    assert {"gemm_conv", "attention", "groupnorm", "upsample_nearest", "pack_latents", "cfg_ddim_step"} <= ops_in_step
    assert {op for op, _ in a.counts("prepare")} >= {"linear_small", "fourier_embed", "conv_direct", "timestep_embedding"}
    # the reference is the same restatement in float64: the fp32 "device" sits far inside every criterion
    assert max(r[5] for r in a.rows if r[2] == "gemm_conv") < 0.05


def _ulp_bf16(x):
    return torch.exp2(torch.floor(torch.log2(x.abs().clamp_min(1e-30))) - 7)


@pytest.mark.parametrize("fault", ["row_4ulp", "residual_dropped"])
def test_one_wrong_gemm_launch_is_reported_alone(tiny, monkeypatch, fault):
    """One launch of the step gets one output row off by 4 bf16 ulps, or loses its residual: that launch fails, no other."""
    emulated = ops.gemm_conv
    hit = {}

    def faulty(*args, **kw):
        chk = hit["chk"]
        pick = chk.stage == "step" and "row" not in hit and (fault == "row_4ulp" or kw.get("residual") is not None)
        if pick and fault == "residual_dropped":
            kw = dict(kw, residual=None)
        out = emulated(*args, **kw)
        if pick:
            hit["row"] = len(chk.rows)  # the checker appends this launch's row after the device call returns
            if fault == "row_4ulp":
                y = out[0] if kw.get("emit_stats") else out
                r = y.shape[0] // 3
                y[r] += 4 * _ulp_bf16(y[r])
        return out

    monkeypatch.setattr(ops, "gemm_conv", faulty)
    un, cn, inp = tiny
    with torch.no_grad(), LaunchChecker(f"tiny, {fault}") as chk:
        hit["chk"] = chk
        denoise_step(chk, un, cn, inp)
    bad = chk.failures()
    assert [r[0] for r in bad] == [hit["row"]], [(r[0], r[4], r[5]) for r in bad]
    assert bad[0][2] == "gemm_conv" and bad[0][1] == "step"
    with pytest.raises(AssertionError, match=r"1 of \d+ launches outside"):
        chk.assert_all_close(log=False)
