"""Launch checker: every call a real model step makes into magicdrive_b200.ops, checked element by element against a
float64 restatement of that same call (tests/ops_emulator.py) computed from the exact inputs the kernel received.

The per-operator GPU tests run hand-picked shapes, often with the kernel route forced; the whole-model tests compare a few
taps by a norm that dilutes a local mistake.  Here the shapes, the planner's routes (CTA-pair kernel, single-CTA kernel,
split-K + finalize) and the activation statistics are the production ones by construction:

    with LaunchChecker("configs[2]") as chk:
        pipe = BEVControlNetDenoiser(...)          # built inside: the denoiser reads its A/B switches at construction
        with chk.phase("step"):
            pipe.run_steps(st, 0, 1)
    chk.assert_all_close()

Each launch is compared with the criterion its per-operator test uses, relative to the reference's largest magnitude so
that real activation scales work; failures are collected, not raised one by one."""
import contextlib
import os
import time
from collections import Counter

import pytest
import torch

from magicdrive_b200 import ops
from tests import ops_emulator as emu
from tests.common import record

# A/B switches that select non-default kernels or launch modes: the checker runs the production defaults
PINNED_ENV = ("MDB_GEMM_VARIANT", "MDB_ATTN_KERNEL", "MDB_ATTN_MULTIQ", "MDB_GN_ROWS", "MDB_GN_TWO_KERNEL",
              "MDB_FUSE_RESIDUAL_ADDS")

# Operators checked: what the emulator restates, except `linear` (it reaches the device through gemm_conv, which is wrapped)
CHECKED = [n for n in emu.EMULATED if n not in ("linear", "workspace_slot")]

# (relative to |ref|, relative to max|ref|, absolute) bound per element; all zero = bit-exact
BF16 = (2.0 ** -7, 2e-3, 0.0)     # one bf16 rounding step plus accumulation-order slack (test_gemm_pair_gpu._close_bf16)
F32 = (0.0, 2e-5, 0.0)            # fp32 outputs of the tensor-core GEMM (test_kernels_gpu.test_gemm_plain)
NORM = (0.0, 8e-3, 0.0)           # GroupNorm / LayerNorm (test_kernels_gpu.test_groupnorm)
ATTN = (5e-3, 2e-2, 0.0)          # xformers' bf16 attention tolerance (test_kernels_gpu.test_attention)
ATTN2 = (5e-3, 3e-2, 0.0)         # two key sets summed (test_kernels_gpu.test_attention_two_sets_cross_view)
SCHED = (1e-6, 1e-6, 0.0)         # guidance + scheduler update in fp32 (test_kernels_gpu.test_cfg_ddim)
TEMB = (0.0, 0.0, 2e-4)           # sinusoidal embedding of timesteps up to 1000 (test_pointwise_and_embeddings)
FOURIER = (0.0, 0.0, 1e-5)        # sin / cos of power-of-two multiples (test_pointwise_and_embeddings)
EXACT = (0.0, 0.0, 0.0)

_FIXED = {"groupnorm": NORM, "layernorm": NORM, "add": EXACT, "upsample_nearest": EXACT, "adaptive_avgpool": F32,
          "linear_small": F32, "timestep_embedding": TEMB, "fourier_embed": FOURIER, "nchw_to_nhwc": EXACT,
          "nhwc_to_nchw": EXACT, "f32_to_bf16": EXACT, "pack_latents": EXACT, "cfg_ddim_step": SCHED,
          "cfg_unipc_step": SCHED, "pin_views": SCHED, "softmax_rows": BF16}


def err_over_tol(out, ref, crit):
    """max over elements of |out - ref| / bound (<= 1 passes).  A bit-exact criterion gives 0 or inf and compares with the
    reference rounded once to the output's dtype (a bf16 conversion must round to nearest even, nothing else)."""
    if crit == EXACT:
        ref = ref.to(out.dtype)
    out, ref = out.double(), ref.double()
    if out.shape != ref.shape:
        return float("inf")
    if out.numel() == 0:
        return 0.0
    rel, of_max, absolute = crit
    err = (out - ref).abs()
    tol = ref.abs() * rel + of_max * ref.abs().max() + absolute
    r = torch.where(err == 0, torch.zeros_like(err), err / tol)  # err / 0 = inf where the criterion is exact
    return float(r.max()) if torch.isfinite(out).all() else float("nan")


def stats_err_over_tol(dev_stats, ref_stats, ref_out):
    """Emitted row statistics: per row, the sum over partial slots of (sum, sum of squares) against the float64 sums of the
    reference output before its bf16 rounding.  Bound: the fp32 output criterion of every element, summed over the row."""
    s, r = dev_stats.data.double().sum(1), ref_stats.data.double().sum(1)
    c, m = ref_out.shape[1], ref_out.double().abs().max().item()
    tol_sum = F32[1] * c * m + 1e-30
    tol_sq = 2 * F32[1] * c * m * m + 1e-30
    e = max(((s[:, 0] - r[:, 0]).abs().max() / tol_sum).item(), ((s[:, 1] - r[:, 1]).abs().max() / tol_sq).item())
    return e if torch.isfinite(s).all() else float("nan")


def _per_image_tiles(n_img, h, w):
    """Several images share one 128-row M tile (capi_gemm.cu choose_box)."""
    return h * w <= 128 and min(128 // (h * w), n_img) > 1


def gemm_route(kw, launches):
    """The kernel mdb_gemm_conv ran: two launches = split-K + finalize on gemm_tc2; otherwise the CTA-pair kernel unless the
    descriptor is one it refuses (fp32 / narrow outputs, a per-image shift with several images per tile, an operand the
    epilogue cannot bulk-copy) -- the conditions of capi_gemm.cu pair_supported."""
    if launches == 2:
        return "splitk"
    n_out, geglu = kw["n_out"], kw.get("geglu", False)
    out_cols = n_out // 2 if geglu else n_out
    rb = kw.get("rowbias")
    misaligned = any(t is not None and t.data_ptr() % 16 for t in (kw.get("bias"), rb, kw.get("ln_colsum")))
    per_image = rb is not None and rb.shape[0] > 1 and (_per_image_tiles(kw["n_img"], kw["h_out"], kw["w_out"]) or rb.stride(0) % 4)
    if kw.get("out_f32") or out_cols % 32 or n_out % 32 or per_image or misaligned:
        return "tc2"
    return "pair"


def _clone(t):
    """A copy with the same strides (a column slice of a wider buffer stays one: the operators read by row stride)."""
    if not torch.is_tensor(t):
        return t
    c = torch.empty_strided(t.size(), t.stride(), dtype=t.dtype, device=t.device)
    c.copy_(t)
    return c


def _fmt(v):
    if torch.is_tensor(v):
        return "x".join(map(str, v.shape)) + ":" + str(v.dtype).replace("torch.", "")
    return repr(v)


def _shape_kw(kw):
    """h_out / w_out of a gemm_conv call as the operator defaults them."""
    taps, stride, pad = kw.get("taps", 1), kw.get("stride", 1), kw.get("pad", 0)
    return {"h_out": kw.get("h_out") or (kw["h_in"] + 2 * pad - taps) // stride + 1,
            "w_out": kw.get("w_out") or (kw["w_in"] + 2 * pad - taps) // stride + 1}


def _gemm_sig(kw):
    taps, stride = kw.get("taps", 1), kw.get("stride", 1)
    h_out, w_out = _shape_kw(kw).values()
    rb = kw.get("rowbias")
    bits = [f"M={kw['n_img'] * h_out * w_out} N={kw['n_out']} K={taps * taps * (kw['c0'] + kw.get('c1', 0))}",
            f"img={kw['n_img']}x{h_out}x{w_out} taps={taps} s={stride}"]
    bits += [f for f, on in (("two-src", kw.get("c1", 0) > 0), ("bias", kw.get("bias") is not None),
                             ("geglu", kw.get("geglu", False)), ("ln", kw.get("ln") is not None),
                             ("stats", kw.get("emit_stats", False)), ("res", kw.get("residual") is not None),
                             ("out=", kw.get("out") is not None)) if on]
    if rb is not None:
        bits.append(f"shift[{rb.shape[0]}]")
    if kw.get("out_scale", 1.0) != 1.0:
        bits.append(f"scale={kw['out_scale']:g}")
    bits.append("f32" if kw.get("out_f32") else "bf16")
    return " ".join(bits)


def _sig(name, args, kw):
    if name == "gemm_conv":
        return _gemm_sig(kw)
    if name == "attention":
        return (f"B={kw['b']} H={kw['heads']} Lq={kw['lq']} Lk={kw['lk']} D={kw['d']} sets={kw.get('n_sets', 1)} "
                f"ld={kw['ldq']}/{kw['ldk']}/{kw['ldv']}" + (f" b_kv={kw['b_kv']}" if kw.get("b_kv") else ""))
    return " ".join([_fmt(a) for a in args] + [f"{k}={_fmt(v)}" for k, v in kw.items() if v is not None])


@contextlib.contextmanager
def _compute_dtype(dtype):
    old, emu.COMPUTE_DTYPE = emu.COMPUTE_DTYPE, dtype
    try:
        yield
    finally:
        emu.COMPUTE_DTYPE = old


class LaunchChecker:
    """Wraps the operators of magicdrive_b200.ops for the duration of a `with` block (see the module docstring).  The
    operators in place when the block is entered are the "device": the CUDA library, or the emulator on a machine
    without a GPU (tests/test_launch_check_cpu.py)."""

    def __init__(self, name: str, ref_dtype=torch.float64):
        self.mp, self.name, self.ref_dtype = pytest.MonkeyPatch(), name, ref_dtype
        self.rows = []  # (index, phase, op, route, signature, err / tol)
        self.stage = ""
        self.t0 = None

    def __enter__(self):
        mp = self.mp
        for k in list(os.environ):
            if k in PINNED_ENV or k.startswith("MDB_PDL"):
                mp.delenv(k)
        mp.setattr(ops, "GEMM_VARIANT", 0)  # read from the environment at import time
        # the reference is float64 throughout; make sure no fp32 path of torch could drop to TF32 either
        mp.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
        mp.setattr(torch.backends.cudnn, "allow_tf32", False)
        mp.setattr(emu, "ROUND_ACTIVATIONS", False)
        for name in CHECKED:
            mp.setattr(ops, name, self._wrap(name, getattr(ops, name)))
        self.t0 = time.time()
        return self

    def __exit__(self, *exc):
        self.seconds = time.time() - self.t0
        self.mp.undo()
        return False

    @contextlib.contextmanager
    def phase(self, label: str):
        old, self.stage = self.stage, label
        try:
            yield
        finally:
            self.stage = old

    def _wrap(self, name, device_fn):
        ref_fn = getattr(emu, name)

        def checked(*args, **kw):
            rargs = [_clone(a) for a in args]
            rkw = {k: (None if k == "out" else _clone(v)) for k, v in kw.items()}
            with _compute_dtype(self.ref_dtype):
                ref = ref_fn(*rargs, **rkw)
            n0 = ops.launch_count()
            got = device_fn(*args, **kw)
            launches = ops.launch_count() - n0
            sig = _sig(name, args, kw)
            route, err = "", 0.0
            if name == "gemm_conv":
                route = gemm_route({**kw, **_shape_kw(kw)}, launches)
                dev, dev_stats = got if kw.get("emit_stats") else (got, None)
                ref_out, ref_stats = ref if kw.get("emit_stats") else (ref, None)
                width = ref_out.shape[1]
                err = err_over_tol(dev[: ref_out.shape[0], :width], ref_out, F32 if kw.get("out_f32") else BF16)
                if dev_stats is not None:
                    err = max(err, stats_err_over_tol(dev_stats, ref_stats, ref_out))
            elif name == "attention":
                c = kw["heads"] * kw["d"]
                err = err_over_tol(got[:, :c], ref, ATTN2 if kw.get("n_sets", 1) > 1 else ATTN)
            elif name == "conv_direct":
                err = err_over_tol(got, ref, F32 if kw.get("out_f32") else BF16)
            else:
                err = err_over_tol(got, ref, _FIXED[name])
            self.rows.append((len(self.rows), self.stage, name, route, sig, err))
            return got

        return checked

    # ------------------------------------------------------------------ results
    def counts(self, phase=None):
        """Counter of (operator, route) over the launches of `phase` (all phases when None)."""
        return Counter((op, route) for _, ph, op, route, _, _ in self.rows if phase is None or ph == phase)

    def failures(self):
        return [r for r in self.rows if not r[5] <= 1.0]

    def worst(self):
        """{(operator, route): (err / tol, signature)} of the worst launch of each."""
        w = {}
        for _, _, op, route, sig, err in self.rows:
            key = (op, route)
            if key not in w or not err <= w[key][0]:
                w[key] = (err, sig)
        return w

    def summary(self) -> str:
        cnt = self.counts()
        by = ", ".join(f"{op}{'/' + rt if rt else ''} {n}" for (op, rt), n in sorted(cnt.items()))
        worst = ", ".join(f"{op}{'/' + rt if rt else ''} {e:.2f}" for (op, rt), (e, _) in sorted(self.worst().items()))
        return (f"[launch-parity] {self.name}: {len(self.rows)} launches checked against float64 ({by}); "
                f"worst err/tol: {worst}; {len(self.failures())} failing; {getattr(self, 'seconds', 0.0):.1f} s")

    def assert_all_close(self, log: bool = True):
        if log:
            record(self.summary())
        bad = self.failures()
        if bad:
            lines = [f"  #{i} [{ph}] {op}{'/' + rt if rt else ''} {sig}: err/tol {e:.3g}" for i, ph, op, rt, sig, e in bad]
            worst = [f"  {op}{'/' + rt if rt else ''}: {e:.3g} at {sig}" for (op, rt), (e, sig) in sorted(self.worst().items())]
            raise AssertionError(f"{self.name}: {len(bad)} of {len(self.rows)} launches outside their criterion\n"
                                 + "\n".join(lines) + "\nworst per operator / route:\n" + "\n".join(worst))


def denoise_step(chk, un, cn, inp, guidance_scale=2.0):
    """prepare() + the first DDIM step of BEVControlNetDenoiser, eager and on one stream, under `chk` (phases "prepare" and
    "step"; call it inside the checker's block: the denoiser reads its A/B switches when it is built).  The single-stream
    branch of the step (pipeline.BEVControlNetDenoiser._step_models) issues the launches of the overlapped production path.
    Returns the number of kernels the step launched."""
    from magicdrive_b200.pipeline import BEVControlNetDenoiser
    pipe = BEVControlNetDenoiser(un, cn, use_cuda_graph=False, overlap_controlnet=False)
    with chk.phase("prepare"):
        st = pipe.prepare(inp["latents"], inp["prompt_embeds"], inp["negative_prompt_embeds"], inp["camera_param"],
                          inp["bboxes_3d_data"], inp["bev_map"], guidance_scale=guidance_scale)
        pipe.set_schedule(st, 50)
    n0 = ops.launch_count()
    with chk.phase("step"):
        pipe.run_steps(st, 0, 1)
    return ops.launch_count() - n0
