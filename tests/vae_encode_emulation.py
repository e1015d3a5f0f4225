"""TEST INFRASTRUCTURE ONLY — what the VAE encoder adds to the operator restatements of tests/ops_emulator.py, kept beside
it: the two new operators (mdb_pack_image_patches, mdb_latent_dist) and gemm_conv with taps past the far edge reading zeros
(Downsample2D(padding=0): pad 0 and h_out = (h_in - 2) // 2 + 1, more output rows than the symmetric pad gives).

`install(monkeypatch)` adds them on top of ops_emulator.install (host-logic tests without a GPU); `checker(monkeypatch)`
registers them with tests/launch_check.py, so a LaunchChecker entered afterwards also checks the two new operators
(the pack bit-exact, the latent step with the scheduler criterion) and the far-edge convolutions against float64."""
import torch
import torch.nn.functional as F

from magicdrive_b200 import ops
from tests import launch_check
from tests import ops_emulator as emu

_base_gemm_conv = emu.gemm_conv


def gemm_conv(a0, w, *, n_img, h_in, w_in, c0, lda0, n_out, taps=1, stride=1, pad=0, h_out=None, w_out=None, a1=None,
              c1=0, lda1=0, **kw):
    """ops_emulator.gemm_conv, plus zero rows / columns past the far edge when h_out / w_out exceed the symmetric-pad size."""
    sym_h, sym_w = (h_in + 2 * pad - taps) // stride + 1, (w_in + 2 * pad - taps) // stride + 1
    h_out, w_out = h_out or sym_h, w_out or sym_w
    far_h = max(0, (h_out - 1) * stride + taps - h_in - 2 * pad)  # input rows the last output's taps read past the far pad
    far_w = max(0, (w_out - 1) * stride + taps - w_in - 2 * pad)
    if far_h == 0 and far_w == 0:
        return _base_gemm_conv(a0, w, n_img=n_img, h_in=h_in, w_in=w_in, c0=c0, lda0=lda0, n_out=n_out, taps=taps,
                               stride=stride, pad=pad, h_out=h_out, w_out=w_out, a1=a1, c1=c1, lda1=lda1, **kw)

    def extend(t, c):
        x = t[:, :c].unflatten(0, (n_img, h_in, w_in))
        return F.pad(x, (0, 0, 0, far_w, 0, far_h)).reshape(-1, c)

    return _base_gemm_conv(extend(a0, c0), w, n_img=n_img, h_in=h_in + far_h, w_in=w_in + far_w, c0=c0, lda0=c0,
                           n_out=n_out, taps=taps, stride=stride, pad=pad, h_out=h_out, w_out=w_out,
                           a1=None if a1 is None else extend(a1, c1), c1=c1, lda1=c1, **kw)


def pack_image_patches(x):
    n, cin, h, w = x.shape
    cols = F.unfold(emu._f(x), 3, padding=1).reshape(n, cin, 9, h * w)  # [n, channel, tap, pixel]
    cols = cols.permute(0, 3, 2, 1).reshape(n * h * w, 9 * cin)          # column (tap, channel)
    return emu._act(F.pad(cols, (0, 64 - 9 * cin)))


def latent_dist(moments, n, h, w, c=4, noise=None, scale=1.0):
    m = emu._f(moments).reshape(n, h, w, -1).permute(0, 3, 1, 2)
    v = m[:, :c]
    if noise is not None:
        v = v + torch.exp(0.5 * m[:, c:2 * c].clamp(-30.0, 20.0)) * emu._f(noise)
    return (scale * v).contiguous()


NEW_OPS = {"pack_image_patches": launch_check.EXACT, "latent_dist": launch_check.SCHED}


def install(monkeypatch):
    """ops_emulator.install plus the encoder's operators (magicdrive_b200.ops swapped for torch restatements)."""
    emu.install(monkeypatch)
    for name, fn in (("gemm_conv", gemm_conv), ("pack_image_patches", pack_image_patches), ("latent_dist", latent_dist)):
        monkeypatch.setattr(ops, name, fn)


def checker(monkeypatch):
    """Make LaunchChecker blocks entered afterwards reference the far-edge gemm_conv and check the two new operators."""
    monkeypatch.setattr(emu, "gemm_conv", gemm_conv)
    for name, crit in NEW_OPS.items():
        monkeypatch.setattr(emu, name, globals()[name], raising=False)
        monkeypatch.setitem(launch_check._FIXED, name, crit)
    monkeypatch.setattr(launch_check, "CHECKED", launch_check.CHECKED + list(NEW_OPS))
