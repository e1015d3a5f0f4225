"""CUDA execution of the two hot-path networks over the C-ABI operators (magicdrive_b200.ops).

Dataflow differs from the reference on purpose (B200-first), results do not:
  * activations are bf16 NHWC == [tokens, C]: the NCHW<->token permutes of Transformer2DModel
    (transformer_2d.py:286,305) and the 1x1-conv / Linear distinction vanish;
  * skip-connection concats (unet_2d_blocks.py:1984,2086) are never materialised: GroupNorm and the convolutions
    read two sources;
  * self / cross-view attention use one fused QKV GEMM; cross-view attention reads the neighbours' K/V in place
    (kv_index) instead of duplicating every view's tokens twice (blocks.py:113-121) and `connector(to_out(.))`
    is folded into one GEMM: Wc(Wo(o_l + o_r) + 2 b_o) + b_c  (blocks.py:203-222);
  * everything that does not depend on the latents is hoisted out of the step: text-context K/V projections,
    camera / box tokens, the BEV-map encoder (computed once per scene, not per view per step), and all 22+10
    `time_emb_proj` linears run as one skinny GEMM.
"""
from dataclasses import dataclass
from typing import Dict, List, Optional

import torch

from . import arch, ops
from .params import pack_conv_weight, pack_geglu

BF16, F32 = torch.bfloat16, torch.float32


@dataclass
class FMap:
    """A feature map: data is [n*h*w, c] bf16 (NHWC)."""
    data: torch.Tensor
    n: int
    h: int
    w: int
    c: int


def _bf(t):
    return t.detach().to(dtype=BF16).contiguous()


def _f32(t):
    return t.detach().to(dtype=F32).contiguous()


class _Weights:
    """Packs a reference state dict into kernel-ready device tensors (bf16 K-major matrices, fp32 biases)."""

    fold_dtype = BF16  # storage of weights that are PRODUCTS of checkpoint tensors (W * gamma); the CPU host-logic tests
    #                    set fp32 so that the fold's algebra is checked to 1e-5, apart from its bf16 rounding

    def __init__(self, sd: Dict[str, torch.Tensor], device):
        self.sd = sd
        self.device = device
        self.t: Dict[str, torch.Tensor] = {}

    def raw(self, key):
        return self.sd[key].detach().to(self.device)

    def conv(self, p):
        if p + ".w" not in self.t:
            self.t[p + ".w"] = pack_conv_weight(self.raw(p + ".weight").float())
            self.t[p + ".b"] = _f32(self.raw(p + ".bias"))
        return self.t[p + ".w"], self.t[p + ".b"]

    def conv_direct(self, p):
        if p + ".wd" not in self.t:
            self.t[p + ".wd"] = _f32(self.raw(p + ".weight").float().permute(2, 3, 1, 0))  # [kh, kw, cin, cout]
            self.t[p + ".b"] = _f32(self.raw(p + ".bias"))
        return self.t[p + ".wd"], self.t[p + ".b"]

    def conv_k_padded(self, p, cpad):
        """3x3 filter with the input channels zero-padded to `cpad` (conv_in: 4 -> 64 so K is a whole 64-block)."""
        if p + ".wk" not in self.t:
            w = self.raw(p + ".weight").float()
            wp = torch.zeros((w.shape[0], cpad, w.shape[2], w.shape[3]), dtype=F32, device=w.device)
            wp[:, : w.shape[1]] = w
            self.t[p + ".wk"] = pack_conv_weight(wp)
            self.t[p + ".b"] = _f32(self.raw(p + ".bias"))
        return self.t[p + ".wk"], self.t[p + ".b"]

    def conv_n_padded(self, p, npad):
        """3x3 filter with the output channels zero-padded to `npad` (conv_out: 4 -> 8, the kernel's N granularity)."""
        if p + ".wn" not in self.t:
            w = self.raw(p + ".weight").float()
            wp = torch.zeros((npad, *w.shape[1:]), dtype=F32, device=w.device)
            wp[: w.shape[0]] = w
            bp = torch.zeros((npad,), dtype=F32, device=w.device)
            bp[: w.shape[0]] = self.raw(p + ".bias").float()
            self.t[p + ".wn"] = pack_conv_weight(wp)
            self.t[p + ".bn"] = bp
        return self.t[p + ".wn"], self.t[p + ".bn"]

    def lin(self, p, bias=True):
        if p + ".w" not in self.t:
            self.t[p + ".w"] = _bf(self.raw(p + ".weight"))
            self.t[p + ".b"] = _f32(self.raw(p + ".bias")) if bias else None
        return self.t[p + ".w"], self.t[p + ".b"]

    def norm(self, p):
        if p + ".g" not in self.t:
            self.t[p + ".g"] = _f32(self.raw(p + ".weight"))
            self.t[p + ".beta"] = _f32(self.raw(p + ".bias"))
        return self.t[p + ".g"], self.t[p + ".beta"]

    def cat_lin(self, name, prefixes, suffix=".weight"):
        if name not in self.t:
            self.t[name] = _bf(torch.cat([self.raw(p + suffix) for p in prefixes], 0))
        return self.t[name]

    def geglu(self, p):
        if p + ".gw" not in self.t:
            w, b = pack_geglu(self.raw(p + ".weight").float(), self.raw(p + ".bias").float())
            self.t[p + ".gw"], self.t[p + ".gb"] = w, b
        return self.t[p + ".gw"], self.t[p + ".gb"]

    def ln_lin(self, name, norm, prefixes, geglu=False):
        """LayerNorm `norm` folded into the linear(s) `prefixes` that consume it (mdb_gemm_desc.ln_*):
        W' = W * gamma (bf16), c = W beta + b (fp32), colsum_n = sum_k W'[n, k] (of the rounded W', fp32).
        Returns (W', c, colsum); with geglu the three are re-ordered to the kernel's [128 value | 128 gate] tiles."""
        if name + ".w" not in self.t:
            w = torch.cat([self.raw(p + ".weight").float() for p in prefixes], 0)
            b = torch.cat([self.raw(p + ".bias").float() if (p + ".bias") in self.sd
                           else torch.zeros(self.sd[p + ".weight"].shape[0], device=w.device) for p in prefixes], 0)
            g, beta = self.raw(norm + ".weight").float(), self.raw(norm + ".bias").float()
            wg = (w * g[None, :]).to(self.fold_dtype)
            c = w @ beta + b
            cs = wg.float().sum(1)
            if geglu:
                wg2, c = pack_geglu(wg.float(), c, dtype=self.fold_dtype)
                _, cs = pack_geglu(wg.float(), cs)
                wg = wg2
            self.t[name + ".w"], self.t[name + ".c"], self.t[name + ".cs"] = wg.contiguous(), _f32(c), _f32(cs)
        return self.t[name + ".w"], self.t[name + ".c"], self.t[name + ".cs"]

    def folded_connector(self, blk, bias_count: int = 2):
        """W' = Wc @ Wo, b' = bias_count * Wc b_o + b_c  (fp32 fold, bf16 storage).  bias_count = attention outputs summed
        before the connector: 2 in 'add' mode (one per neighbour, blocks.py:213-218), 1 in 'concat' / 'self' mode."""
        k = blk + f".attn4.fold{bias_count}"
        if k + ".w" not in self.t:
            wo = self.raw(blk + ".attn4.to_out.0.weight").float()
            bo = self.raw(blk + ".attn4.to_out.0.bias").float()
            wc = self.raw(blk + ".connector.weight").float()
            bc = self.raw(blk + ".connector.bias").float()
            self.t[k + ".w"] = _bf(wc @ wo)
            self.t[k + ".b"] = _f32(float(bias_count) * (wc @ bo) + bc)
        return self.t[k + ".w"], self.t[k + ".b"]


class _Net:
    """Shared machinery of the UNet and the ControlNet encoder."""

    def __init__(self, cfg, sd, device, multiview: bool):
        self.cfg = cfg
        self.W = _Weights(sd, device)
        self.device = device
        self.multiview = multiview
        self.down = arch.down_blocks(cfg, multiview)
        self.mid = arch.mid_block(cfg, multiview)
        self.resnets: List[arch.ResnetSpec] = [rs for b in self.down for rs, _ in b.layers] + [self.mid[0], self.mid[2]]
        self.transformers: List[arch.TransformerSpec] = [tr for b in self.down for _, tr in b.layers if tr] + [self.mid[1]]
        self._kv_idx = {}
        self._kv_sym = {}
        self.view_shard = None  # dist.ShardContext when the cameras of a scene are split across ranks

    # ---------------------------------------------------------------- time embedding
    def _finalize_specs(self):
        self.temb_off, off = {}, 0
        for rs in self.resnets:
            self.temb_off[rs.prefix] = off
            off += rs.cout
        self.temb_total = off

    def time_embed(self, t_f32: torch.Tensor) -> torch.Tensor:
        """t [V] fp32 -> all resnets' time_emb_proj(silu(emb)) as one fp32 [V, sum(cout)] matrix
        (embeddings.py:24-64,186-201; resnet.py:612-616)."""
        cfg = self.cfg
        te = ops.timestep_embedding(t_f32, cfg.block_out_channels[0], cfg.flip_sin_to_cos, float(cfg.freq_shift))
        w1, b1 = self.W.lin("time_embedding.linear_1")
        w2, b2 = self.W.lin("time_embedding.linear_2")
        e = ops.linear_small(te, w1, b1, post_silu=True)
        e = ops.linear_small(e, w2, b2)
        wcat = self.W.cat_lin("temb.wcat", [rs.prefix + ".time_emb_proj" for rs in self.resnets])
        if "temb.bcat" not in self.W.t:
            self.W.t["temb.bcat"] = _f32(torch.cat([self.W.raw(rs.prefix + ".time_emb_proj.bias") for rs in self.resnets]))
        return ops.linear_small(e, wcat, self.W.t["temb.bcat"], pre_silu=True)

    # ---------------------------------------------------------------- blocks
    def resnet(self, rs: arch.ResnetSpec, x: FMap, temb_all: torch.Tensor, skip: Optional[FMap] = None) -> FMap:
        """ResnetBlock2D.forward (resnet.py:590-640); `skip` is the second half of the channel concat."""
        W, cfg = self.W, self.cfg
        c0 = x.c
        c1 = skip.c if skip is not None else 0
        assert c0 + c1 == rs.cin, (rs.prefix, c0, c1, rs.cin)
        hw = x.h * x.w
        x1 = skip.data if skip is not None else None
        g1, be1 = W.norm(rs.prefix + ".norm1")
        h = ops.groupnorm(x.data, c0, c0, x.n, hw, g1, be1, cfg.norm_eps, True, x1=x1, c1=c1, ld1=c1,
                          groups=cfg.norm_num_groups)
        w1, b1 = W.conv(rs.prefix + ".conv1")
        off = self.temb_off[rs.prefix]
        h = ops.gemm_conv(h, w1, n_img=x.n, h_in=x.h, w_in=x.w, c0=rs.cin, lda0=rs.cin, n_out=rs.cout, taps=3, pad=1,
                          bias=b1, rowbias=temb_all[:, off:off + rs.cout])
        g2, be2 = W.norm(rs.prefix + ".norm2")
        h = ops.groupnorm(h, rs.cout, rs.cout, x.n, hw, g2, be2, cfg.norm_eps, True, groups=cfg.norm_num_groups)
        if rs.shortcut:
            ws, bs = W.conv(rs.prefix + ".conv_shortcut")
            res = ops.gemm_conv(x.data, ws, n_img=x.n, h_in=x.h, w_in=x.w, c0=c0, lda0=c0, a1=x1, c1=c1, lda1=c1,
                                n_out=rs.cout, bias=bs)
        else:
            assert skip is None
            res = x.data
        w2, b2 = W.conv(rs.prefix + ".conv2")
        out = ops.gemm_conv(h, w2, n_img=x.n, h_in=x.h, w_in=x.w, c0=rs.cout, lda0=rs.cout, n_out=rs.cout, taps=3,
                            pad=1, bias=b2, residual=res, ldr=rs.cout)
        return FMap(out, x.n, x.h, x.w, rs.cout)

    def kv_index(self, n_views: int) -> torch.Tensor:
        """[V, 2] int32: the two ring neighbours of each view inside its own scene (Nuscenes.yaml:27-33).  With the views
        split across GPUs (dist.ShardContext) an entry is (source << 24) | batch, source 0 = this GPU's K/V buffer,
        1 / 2 = the ring-neighbour GPUs' buffers (mdb_attention_multi)."""
        if n_views not in self._kv_idx:
            nb = self.cfg.neighboring_view_pair
            n_cam = len(nb)
            if self._sharded():
                pl = self.view_shard.plan
                assert n_views % pl.n_local == 0
                _, idx = pl.kv_sources(n_views // pl.n_local)
                idx = [[idx[2 * i], idx[2 * i + 1]] for i in range(n_views)]
            else:
                assert n_views % n_cam == 0
                idx = [[s * n_cam + nb[i][0], s * n_cam + nb[i][1]] for s in range(n_views // n_cam) for i in range(n_cam)]
            self._kv_idx[n_views] = torch.tensor(idx, dtype=torch.int32, device=self.device)
        return self._kv_idx[n_views]

    def _sharded(self) -> bool:
        return self.view_shard is not None and self.view_shard.plan.groups > 1

    def set_view_shard(self, shard) -> None:
        """Split the cameras across ranks (dist.ShardContext) or back to all views on this GPU (None)."""
        self.view_shard = shard
        self._kv_idx = {}
        self._kv_sym = {}

    def _neighbour_kv(self, key, V: int, L: int, C: int):
        """This block's K/V buffer in symmetric memory and the ring-neighbour GPUs' copies of it, as attention sources."""
        hit = self._kv_sym.get((key, V, L, C))
        if hit is None:
            sh = self.view_shard
            pl, grp = sh.plan, sh.half_group
            n_samples = V // pl.n_local
            mx = max(pl.local_views_of(g) for g in range(pl.groups))
            buf, hdl = grp.alloc((n_samples * mx * L, 2 * C), BF16)  # same shape on every rank (uneven view counts padded)
            srcs, _ = pl.kv_sources(n_samples)
            views = []
            for g in srcs:
                vg = n_samples * pl.local_views_of(g)
                t = buf if g == pl.vg else grp.peer_view(hdl, g, (n_samples * mx * L, 2 * C), BF16)
                views.append((t[: vg * L], vg))
            hit = (buf[: V * L], hdl, views)
            self._kv_sym[(key, V, L, C)] = hit
        return hit[0], hit[2]

    def context_kv(self, ctx_bf16: torch.Tensor) -> Dict[str, torch.Tensor]:
        """attn2 K/V projections of the conditioning tokens for every transformer (step-invariant).
        ctx: [V*Lc, 768] bf16 -> {prefix: [V*Lc, 2C] bf16}."""
        out = {}
        for tr in self.transformers:
            blk = tr.prefix + ".transformer_blocks.0"
            wkv = self.W.cat_lin(blk + ".attn2.wkv", [blk + ".attn2.to_k", blk + ".attn2.to_v"])
            out[tr.prefix] = ops.linear(ctx_bf16, wkv)
        return out

    def transformer(self, tr: arch.TransformerSpec, x: FMap, ctx_kv: Dict[str, torch.Tensor], lc: int) -> FMap:
        """Transformer2DModel.forward (transformer_2d.py:276-315) around BasicTransformerBlock (attention.py:123-182)
        or BasicMultiviewTransformerBlock (magicdrive/networks/blocks.py:144-238)."""
        W, cfg = self.W, self.cfg
        C, heads = tr.c, tr.heads
        d = C // heads
        V, L = x.n, x.h * x.w
        M = V * L
        scale = d ** -0.5
        p = tr.prefix
        blk = p + ".transformer_blocks.0"
        g, b = W.norm(p + ".norm")
        h = ops.groupnorm(x.data, C, C, V, L, g, b, 1e-6, False, groups=cfg.norm_num_groups)
        wi, bi = W.conv(p + ".proj_in")
        # The block's LayerNorms never run as kernels: every GEMM that writes the residual stream X also emits per-row
        # (sum, sum of squares) of the bf16 values it stores, and the GEMM that consumes LayerNorm(X) reads the raw X
        # with gamma folded into its weights and normalises in its epilogue (mdb_gemm_desc.ln_stats / stats_out).
        X, sx = ops.linear(h, wi, bias=bi, emit_stats=True)
        # --- self attention
        wqkv, cq, sq = W.ln_lin(blk + ".attn1.lnqkv", blk + ".norm1", [blk + ".attn1.to_q", blk + ".attn1.to_k", blk + ".attn1.to_v"])
        qkv = ops.linear(X, wqkv, bias=cq, ln=sx, ln_colsum=sq)
        o = ops.attention(qkv, qkv[:, C:], qkv[:, 2 * C:], b=V, heads=heads, lq=L, lk=L, d=d, ldq=3 * C, ldk=3 * C,
                          ldv=3 * C, scale=scale)
        wo, bo = W.lin(blk + ".attn1.to_out.0")
        X, sx = ops.linear(o, wo, bias=bo, residual=X, emit_stats=True)
        # --- conditioning cross attention (camera + text + box tokens)
        wq, cq, sq = W.ln_lin(blk + ".attn2.lnq", blk + ".norm2", [blk + ".attn2.to_q"])
        q = ops.linear(X, wq, bias=cq, ln=sx, ln_colsum=sq)
        kv = ctx_kv[p]
        o = ops.attention(q, kv, kv[:, C:], b=V, heads=heads, lq=L, lk=lc, d=d, ldq=C, ldk=2 * C, ldv=2 * C, scale=scale)
        wo, bo = W.lin(blk + ".attn2.to_out.0")
        X, sx = ops.linear(o, wo, bias=bo, residual=X, emit_stats=True)
        # --- cross-view attention
        if tr.multiview:
            at = cfg.neighboring_attn_type
            if at not in ("add", "concat", "self") or cfg.zero_module_type != "zero_linear":
                raise NotImplementedError("neighboring_attn_type must be 'add' / 'concat' / 'self' and the connector zero_linear "
                                          "(blocks.py:74-89; the shipped configs/model/SDv1.5mv_rawbox.yaml:19-20 uses add + zero_linear)")
            if self._sharded() and at != "add":
                raise NotImplementedError("views split across GPUs: only neighboring_attn_type='add' is implemented")
            if at == "self":
                # blocks.py:134-138, 209-211: one attention over the tokens of ALL views of a scene.  The token matrix is
                # scene-major then view-major, so this is the self-attention kernel with batch = scenes and n_cam * L tokens.
                n_cam = len(cfg.neighboring_view_pair)
                wqkv, cq, sq = W.ln_lin(blk + ".attn4.lnqkv", blk + ".norm4",
                                        [blk + ".attn4.to_q", blk + ".attn4.to_k", blk + ".attn4.to_v"])
                qkv = ops.linear(X, wqkv, bias=cq, ln=sx, ln_colsum=sq)
                o = ops.attention(qkv, qkv[:, C:], qkv[:, 2 * C:], b=V // n_cam, heads=heads, lq=n_cam * L, lk=n_cam * L, d=d,
                                  ldq=3 * C, ldk=3 * C, ldv=3 * C, scale=scale)
            elif at == "concat":
                # blocks.py:122-133: ONE softmax over the keys of both neighbours.  Their K/V rows are gathered into one
                # [V, n_nb * L, 2C] buffer (a device copy; this non-default mode is not on the benchmarked path)
                wq, cq, sq = W.ln_lin(blk + ".attn4.lnq", blk + ".norm4", [blk + ".attn4.to_q"])
                wkv, ckv, skv = W.ln_lin(blk + ".attn4.lnkv", blk + ".norm4", [blk + ".attn4.to_k", blk + ".attn4.to_v"])
                q = ops.linear(X, wq, bias=cq, ln=sx, ln_colsum=sq)
                kv = ops.linear(X, wkv, bias=ckv, ln=sx, ln_colsum=skv)
                idx = self.kv_index(V)
                n_nb = idx.shape[1]
                kvc = kv.view(V, L, 2 * C)[idx.long()].reshape(V * n_nb * L, 2 * C)
                o = ops.attention(q, kvc, kvc[:, C:], b=V, heads=heads, lq=L, lk=n_nb * L, d=d, ldq=C, ldk=2 * C, ldv=2 * C,
                                  scale=scale)
            elif not self._sharded():
                wqkv, cq, sq = W.ln_lin(blk + ".attn4.lnqkv", blk + ".norm4",
                                        [blk + ".attn4.to_q", blk + ".attn4.to_k", blk + ".attn4.to_v"])
                qkv = ops.linear(X, wqkv, bias=cq, ln=sx, ln_colsum=sq)
                o = ops.attention(qkv, qkv[:, C:], qkv[:, 2 * C:], b=V, heads=heads, lq=L, lk=L, d=d, ldq=3 * C,
                                  ldk=3 * C, ldv=3 * C, scale=scale, kv_index=self.kv_index(V), n_sets=2)
            else:
                # cameras split across GPUs: K/V of the local views go to a symmetric buffer; after one device-side
                # barrier the attention kernel reads the two ring neighbours' K/V tiles IN PLACE from the neighbour
                # GPUs over NVLink (TMA on peer-mapped addresses) while it works on the local tiles: no gather, no copy
                wq, cq, sq = W.ln_lin(blk + ".attn4.lnq", blk + ".norm4", [blk + ".attn4.to_q"])
                wkv, ckv, skv = W.ln_lin(blk + ".attn4.lnkv", blk + ".norm4", [blk + ".attn4.to_k", blk + ".attn4.to_v"])
                q = ops.linear(X, wq, bias=cq, ln=sx, ln_colsum=sq)
                kv, srcs = self._neighbour_kv(blk, V, L, C)
                ops.linear(X, wkv, bias=ckv, ln=sx, ln_colsum=skv, out=kv, ldo=2 * C)
                self.view_shard.half_group.barrier(0)
                o = ops.attention_multi(q, [(t, t[:, C:], 2 * C, vg) for t, vg in srcs], b=V, heads=heads, lq=L, lk=L, d=d,
                                        ldq=C, scale=scale, kv_index=self.kv_index(V), n_sets=2)
            wf, bf_ = W.folded_connector(blk, bias_count=2 if at == "add" else 1)
            X, sx = ops.linear(o, wf, bias=bf_, residual=X, emit_stats=True)
        # --- GEGLU feed-forward
        wg, cg, sg = W.ln_lin(blk + ".ff.lnproj", blk + ".norm3", [blk + ".ff.net.0.proj"], geglu=True)
        hg = ops.linear(X, wg, bias=cg, geglu=True, ln=sx, ln_colsum=sg)
        w2, b2 = W.lin(blk + ".ff.net.2")
        X = ops.linear(hg, w2, bias=b2, residual=X)
        wp, bp = W.conv(p + ".proj_out")
        out = ops.linear(X, wp, bias=bp, residual=x.data)
        return FMap(out, V, x.h, x.w, C)

    def downsample(self, sp: arch.SamplerSpec, x: FMap) -> FMap:
        w, b = self.W.conv(sp.prefix)
        ho, wo = (x.h + 2 - 3) // 2 + 1, (x.w + 2 - 3) // 2 + 1
        out = ops.gemm_conv(x.data, w, n_img=x.n, h_in=x.h, w_in=x.w, c0=x.c, lda0=x.c, n_out=sp.c, taps=3, stride=2,
                            pad=1, bias=b)
        return FMap(out, x.n, ho, wo, sp.c)

    def encoder(self, x: FMap, temb_all, ctx_kv, lc, on_skip=None):
        """conv_in output -> (mid-block output, skip list).  `on_skip(i)` is called right after the kernels producing skip i
        (and, with i = len(skips), the mid output) were enqueued: the pipeline records a CUDA event there."""
        skips = [x]

        def mark():
            if on_skip is not None:
                on_skip(len(skips) - 1)

        mark()
        for blk in self.down:
            for rs, tr in blk.layers:
                x = self.resnet(rs, x, temb_all)
                if tr is not None:
                    x = self.transformer(tr, x, ctx_kv, lc)
                skips.append(x)
                mark()
            if blk.sampler is not None:
                x = self.downsample(blk.sampler, x)
                skips.append(x)
                mark()
        r0, tr, r1 = self.mid
        x = self.resnet(r0, x, temb_all)
        x = self.transformer(tr, x, ctx_kv, lc)
        x = self.resnet(r1, x, temb_all)
        if on_skip is not None:
            on_skip(len(skips))
        return x, skips

    CIN_PAD = 64  # latent channels are zero-padded to one 64-wide K block so conv_in runs on the tensor-core path

    def conv_in(self, x_pad: torch.Tensor, n, h, w, residual=None) -> FMap:
        """x_pad: [n*h*w, 64] bf16 (ops.pack_latents); optional residual [n*h*w, C0] (the BEV-map embedding)."""
        wk, b = self.W.conv_k_padded("conv_in", self.CIN_PAD)
        c0 = self.cfg.block_out_channels[0]
        out = ops.gemm_conv(x_pad, wk, n_img=n, h_in=h, w_in=w, c0=self.CIN_PAD, lda0=self.CIN_PAD, n_out=c0, taps=3,
                            pad=1, bias=b, residual=residual, ldr=c0)
        return FMap(out, n, h, w, c0)


class UNetEngine(_Net):
    """UNet2DConditionModelMultiview.forward on the GPU (unet_2d_condition_multiview.py:327-527)."""

    def __init__(self, cfg: arch.UNetConfig, sd, device):
        super().__init__(cfg, sd, device, multiview=cfg.multiview)
        self.up = arch.up_blocks(cfg)
        self.resnets += [rs for b in self.up for rs, _ in b.layers]
        self.transformers += [tr for b in self.up for _, tr in b.layers if tr]
        self._finalize_specs()

    COUT_PAD = 8

    def forward(self, latents_pad: torch.Tensor, n, h, w, t_f32, ctx_kv, lc, down_res: Optional[List[torch.Tensor]] = None,
                mid_res: Optional[torch.Tensor] = None, temb_all: Optional[torch.Tensor] = None) -> torch.Tensor:
        """latents [n*h*w, 64] bf16 (channel-padded) -> predicted noise fp32 [n*h*w, 8] (first out_channels valid).
        `temb_all` may carry precomputed time-embedding projections ([1 or n, sum(cout)] fp32)."""
        if temb_all is None:
            temb_all = self.time_embed(t_f32)
        x, skips = self.forward_encoder(latents_pad, n, h, w, temb_all, ctx_kv, lc)
        return self.forward_decoder(x, skips, temb_all, ctx_kv, lc, down_res, mid_res)

    def forward_encoder(self, latents_pad, n, h, w, temb_all, ctx_kv, lc, on_skip=None):
        """conv_in + down blocks + mid block: independent of the ControlNet residuals, so the pipeline runs it
        concurrently with the ControlNet on a second stream."""
        x = self.conv_in(latents_pad, n, h, w)
        return self.encoder(x, temb_all, ctx_kv, lc, on_skip=on_skip)

    def forward_decoder(self, x, skips, temb_all, ctx_kv, lc, down_res=None, mid_res=None) -> torch.Tensor:
        """Up blocks + conv_out.  `skips` / `x` either are the encoder's own tensors with the ControlNet residuals passed in
        `down_res` / `mid_res` (added here), or already carry them (ControlNetEngine.residuals(add_to=...)) with both None."""
        cfg = self.cfg
        skips = list(skips)
        if down_res is not None:
            skips = [FMap(ops.add(s.data, r), s.n, s.h, s.w, s.c) for s, r in zip(skips, down_res)]
        if mid_res is not None:
            x = FMap(ops.add(x.data, mid_res), x.n, x.h, x.w, x.c)
        for blk in self.up:
            for rs, tr in blk.layers:
                x = self.resnet(rs, x, temb_all, skip=skips.pop())
                if tr is not None:
                    x = self.transformer(tr, x, ctx_kv, lc)
            if blk.sampler is not None:
                tgt = skips[-1]
                up = ops.upsample_nearest(x.data, x.n, x.h, x.w, x.c, tgt.h, tgt.w)
                wu, bu = self.W.conv(blk.sampler.prefix)
                out = ops.gemm_conv(up, wu, n_img=x.n, h_in=tgt.h, w_in=tgt.w, c0=x.c, lda0=x.c, n_out=x.c, taps=3, pad=1,
                                    bias=bu)
                x = FMap(out, x.n, tgt.h, tgt.w, x.c)
        g, b = self.W.norm("conv_norm_out")
        hn = ops.groupnorm(x.data, x.c, x.c, x.n, x.h * x.w, g, b, cfg.norm_eps, True, groups=cfg.norm_num_groups)
        wn, bo = self.W.conv_n_padded("conv_out", self.COUT_PAD)
        return ops.gemm_conv(hn, wn, n_img=x.n, h_in=x.h, w_in=x.w, c0=x.c, lda0=x.c, n_out=self.COUT_PAD, taps=3, pad=1,
                             bias=bo, out_f32=True)


class ControlNetEngine(_Net):
    """BEVControlNetModel.forward on the GPU (magicdrive/networks/unet_addon_rawbox.py:707-932)."""

    def __init__(self, cfg: arch.ControlNetConfig, sd, device):
        super().__init__(cfg, sd, device, multiview=False)
        self._finalize_specs()
        self.res_channels = arch.controlnet_residual_channels(cfg)

    # ---------------------------------------------------------------- step-invariant conditioning
    def camera_tokens(self, camera_param: torch.Tensor) -> torch.Tensor:
        """(b, n, 3, 7) -> (b*n, 768) fp32: _embed_camera + cam2token (unet_addon_rawbox.py:288-305, 329)."""
        b, n, c3, e = camera_param.shape
        x = camera_param.to(self.device, F32).permute(0, 1, 3, 2).reshape(b * n * e, c3).contiguous()
        emb = ops.fourier_embed(x, self.cfg.cam_num_freqs).view(b * n, -1)
        w, bias = self.W.lin("cam2token")
        return ops.linear_small(emb, w, bias)

    def uncond_cam_param(self, batch, n_cam):
        w = self.W.raw("uncond_cam.weight")[0].float()
        return w.reshape(1, 1, -1, self.cfg.uncond_cam_in_dim[1]).expand(batch, n_cam, -1, -1)

    def box_tokens(self, bboxes, classes, masks) -> torch.Tensor:
        """(B, N, 8, 3), (B, N), (B, N) -> (B*N, 768) fp32 (bbox_embedder.py:154-189)."""
        W, cfg = self.W, self.cfg
        p = "bbox_embedder"
        B, N = classes.shape
        bb = bboxes.to(self.device, F32).reshape(B * N * cfg.bbox_points, 3).contiguous()
        m = masks.to(self.device).reshape(B * N, 1).to(F32)
        pos = ops.fourier_embed(bb, cfg.bbox_num_freqs).view(B * N, -1)
        # masked select between the embedding and the learned null features: O(B*N*1000) elementwise glue on the
        # step-invariant path (once per call), kept in torch
        pos = pos * m + W.raw(p + ".null_pos_feature").float()[None] * (1 - m)
        cls = W.raw(p + "._class_tokens").float()[classes.to(self.device).reshape(-1)]
        cls = cls * m + W.raw(p + ".null_class_feature").float()[None] * (1 - m)
        w, b = W.lin(p + ".bbox_proj")
        emb = ops.linear_small(pos.contiguous(), w, b, post_silu=True)
        emb = torch.cat([emb, cls], -1).contiguous()
        w, b = W.lin(p + ".second_linear.0")
        emb = ops.linear_small(emb, w, b, post_silu=True)
        w, b = W.lin(p + ".second_linear.2")
        emb = ops.linear_small(emb, w, b, post_silu=True)
        w, b = W.lin(p + ".second_linear.4")
        return ops.linear_small(emb, w, b)

    def context(self, camera_param, bboxes_3d_data, encoder_hidden_states) -> torch.Tensor:
        """encoder_hidden_states_with_cam: (b*n_cam, 1 + len + n_box, 768) fp32 (unet_addon_rawbox.py:743-793)."""
        b, n_cam = camera_param.shape[:2]
        cam = self.camera_tokens(camera_param).view(b, n_cam, 1, -1)
        text = encoder_hidden_states.to(self.device, F32)
        parts = [cam, text.unsqueeze(1).expand(-1, n_cam, -1, -1)]
        if bboxes_3d_data is not None:
            bx = bboxes_3d_data["bboxes"]
            b_box, n_box = bx.shape[:2]
            emb = self.box_tokens(bx.reshape(b_box * n_box, *bx.shape[2:]),
                                  bboxes_3d_data["classes"].reshape(b_box * n_box, -1),
                                  bboxes_3d_data["masks"].reshape(b_box * n_box, -1))
            emb = emb.view(b_box, n_box, -1, emb.shape[-1])
            if n_box != n_cam:
                emb = emb.expand(-1, n_cam, -1, -1)
            parts.append(emb)
        ctx = torch.cat(parts, dim=2)
        return ctx.reshape(b * n_cam, ctx.shape[2], ctx.shape[3]).contiguous()

    def map_embedding(self, cond: torch.Tensor) -> torch.Tensor:
        """BEV map (b, 8, H, W) -> [b, h, w, 320] bf16 NHWC, once per scene (map_embedder.py:66-76)."""
        x = cond.to(self.device, F32).permute(0, 2, 3, 1).contiguous()
        n, h, w = x.shape[0], x.shape[1], x.shape[2]
        layers = arch.map_encoder_layers(self.cfg)
        for i, (name, ci, co, stride, pad) in enumerate(layers):
            wd, bias = self.W.conv_direct(name)
            last = i == len(layers) - 1
            if last and self.cfg.map_embedding_size is not None:
                # BEVControlNetConditioningEmbeddingPlus: AdaptiveAvgPool2d + SiLU ahead of conv_out (map_embedder.py:118, 70-72)
                ho, wo = self.cfg.map_embedding_size
                x = ops.adaptive_avgpool(x, n, h, w, ci, ho, wo, silu=True)
                h, w = ho, wo
            x = ops.conv_direct(x, wd, bias, n=n, h=h, w=w, cin=ci, cout=co, k=3, stride=stride, pad=pad, silu=not last,
                                out_f32=not last)
            h, w = x.shape[1], x.shape[2]
        return x  # bf16 [b, h, w, 320]

    # ---------------------------------------------------------------- per-step
    def forward(self, latents_pad, n, h, w, t_f32, ctx_kv, lc, map_emb_per_view: torch.Tensor,
                conditioning_scale=1.0, temb_all: Optional[torch.Tensor] = None):
        """latents [n*h*w, 64] bf16 channel-padded (n = scenes*views); t_f32 [n]; map_emb_per_view [n, h, w, 320] bf16.
        Returns (12 + 1 residual maps as [pixels, C] bf16 tensors)."""
        x, skips = self.trunk(latents_pad, n, h, w, t_f32, ctx_kv, lc, map_emb_per_view, temb_all)
        down, mid = self.residuals(skips, x, conditioning_scale)
        return down, mid, skips, x

    def trunk(self, latents_pad, n, h, w, t_f32, ctx_kv, lc, map_emb_per_view, temb_all=None):
        """conv_in (+ BEV-map embedding) + down blocks + mid block of the ControlNet (unet_addon_rawbox.py:836-894)."""
        if temb_all is None:
            temb_all = self.time_embed(t_f32)
        x = self.conv_in(latents_pad, n, h, w, residual=map_emb_per_view)
        return self.encoder(x, temb_all, ctx_kv, lc)

    def residuals(self, skips, x, conditioning_scale=1.0, add_to=None, add_to_mid=None, before=None):
        """The 12 + 1 zero convolutions (unet_addon_rawbox.py:898-915).  With `add_to` / `add_to_mid` (the UNet's own skip
        tensors and mid output) every zero convolution takes that tensor as its epilogue residual and returns
        `unet_skip + scale * zero_conv(controlnet_skip)`: the additions of unet_2d_condition_multiview.py:479-497 ride the
        GEMM that produces the residual, which is then never written or re-read.  `before(i)` is called ahead of the
        i-th launch (the pipeline waits there for the event of UNet skip i).  `conditioning_scale`: one factor, or a list of
        len(skips) + 1 factors (guess_mode: torch.logspace(-1, 0, 13) * scale, unet_addon_rawbox.py:897-905)."""
        scales = list(conditioning_scale) if isinstance(conditioning_scale, (list, tuple)) else [conditioning_scale] * (len(skips) + 1)
        assert len(scales) == len(skips) + 1
        down = []
        for i, s in enumerate(skips):
            wz, bz = self.W.conv(f"controlnet_down_blocks.{i}")
            if before is not None:
                before(i)
            down.append(ops.linear(s.data, wz, bias=bz, out_scale=float(scales[i]),
                                   residual=None if add_to is None else add_to[i]))
        wz, bz = self.W.conv("controlnet_mid_block")
        if before is not None:
            before(len(skips))
        mid = ops.linear(x.data, wz, bias=bz, out_scale=float(scales[-1]), residual=add_to_mid)
        return down, mid


class VaeDecoderEngine:
    """AutoencoderKL.decode for the 6 generated views (pipeline_bev_controlnet.py:100-112 -> autoencoder_kl.py:177-196 ->
    vae.py:226-273): the step after the denoising path, built from the same operators (implicit-GEMM 3x3 convolutions,
    single-kernel GroupNorm+SiLU, nearest x2).  The mid block's single-head attention is 512 wide — beyond the fused
    attention kernels' head dims — and runs as three tensor-core GEMMs per image around a row softmax:
    S = Q K^T (fp32, scaled), P = softmax(S) (bf16, key count padded to a K block), V^T = W_v X^T, O = P V + b_v."""

    COUT_PAD = 8

    def __init__(self, cfg: arch.VaeConfig, sd, device):
        self.cfg, self.device = cfg, device
        self.W = _Weights(sd, device)
        self.blocks = arch.vae_decoder_blocks(cfg)

    def _resnet(self, p: str, x: FMap, cout: int) -> FMap:
        """ResnetBlock2D.forward with temb = None (resnet.py:590-640)."""
        W, g = self.W, self.cfg.norm_num_groups
        hw = x.h * x.w
        g1, b1 = W.norm(p + ".norm1")
        h = ops.groupnorm(x.data, x.c, x.c, x.n, hw, g1, b1, 1e-6, True, groups=g)
        w1, c1 = W.conv(p + ".conv1")
        h = ops.gemm_conv(h, w1, n_img=x.n, h_in=x.h, w_in=x.w, c0=x.c, lda0=x.c, n_out=cout, taps=3, pad=1, bias=c1)
        g2, b2 = W.norm(p + ".norm2")
        h = ops.groupnorm(h, cout, cout, x.n, hw, g2, b2, 1e-6, True, groups=g)
        res = x.data
        if x.c != cout:
            ws, bs = W.conv(p + ".conv_shortcut")
            res = ops.gemm_conv(x.data, ws, n_img=x.n, h_in=x.h, w_in=x.w, c0=x.c, lda0=x.c, n_out=cout, bias=bs)
        w2, c2 = W.conv(p + ".conv2")
        out = ops.gemm_conv(h, w2, n_img=x.n, h_in=x.h, w_in=x.w, c0=cout, lda0=cout, n_out=cout, taps=3, pad=1, bias=c2,
                            residual=res, ldr=cout)
        return FMap(out, x.n, x.h, x.w, cout)

    def _attention(self, x: FMap, a: str) -> FMap:
        """Attention(heads=1, dim_head=C, GroupNorm, residual) of UNetMidBlock2D (unet_2d_blocks.py:433-446); `a` is its
        key prefix (decoder.mid_block.attentions.0 or encoder.mid_block.attentions.0)."""
        W, C, L = self.W, x.c, x.h * x.w
        g, b = W.norm(a + ".group_norm")
        t = ops.groupnorm(x.data, C, C, x.n, L, g, b, 1e-6, False, groups=self.cfg.norm_num_groups)
        wq, bq = W.lin(a + ".to_q")
        wk, bk = W.lin(a + ".to_k")
        wv, bv = W.lin(a + ".to_v")
        q = ops.linear(t, wq, bias=bq)
        lp = (L + 63) // 64 * 64  # keys padded to whole K blocks of the P.V product
        # persistent scratch (no per-call allocation or zero-fill: the decode is captured in a CUDA graph): scores and
        # probabilities [L, lp] per image, V^T [C, lp] whose pad columns stay zero from allocation (P is zero there too)
        key = ("vae_attn", a, x.n, L, C)
        if key not in W.t:
            dev = q.device
            # keys live in a buffer with lp - L spare rows so that every image's score GEMM can take lp "keys" (its n_out must
            # be a multiple of 8): the extra columns are another image's keys or the zero tail, and softmax_rows drops them
            W.t[key] = (torch.empty((x.n, L, lp), dtype=F32, device=dev), torch.zeros((x.n, C, lp), dtype=q.dtype, device=dev),
                        torch.empty((x.n * L, C), dtype=q.dtype, device=dev), torch.zeros((x.n * L + lp - L, C), dtype=q.dtype, device=dev),
                        torch.zeros((x.n * L + lp - L, C), dtype=q.dtype, device=dev))
        sbuf, vtbuf, o, kbuf, tbuf = W.t[key]
        ops.linear(t, wk, bias=bk, out=kbuf[: x.n * L], ldo=C)
        if lp != L:  # the V^T GEMM likewise takes lp token rows per image (finite values in the spare columns, P is zero there)
            tbuf[: x.n * L].copy_(t)
            t = tbuf
        for i in range(x.n):
            rows = slice(i * L, (i + 1) * L)
            ops.linear(q[rows], kbuf[i * L: i * L + lp], out_f32=True, out_scale=C ** -0.5, out=sbuf[i], ldo=lp)  # [L, lp]: q . k_j / sqrt(C)
            p = ops.softmax_rows(sbuf[i], L, lp)                                                    # bf16, padded keys get 0
            ops.linear(wv, t[i * L: i * L + lp] if lp != L else t[rows], out=vtbuf[i], ldo=lp)      # [C, lp] = W_v X^T  (V^T, no bias)
            ops.linear(p, vtbuf[i], bias=bv, out=o[rows], ldo=C)                                    # P V + b_v (rows of P sum to 1)
        wo, bo = W.lin(a + ".to_out.0")
        out = ops.linear(o, wo, bias=bo, residual=x.data)
        return FMap(out, x.n, x.h, x.w, C)

    def decode(self, z_nhwc: torch.Tensor, n: int, h: int, w: int, scale: float = 1.0, to_unit_range: bool = False):
        """z_nhwc: fp32 [n*h*w, 4] latents (the denoiser's resident layout); `scale` multiplies them first
        (1 / scaling_factor).  Returns fp32 [n, 8h, 8w, 3] (with to_unit_range: image / 2 + 0.5 clamped to [0, 1])."""
        cfg, W = self.cfg, self.W
        key = ("pq", float(scale))
        if key not in W.t:  # 1x1 post_quant_conv with the latent scale folded into its weights
            W.t[key] = (_f32(W.raw("post_quant_conv.weight").float().permute(2, 3, 1, 0) * scale), _f32(W.raw("post_quant_conv.bias")))
        wq, bq = W.t[key]
        lc = cfg.latent_channels
        x = ops.conv_direct(z_nhwc.reshape(n, h, w, lc), wq, bq, n=n, h=h, w=w, cin=lc, cout=lc, k=1, pad=(0, 0), out_f32=True)
        wd, bd = W.conv_direct("decoder.conv_in")
        c = cfg.block_out_channels[-1]
        x = ops.conv_direct(x, wd, bd, n=n, h=h, w=w, cin=lc, cout=c, k=3)
        x = FMap(x.reshape(n * h * w, c), n, h, w, c)
        x = self._resnet("decoder.mid_block.resnets.0", x, c)
        x = self._attention(x, "decoder.mid_block.attentions.0")
        x = self._resnet("decoder.mid_block.resnets.1", x, c)
        for _, resnets, up in self.blocks:
            for p, _, cout in resnets:
                x = self._resnet(p, x, cout)
            if up:
                u = ops.upsample_nearest(x.data, x.n, x.h, x.w, x.c, 2 * x.h, 2 * x.w)
                wu, bu = W.conv(up)
                out = ops.gemm_conv(u, wu, n_img=x.n, h_in=2 * x.h, w_in=2 * x.w, c0=x.c, lda0=x.c, n_out=x.c, taps=3, pad=1,
                                    bias=bu)
                x = FMap(out, x.n, 2 * x.h, 2 * x.w, x.c)
        g, b = W.norm("decoder.conv_norm_out")
        hn = ops.groupnorm(x.data, x.c, x.c, x.n, x.h * x.w, g, b, 1e-6, True, groups=cfg.norm_num_groups)
        wn, bo = W.conv_n_padded("decoder.conv_out", self.COUT_PAD)
        if to_unit_range:  # image / 2 + 0.5 in the epilogue: 0.5 * (acc + bias + 1)
            if "decoder.conv_out.b01" not in W.t:
                b01 = bo.clone()
                b01[: cfg.out_channels] += 1.0
                W.t["decoder.conv_out.b01"] = b01
            bo = W.t["decoder.conv_out.b01"]
        img = ops.gemm_conv(hn, wn, n_img=x.n, h_in=x.h, w_in=x.w, c0=x.c, lda0=x.c, n_out=self.COUT_PAD, taps=3, pad=1,
                            bias=bo, out_f32=True, out_scale=0.5 if to_unit_range else 1.0)
        img = img.reshape(x.n, x.h, x.w, self.COUT_PAD)[..., : cfg.out_channels]
        return img.clamp(0, 1) if to_unit_range else img


class VaeEncoderEngine(VaeDecoderEngine):
    """AutoencoderKL.encode up to the moments (autoencoder_kl.py:160-171 -> Encoder.forward, vae.py:99-133, then
    quant_conv).  It extends the decoder engine: the resnets, the single-head mid-block attention and the packed-weight
    cache are the decoder's, so a module with both halves keeps one engine and can decode as well.
      * conv_in (3 -> C0, 3x3) is one K = 64 GEMM over the image-patch matrix of mdb_pack_image_patches;
      * Downsample2D(padding=0) (resnet.py:215-220) is the stride-2 implicit GEMM with pad 0 and h_out = (h - 2) // 2 + 1:
        the F.pad(0, 1, 0, 1) row and column are the taps past the far edge, which read zeros;
      * quant_conv (1x1, 8 -> 8) is folded into conv_out in fp32 (W' = W_q W_out per tap, b' = W_q b_out + b_q), whose fp32
        epilogue writes the NHWC moments [pixels, 8] directly."""

    PATCH_K = 64  # columns of the image-patch matrix: 27 taps x channels, zero-padded to one K block

    def __init__(self, cfg: arch.VaeConfig, sd, device):
        super().__init__(cfg, sd, device)
        if 9 * cfg.in_channels > self.PATCH_K:
            raise ValueError(f"VAE encoder: in_channels={cfg.in_channels} does not fit the {self.PATCH_K}-column patch matrix")
        self.down = arch.vae_encoder_blocks(cfg)

    def _conv_in_weight(self):
        W = self.W
        if "encoder.conv_in.wp" not in W.t:  # [C0, 3, 3, 3] -> [C0, 64], column (r*3 + s)*cin + c like the patch matrix
            w = W.raw("encoder.conv_in.weight").float()
            wp = torch.zeros((w.shape[0], self.PATCH_K), dtype=F32, device=w.device)
            wp[:, : 9 * w.shape[1]] = w.permute(0, 2, 3, 1).reshape(w.shape[0], -1)
            W.t["encoder.conv_in.wp"] = _bf(wp)
            W.t["encoder.conv_in.b"] = _f32(W.raw("encoder.conv_in.bias"))
        return W.t["encoder.conv_in.wp"], W.t["encoder.conv_in.b"]

    @property
    def moments_ld(self) -> int:
        """Row stride of the moments: 2 * latent_channels rounded up to the GEMM's 8-column output granularity."""
        return (2 * self.cfg.latent_channels + 7) // 8 * 8

    def _conv_out_weight(self):
        W = self.W
        if "encoder.conv_out.wq" not in W.t:
            wq = W.raw("quant_conv.weight").float()[:, :, 0, 0]  # [2c, 2c]
            wo = W.raw("encoder.conv_out.weight").float()        # [2c, C, 3, 3]
            m = wq.shape[0]
            wf = torch.zeros((self.moments_ld, *wo.shape[1:]), dtype=F32, device=wo.device)
            bf = torch.zeros((self.moments_ld,), dtype=F32, device=wo.device)
            wf[:m] = torch.einsum("ij,jkrs->ikrs", wq, wo)
            bf[:m] = wq @ W.raw("encoder.conv_out.bias").float() + W.raw("quant_conv.bias").float()
            # pack_conv_weight's (tap, channel) K order, stored in fold_dtype like the other folded products
            W.t["encoder.conv_out.wq"] = wf.permute(0, 2, 3, 1).reshape(wf.shape[0], -1).contiguous().to(W.fold_dtype)
            W.t["encoder.conv_out.bq"] = bf
        return W.t["encoder.conv_out.wq"], W.t["encoder.conv_out.bq"]

    def encode(self, images: torch.Tensor) -> torch.Tensor:
        """images: NCHW [n, in_channels, H, W] fp32 or bf16 (H, W divisible by 8) -> fp32 NHWC moments
        [n * H/8 * W/8, moments_ld], columns [0, c) the mean and [c, 2c) the logvar before its clamp."""
        cfg, W = self.cfg, self.W
        n, _, h, w = images.shape
        c0 = cfg.block_out_channels[0]
        wi, bi = self._conv_in_weight()
        xp = ops.pack_image_patches(images)
        x = FMap(ops.linear(xp, wi, bias=bi), n, h, w, c0)
        for _, resnets, down in self.down:
            for p, _, cout in resnets:
                x = self._resnet(p, x, cout)
            if down:
                wd, bd = W.conv(down)
                ho, wo = (x.h - 2) // 2 + 1, (x.w - 2) // 2 + 1
                out = ops.gemm_conv(x.data, wd, n_img=x.n, h_in=x.h, w_in=x.w, c0=x.c, lda0=x.c, n_out=x.c, taps=3, stride=2,
                                    pad=0, h_out=ho, w_out=wo, bias=bd)
                x = FMap(out, x.n, ho, wo, x.c)
        x = self._resnet("encoder.mid_block.resnets.0", x, x.c)
        x = self._attention(x, "encoder.mid_block.attentions.0")
        x = self._resnet("encoder.mid_block.resnets.1", x, x.c)
        g, b = W.norm("encoder.conv_norm_out")
        hn = ops.groupnorm(x.data, x.c, x.c, x.n, x.h * x.w, g, b, 1e-6, True, groups=cfg.norm_num_groups)
        wo_, bo = self._conv_out_weight()
        return ops.gemm_conv(hn, wo_, n_img=x.n, h_in=x.h, w_in=x.w, c0=x.c, lda0=x.c, n_out=self.moments_ld, taps=3, pad=1,
                             bias=bo, out_f32=True)
