"""B200-native SDXL ``UNet2DConditionModel``: drop-in for the diffusers class the reference trains
(train.py:1458-1465 loads it, train.py:2660-2667 configures it, train.py:2760-2761 calls it, train.py:2765 backprops).

Contract kept (SURVEY.md 8b): identical ``named_parameters()`` names / shapes / registration order (so Raven's
index-keyed checkpoints and the reference's ``get_unet_key_mapping`` stay valid), ``forward(sample, timestep,
encoder_hidden_states, added_cond_kwargs=...)`` returning an object with ``.sample`` (NCHW bf16), autograd
compatibility (``loss.backward()`` fills ``p.grad`` in the parameter dtype), ``enable_gradient_checkpointing`` /
``set_attn_processor`` / ``enable_xformers_memory_efficient_attention`` accepted as no-ops.

What is different (B200-first): activations are channels-last bf16 end to end, every op is a hand-written sm_100a
kernel from ``libaozora_b200.so`` (tcgen05 GEMM / implicit-GEMM conv / flash attention, fused norms and epilogues),
and the backward pass is an explicit reverse sweep over recorded closures -- no autograd graph inside the UNet, no
ATen kernels, no recompute (180 GB of HBM holds every activation of a 1024x1024 batch, so the reference's
always-on gradient checkpointing, train.py:2660, is unnecessary).  The ``nn.Conv2d`` / ``nn.Linear`` / ``nn.GroupNorm``
/ ``nn.LayerNorm`` children are used purely as parameter containers; their ``forward`` is never called.
"""
from __future__ import annotations

from types import SimpleNamespace

import torch
import torch.nn as nn

from . import _lib, ops

BF16 = torch.bfloat16


# ------------------------------------------------------------------------------------------------------------
# parameter containers (names and registration order follow diffusers; see SURVEY.md 8a appendix / 8b)
# ------------------------------------------------------------------------------------------------------------


class TimestepEmbedding(nn.Module):
    def __init__(self, in_dim, dim):
        super().__init__()
        self.linear_1 = nn.Linear(in_dim, dim)
        self.linear_2 = nn.Linear(dim, dim)


class ResnetBlock2D(nn.Module):
    def __init__(self, cin, cout, temb_dim, groups):
        super().__init__()
        self.norm1 = nn.GroupNorm(groups, cin, eps=1e-5)
        self.conv1 = nn.Conv2d(cin, cout, 3, padding=1)
        self.time_emb_proj = nn.Linear(temb_dim, cout)
        self.norm2 = nn.GroupNorm(groups, cout, eps=1e-5)
        self.conv2 = nn.Conv2d(cout, cout, 3, padding=1)
        self.conv_shortcut = nn.Conv2d(cin, cout, 1) if cin != cout else None


class Attention(nn.Module):
    def __init__(self, dim, ctx_dim):
        super().__init__()
        self.to_q = nn.Linear(dim, dim, bias=False)
        self.to_k = nn.Linear(ctx_dim, dim, bias=False)
        self.to_v = nn.Linear(ctx_dim, dim, bias=False)
        self.to_out = nn.ModuleList([nn.Linear(dim, dim), nn.Identity()])


class GEGLU(nn.Module):
    def __init__(self, dim, inner):
        super().__init__()
        self.proj = nn.Linear(dim, inner * 2)


class FeedForward(nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.net = nn.ModuleList([GEGLU(dim, dim * 4), nn.Identity(), nn.Linear(dim * 4, dim)])


class BasicTransformerBlock(nn.Module):
    def __init__(self, dim, ctx_dim):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim, eps=1e-5)
        self.attn1 = Attention(dim, dim)
        self.norm2 = nn.LayerNorm(dim, eps=1e-5)
        self.attn2 = Attention(dim, ctx_dim)
        self.norm3 = nn.LayerNorm(dim, eps=1e-5)
        self.ff = FeedForward(dim)


class Transformer2DModel(nn.Module):
    def __init__(self, dim, depth, ctx_dim, groups):
        super().__init__()
        self.norm = nn.GroupNorm(groups, dim, eps=1e-6)
        self.proj_in = nn.Linear(dim, dim)
        self.transformer_blocks = nn.ModuleList([BasicTransformerBlock(dim, ctx_dim) for _ in range(depth)])
        self.proj_out = nn.Linear(dim, dim)


class Downsample2D(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.conv = nn.Conv2d(c, c, 3, stride=2, padding=1)


class Upsample2D(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.conv = nn.Conv2d(c, c, 3, padding=1)


class DownBlock(nn.Module):
    def __init__(self, cfg, cin, cout, depth, has_attn, add_down):
        super().__init__()
        self.attentions = nn.ModuleList([Transformer2DModel(cout, depth, cfg.cross_attention_dim, cfg.norm_num_groups)
                                         for _ in range(cfg.layers_per_block)]) if has_attn else None
        self.resnets = nn.ModuleList([ResnetBlock2D(cin if i == 0 else cout, cout, cfg.time_embed_dim, cfg.norm_num_groups)
                                      for i in range(cfg.layers_per_block)])
        self.downsamplers = nn.ModuleList([Downsample2D(cout)]) if add_down else None


class MidBlock(nn.Module):
    def __init__(self, cfg, c, depth):
        super().__init__()
        self.attentions = nn.ModuleList([Transformer2DModel(c, depth, cfg.cross_attention_dim, cfg.norm_num_groups)])
        self.resnets = nn.ModuleList([ResnetBlock2D(c, c, cfg.time_embed_dim, cfg.norm_num_groups) for _ in range(2)])


class UpBlock(nn.Module):
    def __init__(self, cfg, cin, cout, cprev, depth, has_attn, add_up):
        super().__init__()
        n = cfg.layers_per_block + 1
        self.attentions = nn.ModuleList([Transformer2DModel(cout, depth, cfg.cross_attention_dim, cfg.norm_num_groups)
                                         for _ in range(n)]) if has_attn else None
        resnets = []
        for i in range(n):
            skip = cin if i == n - 1 else cout
            rin = cprev if i == 0 else cout
            resnets.append(ResnetBlock2D(rin + skip, cout, cfg.time_embed_dim, cfg.norm_num_groups))
        self.resnets = nn.ModuleList(resnets)
        self.upsamplers = nn.ModuleList([Upsample2D(cout)]) if add_up else None


class UNetConfig(SimpleNamespace):
    @property
    def time_embed_dim(self):
        return self.block_out_channels[0] * 4

    @property
    def add_in_dim(self):
        return self.pooled_dim + 6 * self.addition_time_embed_dim


def sdxl_config(in_channels=4, out_channels=4):
    return UNetConfig(in_channels=in_channels, out_channels=out_channels, block_out_channels=(320, 640, 1280),
                      layers_per_block=2, transformer_layers_per_block=(1, 2, 10), attention_head_dim=64,
                      cross_attention_dim=2048, norm_num_groups=32, addition_time_embed_dim=256, pooled_dim=1280,
                      down_has_attn=(False, True, True))


def tiny_config():
    """SDXL topology (3 levels, cross-attention on levels 1-2, skip concat) at small widths: parity-test size."""
    return UNetConfig(in_channels=4, out_channels=4, block_out_channels=(64, 128, 256), layers_per_block=2,
                      transformer_layers_per_block=(1, 1, 2), attention_head_dim=64, cross_attention_dim=128,
                      norm_num_groups=32, addition_time_embed_dim=32, pooled_dim=64, down_has_attn=(False, True, True))


# ------------------------------------------------------------------------------------------------------------
# gradient sink and layer closures
# ------------------------------------------------------------------------------------------------------------
class GradSink:
    """Collects parameter gradients produced by the reverse sweep (summing when a parameter is hit twice)."""

    def __init__(self):
        self.grads = {}
        self.on_grad = None        # optional callback(param, grad): data-parallel bucket scheduling during the sweep
        self.pending = []          # deferred Linear weight gradients: (params stacked by rows, dy, x)
        self.pending_late = []     # the same, flushed once per Transformer2DModel (cross-attention k/v: K = text tokens)
        self.dest = None           # optional callback(param) -> tensor the gradient must be written to (data-parallel flat buffer)

    def out_for(self, params):
        """Destination for the gradient of ``params`` (one parameter, or several stacked by rows): a view of the caller's
        gradient storage when it provides one and the row blocks are contiguous there, else None (fresh tensor)."""
        if self.dest is None:
            return None
        if not isinstance(params, (tuple, list)):
            return None if params in self.grads else self.dest(params)
        if any(p in self.grads for p in params):
            return None
        d0 = self.dest(params[0])
        if d0 is None:
            return None
        if len(params) == 1:
            return d0
        K = params[0].shape[1]
        rows = 0
        for p in params:
            d = self.dest(p)
            if d is None or d.data_ptr() != d0.data_ptr() + rows * K * d0.element_size():
                return None
            rows += p.shape[0]
        return torch.as_strided(d0, (rows, K), (K, 1))

    def wgrad(self, params, dy, x, defer=False):
        """dW = dyᵀ x for ``params`` (one parameter, or several stacked by rows).  ``defer``: queue it; ``flush`` then runs
        every queued gradient that shares the token count as ONE grouped persistent GEMM launch (a transformer block's
        six weight gradients = ~900 tiles = ~6 full waves on 148 SMs, instead of six ragged launches + split-K reduces)."""
        if defer == "late":
            self.pending_late.append((params, dy, x))
        elif defer:
            self.pending.append((params, dy, x))
        else:
            self._hand_out(params, ops.gemm(dy, x, a_mn=True, b_mn=True, out=self.out_for(params)))

    def bias_grad(self, b, dy):
        """db = column sums of dy."""
        self.add(b, ops.colsum(dy, out=self.out_for(b)))

    def _hand_out(self, params, dw):
        r = 0
        for p in params:
            self.add(p, dw[r:r + p.shape[0]])
            r += p.shape[0]

    def flush(self, late=False):
        if late:
            jobs, self.pending_late = self.pending_late, []
        else:
            jobs, self.pending = self.pending, []
        by_k = {}
        for job in jobs:
            by_k.setdefault(job[2].shape[0], []).append(job)
        for group in by_k.values():
            if len(group) == 1:
                params, dy, x = group[0]
                self._hand_out(params, ops.gemm(dy, x, a_mn=True, b_mn=True, out=self.out_for(params)))
                continue
            outs = ops.gemm_grouped([(dy, x, self.out_for(params)) for params, dy, x in group], a_mn=True, b_mn=True)
            for (params, _, _), dw in zip(group, outs):
                self._hand_out(params, dw)

    def add(self, p, g):
        g = g.view_as(p)
        cur = self.grads.get(p)
        if cur is None:
            self.grads[p] = g
            if self.on_grad is not None:
                self.on_grad(p, g)
        elif self.on_grad is not None:
            # under data parallel on_grad may already have launched the reduce-scatter of this parameter's bucket: a later
            # contribution would be lost silently.  No SDXL parameter is used twice; anything else must fail loudly.
            raise _lib.AozoraError("GradSink: second gradient contribution to a parameter whose gradient was already handed to on_grad")
        else:
            ops.add(cur, g, out=cur)


class _PackCache:
    """Packed conv weights, re-packed only when the parameter changed (tensor version counter)."""

    def __init__(self):
        self.d = {}

    def get(self, w, need_dgrad):
        key = id(w)
        ent = self.d.get(key)
        if ent is not None and ent[0] == w._version and ent[1] is w and (ent[3] is not None or not need_dgrad):
            return ent[2], ent[3]
        wf, wd = ops.pack_conv_weight(w.detach(), need_dgrad=need_dgrad)
        self.d[key] = (w._version, w, wf, wd)
        return wf, wd


def _linear(x, w, b, G, *, residual=None, need_dx=True, w_param=None, defer=False):
    """y = x Wᵀ + b (+ residual); returns (y, bwd) with bwd(dy, out=None, accumulate=False) -> dx.
    ``w_param``: the parameter ``w`` is a reshaped view of (1x1 conv weights used as a matrix).
    ``defer``: queue the weight gradient for a grouped launch (``G.flush()``)."""
    y = ops.gemm(x, w, bias=b, residual=residual)
    wp = w if w_param is None else w_param

    def bwd(dy, out=None, accumulate=False, bias_done=False):
        """``bias_done``: the producer of ``dy`` (a LayerNorm backward, see ``_layernorm``) already formed this layer's bias gradient."""
        if wp.requires_grad:
            if w_param is None:
                G.wgrad((wp,), dy, x, defer=defer)
            else:
                G.add(wp, ops.gemm(dy, x, a_mn=True, b_mn=True))
        if b is not None and b.requires_grad and not bias_done:
            G.bias_grad(b, dy)          # right away: dy is still L2-resident (deferring it to the block's flush measured slower)
        if not need_dx:
            return None
        return ops.gemm(dy, w, b_mn=True, out=out, accumulate=accumulate, splits=1 if accumulate else None)

    return y, bwd


def _geglu(x, w, b, G, defer=False):
    aux = torch.empty((x.shape[0], w.shape[0]), dtype=BF16, device=x.device)
    y = ops.gemm(x, w, bias=b, epi=ops.EPI_GEGLU, aux=aux)

    def bwd(dy):
        daux = ops.geglu_bwd(dy, aux)
        if b.requires_grad:
            G.bias_grad(b, daux)
        if w.requires_grad:
            G.wgrad((w,), daux, x, defer=defer)
        return ops.gemm(daux, w, b_mn=True)

    return y, bwd


def _conv(x, mod, G, packs, *, stride=1, rowgroup_bias=None, residual=None, need_dx=True, cin_real=None):
    """3x3 conv (pad 1) over NHWC; returns (y, bwd).  ``cin_real`` < x.shape[-1] means x carries zero-padded channels."""
    w, b = mod.weight, mod.bias
    cout, ks = w.shape[0], w.shape[2]
    wf, wd = packs.get(w, need_dgrad=need_dx)
    y = ops.conv_fwd(x, wf, cout, ks, stride=stride, pad=ks // 2, bias=b, rowgroup_bias=rowgroup_bias, residual=residual)

    def bwd(dy):
        # dy may carry zero-padded output channels (conv_out: 4 real channels of 8)
        if w.requires_grad:
            gw = G.out_for(w) if dy.shape[-1] == cout else None           # padded output channels: slice a temporary instead
            dw = ops.conv_wgrad(dy, x, ks, stride=stride, pad=ks // 2, cin_real=cin_real, grad_w=gw)
            G.add(w, dw[:cout])
        if b.requires_grad:
            gb = G.out_for(b) if dy.shape[-1] == cout else None
            G.add(b, ops.colsum(dy.view(-1, dy.shape[-1]), out=gb)[:cout])
        if not need_dx:
            return None
        cin = x.shape[-1]
        if stride == 1:
            return ops.conv_fwd(dy, wd, cin, ks, stride=1, pad=ks // 2, flip=True)
        dyz = ops.zero_insert2x(dy, x.shape[1], x.shape[2])
        return ops.conv_fwd(dyz, wd, cin, ks, stride=1, pad=ks // 2, flip=True)

    return y, bwd


def _groupnorm(x, mod, G, silu):
    y, mean, rstd = ops.groupnorm_fwd(x, mod.weight, mod.bias, mod.eps, silu)

    def bwd(dy, dres=None):
        need = mod.weight.requires_grad or mod.bias.requires_grad
        both = mod.weight.requires_grad and mod.bias.requires_grad
        dx, dg, db = ops.groupnorm_bwd(dy, x, mod.weight, mod.bias, mean, rstd, silu, need_param_grads=need, dres=dres,
                                       dgamma=G.out_for(mod.weight) if both else None, dbeta=G.out_for(mod.bias) if both else None)
        if mod.weight.requires_grad:
            G.add(mod.weight, dg)
        if mod.bias.requires_grad:
            G.add(mod.bias, db)
        return dx

    return y, bwd


def _layernorm(x, mod, G):
    y, mean, rstd = ops.layernorm_fwd(x, mod.weight, mod.bias, mod.eps)

    def bwd(dy, dres=None, bias_of_dx=None):
        """``bias_of_dx``: the bias of the Linear whose output is this LayerNorm's input (the previous sublayer's to_out / ff.net.2,
        or proj_in): its gradient is the column sum of the dx computed here, formed in the same pass (the consumer of dx is then
        called with ``bias_done=True``)."""
        both = mod.weight.requires_grad and mod.bias.requires_grad
        dcol = None
        if bias_of_dx is not None and bias_of_dx.requires_grad:
            dcol = G.out_for(bias_of_dx)
            if dcol is None:
                dcol = torch.empty_like(bias_of_dx)
        dx, dg, db = ops.layernorm_bwd(dy, x, mod.weight, mean, rstd, dres=dres, dgamma=G.out_for(mod.weight) if both else None,
                                       dbeta=G.out_for(mod.bias) if both else None, dx_colsum=dcol)
        if mod.weight.requires_grad:
            G.add(mod.weight, dg)
        if mod.bias.requires_grad:
            G.add(mod.bias, db)
        if dcol is not None:
            G.add(bias_of_dx, dcol)
        return dx

    return y, bwd


def _attention(q2d, k2d, v2d, B, Tq, Tk):
    """q2d / k2d / v2d: [B*T, C] (column blocks of a fused projection output are fine: only the row stride differs).
    bwd(do2d, out=None): ``out`` = optional (dq2d, dk2d, dv2d) destinations of the same kind."""
    C = q2d.shape[1]
    H = C // 64
    q, k, v = q2d.view(B, Tq, H, 64), k2d.view(B, Tk, H, 64), v2d.view(B, Tk, H, 64)
    o, lse = ops.attn_fwd(q, k, v, 0.125)

    def bwd(do2d, out=None):
        if out is not None:
            out = (out[0].view(B, Tq, H, 64), out[1].view(B, Tk, H, 64), out[2].view(B, Tk, H, 64))
        dq, dk, dv = ops.attn_bwd(q, k, v, o, do2d.view(B, Tq, H, 64), lse, 0.125, out=out)
        return dq.view(B * Tq, C), dk.view(B * Tk, C), dv.view(B * Tk, C)

    return o.view(B * Tq, C), bwd


def _stacked(params):
    """One [sum(rows), K] matrix over Linear weights that lie back to back in the same storage (see
    ``fuse_projection_storage``), or None.  The fused matrix lets to_q/to_k/to_v (and cross-attention to_k/to_v) run as
    ONE projection GEMM forward, one dgrad and one wgrad instead of three each."""
    w0 = params[0]
    if len({p.requires_grad for p in params}) != 1:
        return None
    K = w0.shape[1]
    base = w0.untyped_storage().data_ptr()
    rows = 0
    for w in params:
        if (w.dtype != w0.dtype or w.dim() != 2 or w.shape[1] != K or not w.is_contiguous()
                or w.untyped_storage().data_ptr() != base or w.data_ptr() != w0.data_ptr() + rows * K * w.element_size()):
            return None
        rows += w.shape[0]
    return torch.as_strided(w0.detach(), (rows, K), (K, 1))


def _linear_stacked(x, wcat, params, G, *, need_dx=True, defer=False):
    """y = x [W_0; W_1; ...]ᵀ for bias-free projections sharing the input; returns (y [M, sum rows], bwd).
    bwd(dy [M, sum rows]) -> dx; the weight gradient is produced by one GEMM and handed out as row blocks."""
    y = ops.gemm(x, wcat)

    def bwd(dy):
        if params[0].requires_grad:
            G.wgrad(params, dy, x, defer=defer)
        if not need_dx:
            return None
        return ops.gemm(dy, wcat, b_mn=True)

    return y, bwd


def _cross_kv(blocks, ctx, G):
    """attn2 key/value projections of every block of a Transformer2DModel in ONE grouped launch: they all read the same text
    embedding (M = B x 77 rows) and do not depend on the blocks before them, so ten 15-microsecond GEMMs that each fill a
    fraction of the GPU become one.  Returns {block index: kv [B*Tc, 2C]} for the blocks whose k/v weights are stacked."""
    idx, probs = [], []
    for i, blk in enumerate(blocks):
        w = _stacked((blk.attn2.to_k.weight, blk.attn2.to_v.weight))
        if w is not None:
            idx.append(i)
            probs.append((ctx, w, None))
    if len(probs) < 2:
        return {}
    return dict(zip(idx, ops.gemm_grouped(probs, a_mn=False, b_mn=False)))


def _basic_block(blk, x, ctx, B, T, Tc, G, kv_pre=None):
    """Pre-LN self-attention, cross-attention and GEGLU feed-forward, each with a residual fused into the
    producing GEMM's epilogue.  x: [B*T, C]; ctx: [B*Tc, ctx_dim]."""
    a1, a2, ff = blk.attn1, blk.attn2, blk.ff
    C = x.shape[1]
    n1, b_n1 = _layernorm(x, blk.norm1, G)
    p_qkv = (a1.to_q.weight, a1.to_k.weight, a1.to_v.weight)
    w_qkv = _stacked(p_qkv)
    if w_qkv is not None:
        qkv, b_qkv = _linear_stacked(n1, w_qkv, p_qkv, G, defer=True)
        q, k, v = qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:]
    else:
        q, b_q = _linear(n1, a1.to_q.weight, None, G, defer=True)
        k, b_k = _linear(n1, a1.to_k.weight, None, G, defer=True)
        v, b_v = _linear(n1, a1.to_v.weight, None, G, defer=True)
    o1, b_at1 = _attention(q, k, v, B, T, T)
    x1, b_o1 = _linear(o1, a1.to_out[0].weight, a1.to_out[0].bias, G, residual=x, defer=True)
    n2, b_n2 = _layernorm(x1, blk.norm2, G)
    q2, b_q2 = _linear(n2, a2.to_q.weight, None, G, defer=True)
    p_kv = (a2.to_k.weight, a2.to_v.weight)
    w_kv = _stacked(p_kv)
    if w_kv is not None and kv_pre is not None:
        kv2 = kv_pre                                 # computed with the other blocks' (see _cross_kv); gradient flushed "late"

        def b_kv2(dkv):
            if p_kv[0].requires_grad:
                G.wgrad(p_kv, dkv, ctx, defer="late")
        k2, v2 = kv2[:, :C], kv2[:, C:]
    elif w_kv is not None:
        kv2, b_kv2 = _linear_stacked(ctx, w_kv, p_kv, G, need_dx=False)
        k2, v2 = kv2[:, :C], kv2[:, C:]
    else:
        k2, b_k2 = _linear(ctx, a2.to_k.weight, None, G, need_dx=False)
        v2, b_v2 = _linear(ctx, a2.to_v.weight, None, G, need_dx=False)
    o2, b_at2 = _attention(q2, k2, v2, B, T, Tc)
    x2, b_o2 = _linear(o2, a2.to_out[0].weight, a2.to_out[0].bias, G, residual=x1, defer=True)
    n3, b_n3 = _layernorm(x2, blk.norm3, G)
    g, b_g = _geglu(n3, ff.net[0].proj.weight, ff.net[0].proj.bias, G, defer=True)
    x3, b_f2 = _linear(g, ff.net[2].weight, ff.net[2].bias, G, residual=x2, defer=True)
    M, Mc = x.shape[0], ctx.shape[0]
    del n1, q, k, v, o1, n2, q2, k2, v2, o2, n3, g

    def bwd(dy, dy_bias_done=False, prev_bias=None):
        """``dy_bias_done``: ff.net.2's bias gradient (column sums of dy) came with dy from the LayerNorm backward that produced it;
        ``prev_bias``: the bias whose gradient is the column sum of the dx returned here (the previous block's ff.net.2, or proj_in)."""
        dg = b_f2(dy, bias_done=dy_bias_done)
        dn3 = b_g(dg)
        dx2 = b_n3(dn3, dres=dy, bias_of_dx=a2.to_out[0].bias)
        do2 = b_o2(dx2, bias_done=True)
        if w_kv is not None:
            dkv2 = torch.empty((Mc, 2 * C), dtype=BF16, device=dy.device)
            dq2 = torch.empty((M, C), dtype=BF16, device=dy.device)
            b_at2(do2, out=(dq2, dkv2[:, :C], dkv2[:, C:]))
            b_kv2(dkv2)
        else:
            dq2, dk2, dv2 = b_at2(do2)
            b_k2(dk2)
            b_v2(dv2)
        dn2 = b_q2(dq2)
        dx1 = b_n2(dn2, dres=dx2, bias_of_dx=a1.to_out[0].bias)
        do1 = b_o1(dx1, bias_done=True)
        if w_qkv is not None:
            dqkv = torch.empty((M, 3 * C), dtype=BF16, device=dy.device)
            b_at1(do1, out=(dqkv[:, :C], dqkv[:, C:2 * C], dqkv[:, 2 * C:]))
            dn1 = b_qkv(dqkv)
        else:
            dq, dk, dv = b_at1(do1)
            dn1 = b_q(dq)
            b_k(dk, out=dn1, accumulate=True)
            b_v(dv, out=dn1, accumulate=True)
        G.flush()                      # this block's queued weight gradients: one grouped launch
        return b_n1(dn1, dres=dx1, bias_of_dx=prev_bias)

    return x3, bwd


def _transformer(tr, x, ctx, Tc, G):
    """Transformer2DModel with linear projections: x + proj_out(blocks(proj_in(GN(x)))); x: [B,H,W,C]."""
    B, H, W, C = x.shape
    T = H * W
    hn, b_gn = _groupnorm(x, tr.norm, G, silu=False)
    h, b_pi = _linear(hn.view(B * T, C), tr.proj_in.weight, tr.proj_in.bias, G)
    del hn
    blocks = []
    kv_pre = _cross_kv(tr.transformer_blocks, ctx, G)
    for i, blk in enumerate(tr.transformer_blocks):
        h, b_blk = _basic_block(blk, h, ctx, B, T, Tc, G, kv_pre=kv_pre.get(i))
        blocks.append(b_blk)
    del kv_pre
    y, b_po = _linear(h, tr.proj_out.weight, tr.proj_out.bias, G, residual=x.view(B * T, C))
    del h

    def bwd(dy):
        dy2 = dy.view(B * T, C)
        dh = b_po(dy2)
        # the dx a block returns is the gradient of the PREVIOUS Linear's output -- the block before it's ff.net.2, or proj_in --
        # so that layer's bias gradient (column sums of dx) is formed by the block's first LayerNorm backward
        n = len(blocks)
        for i in range(n - 1, -1, -1):
            prev_bias = tr.transformer_blocks[i - 1].ff.net[2].bias if i > 0 else tr.proj_in.bias
            dh = blocks[i](dh, dy_bias_done=(i < n - 1), prev_bias=prev_bias)
            blocks[i] = None
        blocks.clear()
        G.flush(late=True)             # cross-attention k/v weight gradients of all blocks: one grouped launch
        dhn = b_pi(dh, bias_done=True)
        return b_gn(dhn.view(B, H, W, C), dres=dy)

    return y.view(B, H, W, C), bwd


def _resnet(res, x, semb, G, packs):
    """ResnetBlock2D: x + conv2(silu(gn2(conv1(silu(gn1(x))) + temb))) with a 1x1 shortcut when Cin != Cout.
    The time-embedding add and the residual add live in the conv epilogues."""
    B, H, W, Cin = x.shape
    Cout = res.conv1.weight.shape[0]
    h1, b_g1 = _groupnorm(x, res.norm1, G, silu=True)
    t, b_t = _linear(semb, res.time_emb_proj.weight, res.time_emb_proj.bias, G)
    c1, b_c1 = _conv(h1, res.conv1, G, packs, rowgroup_bias=t)
    del h1
    h2, b_g2 = _groupnorm(c1, res.norm2, G, silu=True)
    if res.conv_shortcut is not None:
        scw = res.conv_shortcut.weight
        sc, b_sc = _linear(x.view(B * H * W, Cin), scw.detach().view(Cout, Cin), res.conv_shortcut.bias, G, w_param=scw)
        sc = sc.view(B, H, W, Cout)
    else:
        sc, b_sc = x, None
    y, b_c2 = _conv(h2, res.conv2, G, packs, residual=sc)
    del h2, sc, c1

    def bwd(dy):
        dh2 = b_c2(dy)
        dc1 = b_g2(dh2)
        dt = ops.colsum_grouped(dc1)
        dsemb = b_t(dt)
        dh1 = b_c1(dc1)
        dsc = b_sc(dy.view(B * H * W, Cout)).view(B, H, W, Cin) if b_sc is not None else dy
        return b_g1(dh1, dres=dsc), dsemb

    return y, bwd


# ------------------------------------------------------------------------------------------------------------
# the model
# ------------------------------------------------------------------------------------------------------------
class UNet2DConditionModel(nn.Module):
    def __init__(self, cfg: UNetConfig | None = None):
        super().__init__()
        cfg = cfg or sdxl_config()
        self.cfg = cfg
        self.config = SimpleNamespace(in_channels=cfg.in_channels, out_channels=cfg.out_channels)
        boc = cfg.block_out_channels
        self.conv_in = nn.Conv2d(cfg.in_channels, boc[0], 3, padding=1)
        self.time_embedding = TimestepEmbedding(boc[0], cfg.time_embed_dim)
        self.add_embedding = TimestepEmbedding(cfg.add_in_dim, cfg.time_embed_dim)
        self.down_blocks = nn.ModuleList()
        self.up_blocks = nn.ModuleList()          # registered before mid_block, as diffusers does
        cout = boc[0]
        for i, c in enumerate(boc):
            cin, cout = cout, c
            self.down_blocks.append(DownBlock(cfg, cin, cout, cfg.transformer_layers_per_block[i], cfg.down_has_attn[i],
                                              add_down=(i != len(boc) - 1)))
        self.mid_block = MidBlock(cfg, boc[-1], cfg.transformer_layers_per_block[-1])
        rev = list(reversed(boc))
        rdepth = list(reversed(cfg.transformer_layers_per_block))
        rattn = list(reversed(cfg.down_has_attn))
        cout = rev[0]
        for i, c in enumerate(rev):
            cprev, cout = cout, c
            cin = rev[min(i + 1, len(boc) - 1)]
            self.up_blocks.append(UpBlock(cfg, cin, cout, cprev, rdepth[i], rattn[i], add_up=(i != len(boc) - 1)))
        self.conv_norm_out = nn.GroupNorm(cfg.norm_num_groups, boc[0], eps=1e-5)
        self.conv_out = nn.Conv2d(boc[0], cfg.out_channels, 3, padding=1)
        self._packs = _PackCache()
        self.gradient_checkpointing = False
        self._fused_storage_ok = False

    # ---- fused projection storage ------------------------------------------------------------------------------
    def _apply(self, fn, *a, **k):
        # .to() / .cuda() / .bfloat16() give every parameter fresh storage: the stacked layout must be rebuilt
        self._fused_storage_ok = False
        return super()._apply(fn, *a, **k)

    def fuse_projection_storage(self):
        """Place attn1.{to_q,to_k,to_v}.weight and attn2.{to_k,to_v}.weight of every transformer block back to back in one
        buffer (the parameters become row-block views; names, shapes, values and order are untouched) so each group runs
        as ONE projection GEMM.  Groups with mixed ``requires_grad`` or parameters owned by a
        data-parallel flat buffer (already adjacent there) are left as they are.  Idempotent; called lazily by forward."""
        for m in self.modules():
            if not isinstance(m, BasicTransformerBlock):
                continue
            for group in ((m.attn1.to_q.weight, m.attn1.to_k.weight, m.attn1.to_v.weight), (m.attn2.to_k.weight, m.attn2.to_v.weight)):
                if _stacked(group) is not None or len({p.requires_grad for p in group}) != 1:
                    continue
                if any(getattr(p, "_aoz_flat", False) for p in group) or len({(p.dtype, p.shape[1]) for p in group}) != 1:
                    continue
                with torch.no_grad():
                    buf = torch.cat([p.detach() for p in group], dim=0)
                    r = 0
                    for p in group:
                        p.data = buf[r:r + p.shape[0]]
                        r += p.shape[0]
        self._fused_storage_ok = True

    # ---- reference boundary: UNet2DConditionModel.from_single_file (train.py:1458-1464) -------------------
    @classmethod
    def from_single_file(cls, path, torch_dtype=None, low_cpu_mem_usage=True, in_channels=None, out_channels=None, device="cpu", **_):
        """Load the UNet of an SDXL single-file ``.safetensors`` checkpoint (LDM key names) -- see ``checkpoint.py``."""
        from .checkpoint import load_unet_single_file
        return load_unet_single_file(path, torch_dtype=torch_dtype or BF16, device=device, in_channels=in_channels, out_channels=out_channels)

    # ---- reference boundary no-ops (train.py:199-229, 2660) ----------------------------------------------
    def enable_gradient_checkpointing(self):
        self.gradient_checkpointing = True        # accepted; nothing is recomputed on B200 (see module docstring)

    def set_attn_processor(self, processor):
        pass

    def enable_xformers_memory_efficient_attention(self, *a, **k):
        pass

    # ---- core: forward over channels-last tensors, returning the reverse-sweep closure -------------------
    def _forward_units(self):
        """The modules ``forward_nhwc`` announces to ``param_gate`` before it first reads their parameters, in execution order
        (data parallel with a deferred all-gather orders its buckets by this and lets every unit wait only for its own)."""
        yield self.time_embedding
        yield self.add_embedding
        yield self.conv_in
        for blk in self.down_blocks:
            for i, res in enumerate(blk.resnets):
                yield res
                if blk.attentions is not None:
                    yield blk.attentions[i]
            if blk.downsamplers is not None:
                yield blk.downsamplers[0]
        yield self.mid_block.resnets[0]
        yield self.mid_block.attentions[0]
        yield self.mid_block.resnets[1]
        for blk in self.up_blocks:
            for i, res in enumerate(blk.resnets):
                yield res
                if blk.attentions is not None:
                    yield blk.attentions[i]
            if blk.upsamplers is not None:
                yield blk.upsamplers[0]
        yield self.conv_norm_out
        yield self.conv_out

    def forward_nhwc(self, x8, cond, ctx, text_embeds, time_ids, taps=None):
        """x8: [B,H,W,8] bf16 (latent channels zero-padded to 8); cond: fp32 [B] timesteps; ctx: [B,Tc,ctx_dim] bf16;
        text_embeds [B,pooled] bf16; time_ids [B,6] (bf16 values).  Returns (pred [B,H,W,out_channels] bf16, bwd) where
        ``bwd(dpred8)`` takes dL/dpred padded to 8 channels and returns {param: grad}."""
        cfg = self.cfg
        if not self._fused_storage_ok:
            self.fuse_projection_storage()
        G = GradSink()
        packs = self._packs
        B = x8.shape[0]
        Tc = ctx.shape[1]
        ctx2 = ctx.reshape(B * Tc, ctx.shape[2]).contiguous()
        gate = getattr(self, "param_gate", None) or (lambda mod: None)       # see _forward_units

        # --- embeddings (Timesteps -> MLP; text_time addition embedding) ---
        t_emb = ops.timestep_embedding(cond.float().contiguous(), cfg.block_out_channels[0])
        gate(self.time_embedding)
        e1, b_te1 = _linear(t_emb, self.time_embedding.linear_1.weight, self.time_embedding.linear_1.bias, G, need_dx=False)
        e1s = ops.silu_fwd(e1)
        e2, b_te2 = _linear(e1s, self.time_embedding.linear_2.weight, self.time_embedding.linear_2.bias, G)
        tid = ops.timestep_embedding(time_ids.reshape(-1).float().contiguous(), cfg.addition_time_embed_dim)
        add_in = torch.empty((B, cfg.add_in_dim), dtype=BF16, device=x8.device)
        ops.copy_channels(text_embeds.contiguous(), 0, add_in, 0, cfg.pooled_dim)
        ops.copy_channels(tid.view(B, 6 * cfg.addition_time_embed_dim), 0, add_in, cfg.pooled_dim, 6 * cfg.addition_time_embed_dim)
        gate(self.add_embedding)
        a1, b_ae1 = _linear(add_in, self.add_embedding.linear_1.weight, self.add_embedding.linear_1.bias, G, need_dx=False)
        a1s = ops.silu_fwd(a1)
        emb, b_ae2 = _linear(a1s, self.add_embedding.linear_2.weight, self.add_embedding.linear_2.bias, G, residual=e2)
        semb = ops.silu_fwd(emb)

        tape = []          # closures in forward order: (kind, fn)

        # --- down path ---
        gate(self.conv_in)
        x, b_cin = _conv(x8, self.conv_in, G, packs, need_dx=False, cin_real=cfg.in_channels)
        skips = [x]
        tape.append(("conv_in", b_cin))
        for bi, blk in enumerate(self.down_blocks):
            for i, res in enumerate(blk.resnets):
                gate(res)
                x, b_r = _resnet(res, x, semb, G, packs)
                tape.append(("res", b_r))
                if blk.attentions is not None:
                    gate(blk.attentions[i])
                    x, b_a = _transformer(blk.attentions[i], x, ctx2, Tc, G)
                    tape.append(("attn", b_a))
                skips.append(x)
                tape.append(("skip_out", None))
            if blk.downsamplers is not None:
                gate(blk.downsamplers[0])
                x, b_d = _conv(x, blk.downsamplers[0].conv, G, packs, stride=2)
                tape.append(("conv", b_d))
                skips.append(x)
                tape.append(("skip_out", None))
            if taps is not None:
                taps[f"down_blocks.{bi}"] = x
        # --- mid ---
        gate(self.mid_block.resnets[0])
        x, b_r = _resnet(self.mid_block.resnets[0], x, semb, G, packs)
        tape.append(("res", b_r))
        gate(self.mid_block.attentions[0])
        x, b_a = _transformer(self.mid_block.attentions[0], x, ctx2, Tc, G)
        tape.append(("attn", b_a))
        gate(self.mid_block.resnets[1])
        x, b_r = _resnet(self.mid_block.resnets[1], x, semb, G, packs)
        tape.append(("res", b_r))
        if taps is not None:
            taps["mid_block"] = x
        # --- up path ---
        for bi, blk in enumerate(self.up_blocks):
            for i, res in enumerate(blk.resnets):
                skip = skips.pop()
                cat = ops.concat_channels(x, skip)
                tape.append(("cat", (x.shape[-1], skip.shape[-1])))
                gate(res)
                x, b_r = _resnet(res, cat, semb, G, packs)
                del cat
                tape.append(("res", b_r))
                if blk.attentions is not None:
                    gate(blk.attentions[i])
                    x, b_a = _transformer(blk.attentions[i], x, ctx2, Tc, G)
                    tape.append(("attn", b_a))
            if blk.upsamplers is not None:
                gate(blk.upsamplers[0])
                xu = ops.upsample2x_fwd(x)
                x, b_u = _conv(xu, blk.upsamplers[0].conv, G, packs)
                del xu
                tape.append(("up", b_u))
            if taps is not None:
                taps[f"up_blocks.{bi}"] = x
        gate(self.conv_norm_out)
        hn, b_gno = _groupnorm(x, self.conv_norm_out, G, silu=True)
        gate(self.conv_out)
        pred, b_cout = _conv(hn, self.conv_out, G, packs)
        del hn, x
        n_skips = 3 * len(self.up_blocks)

        def bwd(dpred8, on_grad=None, dest=None):
            G.on_grad = on_grad
            G.dest = dest
            dsemb = None

            def acc_semb(d):
                nonlocal dsemb
                if dsemb is None:
                    dsemb = d
                else:
                    ops.add(dsemb, d, out=dsemb)

            dx = b_gno(b_cout(dpred8))
            skip_grads = []                      # gradients of skip tensors, produced in up-path reverse order
            while tape:
                kind, fn = tape.pop()
                if kind == "res":
                    dx, ds = fn(dx)
                    acc_semb(ds)
                elif kind == "attn" or kind == "conv":
                    dx = fn(dx)
                elif kind == "up":
                    dx = ops.upsample2x_bwd(fn(dx))
                elif kind == "cat":
                    ca, cb = fn
                    dskip = torch.empty(tuple(dx.shape[:-1]) + (cb,), dtype=BF16, device=dx.device)
                    ops.copy_channels(dx, ca, dskip, 0, cb)
                    dxa = torch.empty(tuple(dx.shape[:-1]) + (ca,), dtype=BF16, device=dx.device)
                    ops.copy_channels(dx, 0, dxa, 0, ca)
                    skip_grads.append(dskip)
                    dx = dxa
                elif kind == "skip_out":
                    # this tensor was also consumed by an up-block concat.  The reverse sweep met the concats in
                    # order skip[0], skip[1], ... and now walks the skips from the last one pushed: LIFO.
                    ops.add(dx, skip_grads.pop(), out=dx)
                elif kind == "conv_in":
                    ops.add(dx, skip_grads.pop(), out=dx)
                    fn(dx)
            assert not skip_grads
            # --- embedding MLPs ---
            demb = ops.silu_bwd(dsemb, emb)
            da1s = b_ae2(demb)                        # also: d e2 = demb (residual)
            b_ae1(ops.silu_bwd(da1s, a1))
            de1s = b_te2(demb)
            b_te1(ops.silu_bwd(de1s, e1))
            G.flush()
            G.flush(late=True)
            return G.grads

        assert len(skips) == 0 and n_skips >= 0
        return pred, bwd

    # ---- drop-in call (train.py:2760-2761) ------------------------------------------------------------------
    def forward(self, sample, timestep, encoder_hidden_states, added_cond_kwargs=None, **_):
        if not sample.is_cuda:
            raise _lib.AozoraError("UNet2DConditionModel: CUDA tensors required (the B200 path has no CPU fallback)")
        params = [p for p in self.parameters()]
        te = added_cond_kwargs["text_embeds"]
        ti = added_cond_kwargs["time_ids"]
        B = sample.shape[0]
        ts = timestep if torch.is_tensor(timestep) else torch.tensor([timestep], device=sample.device)
        if ts.dim() == 0:
            ts = ts[None]
        ts = ts.to(sample.device).float().expand(B).contiguous()
        out = _UNetFunction.apply(self, sample, ts, encoder_hidden_states, te, ti, *params)
        return SimpleNamespace(sample=out)


class _UNetFunction(torch.autograd.Function):
    """Bridges the explicit reverse sweep into autograd so that ``loss.backward()`` (train.py:2765) works unchanged."""

    @staticmethod
    def forward(ctx, model, sample, ts, ehs, text_embeds, time_ids, *params):
        x8 = ops.nchw_to_nhwc(sample.detach().contiguous(), cpad=8)
        pred, bwd = model.forward_nhwc(x8, ts, ehs.detach().to(BF16).contiguous(), text_embeds.detach().to(BF16),
                                       time_ids.detach())
        ctx.bwd = bwd
        ctx.params = params
        if not any(p.requires_grad for p in params):
            ctx.bwd = None                      # inference call: drop the saved activations right away
        return ops.nhwc_to_nchw(pred, c=model.cfg.out_channels)

    @staticmethod
    def backward(ctx, dsample):
        bwd, ctx.bwd = ctx.bwd, None
        d8 = ops.nchw_to_nhwc(dsample.contiguous(), cpad=8)
        grads = bwd(d8)
        out = [None] * 6
        for p in ctx.params:
            g = grads.get(p) if p.requires_grad else None
            out.append(g)
        return tuple(out)


def init_weights_(model: nn.Module, seed: int = 42, std: float = 0.02):
    """Fixed synthetic init (SURVEY.md 8d): drawn in ``named_parameters()`` order from one CPU generator, so any
    module with the same names / shapes / order (the oracle's restatement included) receives identical tensors."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    with torch.no_grad():
        for name, p in model.named_parameters():
            t = torch.randn(p.shape, generator=g, dtype=torch.float32) * std
            if p.dim() == 1 and name.endswith("weight"):
                t = t + 1.0
            p.copy_(t.to(p.dtype))
    return model


def init_weights_fast_(model: nn.Module, seed: int = 42, std: float = 0.02):
    """On-device synthetic init for benchmarks: N(0, std) matrices / filters, unit norm scales, zero biases."""
    dev = next(model.parameters()).device
    g = torch.Generator(device=dev).manual_seed(seed)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if p.dim() == 1:
                p.fill_(1.0 if name.endswith("weight") else 0.0)
            else:
                p.normal_(0.0, std, generator=g)
    return model
