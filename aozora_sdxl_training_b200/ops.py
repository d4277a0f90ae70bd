"""Raw (non-autograd) Python wrappers over the C ABI: torch tensors in, kernels launched on the current stream.

PyTorch is plumbing here (device memory, streams).  Every function launches hand-written sm_100a kernels from
``libaozora_b200.so``; nothing falls back to ATen or the CPU.  A launch counter (``launch_count``) feeds
``bench.py``'s ``gpu_launches``.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib

BF16 = torch.bfloat16
_DT = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}

launch_count = 0          # number of aoz_* compute calls issued (each is >= 1 kernel launch)
trace = None              # tools/gemm_in_step.py: when a list, every GEMM / conv call appends (kind, shape...) in launch order


def _count(n=1):
    global launch_count
    launch_count += n


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return 0 if t is None else t.data_ptr()


def _chk(t, name, dtype=BF16, contiguous=True):
    if not t.is_cuda:
        raise _lib.AozoraError(f"{name}: expected a CUDA tensor (aozora-b200 has no CPU path)")
    if dtype is not None and t.dtype != dtype:
        raise _lib.AozoraError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if contiguous and not t.is_contiguous():
        raise _lib.AozoraError(f"{name}: expected a contiguous tensor")
    return t


_workspaces = {}


def workspace(nfloats: int, device) -> torch.Tensor:
    """Stream-ordered shared fp32 scratch (grown on demand, never shrunk)."""
    key = (device.index if device.index is not None else torch.cuda.current_device())
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nfloats:
        ws = torch.empty(max(int(nfloats), 1 << 22), dtype=torch.float32, device=device)
        _workspaces[key] = ws
    return ws


# ------------------------------------------------------------------------------------------------------------
# GEMM / conv
# ------------------------------------------------------------------------------------------------------------
EPI_STORE, EPI_GEGLU = 0, 1

_gemm_scratch = {}
GEMM_SCRATCH_BYTES = 24 << 20          # fp32 K slices of tail tiles (csrc/gemm.cu: tail split); 148 x 128 x 256 x 4 B fits


def _ensure_gemm_scratch(device):
    """Hand the library its caller-owned scratch once per device (one device per process: the pointer is process-global)."""
    key = device.index if device.index is not None else torch.cuda.current_device()
    if key not in _gemm_scratch:
        if _gemm_scratch:
            raise _lib.AozoraError("aozora-b200 drives one GPU per process (launch one process per GPU)")
        buf = torch.empty(GEMM_SCRATCH_BYTES, dtype=torch.uint8, device=device)
        _lib.call("aoz_gemm_set_scratch", buf.data_ptr(), buf.numel())
        _gemm_scratch[key] = buf


def gemm(a, b, *, a_mn=False, b_mn=False, bias=None, residual=None, rowgroup_bias=None, rows_per_group=0,
         epi=EPI_STORE, aux=None, out=None, accumulate=False, splits=None):
    """C[M,N] = A·Bᵀ with fused epilogue.

    a: [M,K] (a_mn=False) or [K,M] (a_mn=True); b: [N,K] (b_mn=False) or [K,N] (b_mn=True); bf16, row-major
    (a leading dimension larger than the row length is allowed via 2-D strided views)."""
    _chk(a, "gemm a", contiguous=False)
    _chk(b, "gemm b", contiguous=False)
    if a.dim() != 2 or b.dim() != 2 or a.stride(1) != 1 or b.stride(1) != 1:
        raise _lib.AozoraError("gemm: operands must be 2-D with unit inner stride")
    (M, K) = (a.shape[1], a.shape[0]) if a_mn else (a.shape[0], a.shape[1])
    (N, Kb) = (b.shape[1], b.shape[0]) if b_mn else (b.shape[0], b.shape[1])
    if K != Kb:
        raise _lib.AozoraError(f"gemm: K mismatch {K} vs {Kb}")
    n_out = N // 2 if epi == EPI_GEGLU else N
    _ensure_gemm_scratch(a.device)
    if out is None:
        out = torch.empty((M, n_out), dtype=BF16, device=a.device)
    _chk(out, "gemm out", contiguous=False)
    if splits is None:
        fused = bias is not None or residual is not None or rowgroup_bias is not None or epi != EPI_STORE or accumulate
        splits = 1 if fused else _lib.query("aoz_gemm_auto_splits", M, N, K, int(b_mn))     # host cost model (gemm.cu)
    ws = None
    if splits > 1:
        ws = workspace(splits * M * N, a.device)
    if trace is not None:
        trace.append(("gemm", M, N, K, int(a_mn), int(b_mn), int(epi), int(splits), 2.0 * M * N * K))
    _lib.call("aoz_gemm_bf16", a.data_ptr(), a.stride(0), int(a_mn), b.data_ptr(), b.stride(0), int(b_mn),
              out.data_ptr(), out.stride(0), M, N, K, _p(bias), _p(rowgroup_bias), int(rows_per_group),
              0 if rowgroup_bias is None else rowgroup_bias.stride(0), _p(residual),
              0 if residual is None else residual.stride(0), epi, _p(aux), 0 if aux is None else aux.stride(0),
              int(accumulate), int(splits), _p(ws), _stream())
    _count(2 if splits > 1 else 1)
    return out


MAX_GROUPED = 10


def gemm_grouped(problems, *, a_mn, b_mn):
    """One persistent launch for up to 10 GEMMs that share K and the operand majors (plain bf16 store, no epilogue fusion):
    ``problems`` = [(a, b, out_or_None), ...] with the operand conventions of :func:`gemm`.  Returns the outputs."""
    import ctypes
    n = len(problems)
    if n == 0:
        return []
    if n > MAX_GROUPED:
        return gemm_grouped(problems[:MAX_GROUPED], a_mn=a_mn, b_mn=b_mn) + gemm_grouped(problems[MAX_GROUPED:], a_mn=a_mn, b_mn=b_mn)
    Ks, Ms, Ns, outs = set(), [], [], []
    for a, b, out in problems:
        _chk(a, "gemm_grouped a", contiguous=False)
        _chk(b, "gemm_grouped b", contiguous=False)
        if a.dim() != 2 or b.dim() != 2 or a.stride(1) != 1 or b.stride(1) != 1:
            raise _lib.AozoraError("gemm_grouped: operands must be 2-D with unit inner stride")
        (M, K) = (a.shape[1], a.shape[0]) if a_mn else (a.shape[0], a.shape[1])
        (N, Kb) = (b.shape[1], b.shape[0]) if b_mn else (b.shape[0], b.shape[1])
        if K != Kb:
            raise _lib.AozoraError(f"gemm_grouped: K mismatch {K} vs {Kb}")
        Ks.add(K)
        if out is None:
            out = torch.empty((M, N), dtype=BF16, device=a.device)
        _chk(out, "gemm_grouped out", contiguous=False)
        Ms.append(M)
        Ns.append(N)
        outs.append(out)
    if len(Ks) != 1:
        raise _lib.AozoraError(f"gemm_grouped: all problems must share K (got {sorted(Ks)})")
    _ensure_gemm_scratch(problems[0][0].device)
    u64, i64, i32 = ctypes.c_uint64 * n, ctypes.c_longlong * n, ctypes.c_int * n
    ap, bp, cp = u64(*[p[0].data_ptr() for p in problems]), u64(*[p[1].data_ptr() for p in problems]), u64(*[o.data_ptr() for o in outs])
    la, lb, lc = i64(*[p[0].stride(0) for p in problems]), i64(*[p[1].stride(0) for p in problems]), i64(*[o.stride(0) for o in outs])
    ms, ns = i32(*Ms), i32(*Ns)
    K = Ks.pop()
    if trace is not None:
        trace.append(("grouped", sum(Ms), max(Ns), K, int(a_mn), int(b_mn), 0, 1, 2.0 * K * sum(m * nn for m, nn in zip(Ms, Ns))))
    _lib.call("aoz_gemm_grouped_bf16", n, ctypes.addressof(ap), ctypes.addressof(la), ctypes.addressof(bp), ctypes.addressof(lb),
              ctypes.addressof(cp), ctypes.addressof(lc), ctypes.addressof(ms), ctypes.addressof(ns), K, int(a_mn), int(b_mn), _stream())
    _count()
    return outs


def pack_conv_weight(w, need_dgrad=True):
    """OIHW bf16 -> (wf [Cout, taps*CinPad], wd [Cin, taps*CoutPad]) with channel pads to multiples of 64."""
    _chk(w, "pack_conv_weight w")
    Cout, Cin, ks, _ = w.shape
    taps = ks * ks
    cin_pad = (Cin + 63) // 64 * 64
    cout_pad = (Cout + 63) // 64 * 64
    wf = torch.empty((Cout, taps * cin_pad), dtype=BF16, device=w.device)
    wd = torch.empty((Cin, taps * cout_pad), dtype=BF16, device=w.device) if need_dgrad else None
    _lib.call("aoz_pack_conv_weight", w.data_ptr(), Cout, Cin, ks, cin_pad, cout_pad, wf.data_ptr(), _p(wd), _stream())
    _count()
    return wf, wd


def conv_fwd(x, wpack, cout, ks, *, stride=1, pad=1, flip=False, bias=None, rowgroup_bias=None, residual=None, out=None):
    """x: [NB, Hin, Win, Cin] bf16 NHWC; wpack from pack_conv_weight; returns [NB, H, W, cout]."""
    _chk(x, "conv_fwd x")
    NB, Hin, Win, Cin = x.shape
    H = (Hin + 2 * pad - ks) // stride + 1
    W = (Win + 2 * pad - ks) // stride + 1
    _ensure_gemm_scratch(x.device)
    if out is None:
        out = torch.empty((NB, H, W, cout), dtype=BF16, device=x.device)
    if trace is not None:
        trace.append(("conv_dgrad" if flip else "conv_fwd", NB * H * W, cout, ks * ks * Cin, 0, 0, 0, 1, 2.0 * NB * H * W * cout * ks * ks * Cin))
    _lib.call("aoz_conv_fwd_bf16", x.data_ptr(), NB, Hin, Win, Cin, wpack.data_ptr(), cout, ks, stride, pad, int(flip),
              out.data_ptr(), _p(bias), _p(rowgroup_bias), _p(residual), 0, _stream())
    _count()
    return out


def conv_wgrad(dy, x, ks, *, stride=1, pad=1, grad_w=None, accumulate=False, cin_real=None, splits=None):
    """dW (OIHW bf16 [Cout, Cin, ks, ks]) from dy [NB,H,W,Cout] and x [NB,Hin,Win,Cin]."""
    _chk(dy, "conv_wgrad dy")
    _chk(x, "conv_wgrad x")
    NB, H, W, Cout = dy.shape
    _, Hin, Win, Cin = x.shape
    taps = ks * ks
    cin_real = cin_real or Cin
    if grad_w is None:
        grad_w = torch.empty((Cout, cin_real, ks, ks), dtype=BF16, device=x.device)
    if splits is None:
        splits = _lib.query("aoz_conv_wgrad_auto_splits", NB, H, W, Cout, Cin, ks)      # host cost model (gemm.cu)
    ws = workspace(splits * Cout * taps * Cin, x.device)
    if trace is not None:
        trace.append(("conv_wgrad", Cout, taps * Cin, NB * H * W, 1, 1, 0, int(splits), 2.0 * NB * H * W * Cout * taps * Cin))
    _lib.call("aoz_conv_wgrad_bf16", dy.data_ptr(), x.data_ptr(), NB, H, W, Cout, Hin, Win, Cin, ks, stride, pad, cin_real,
              grad_w.data_ptr(), int(accumulate), splits, ws.data_ptr(), _stream())
    _count(2)
    return grad_w


# ------------------------------------------------------------------------------------------------------------
# attention
# ------------------------------------------------------------------------------------------------------------
def attn_fwd(q, k, v, scale):
    """q: [B,Tq,H,64], k/v: [B,Tk,H,64] (views with row stride allowed: last two dims dense). -> (o, lse)."""
    B, Tq, H, D = q.shape
    Tk = k.shape[1]
    assert D == 64
    o = torch.empty((B, Tq, H, D), dtype=BF16, device=q.device)
    lse = torch.empty((B, H, Tq), dtype=torch.float32, device=q.device)
    _lib.call("aoz_attn_fwd", q.data_ptr(), q.stride(1), k.data_ptr(), k.stride(1), v.data_ptr(), v.stride(1),
              o.data_ptr(), o.stride(1), lse.data_ptr(), B, H, Tq, Tk, float(scale), _stream())
    _count(1)
    return o, lse


def attn_bwd(q, k, v, o, do, lse, scale, out=None):
    """-> (dq, dk, dv).  ``out``: optional (dq, dk, dv) destination views [B,T,H,64] with a row stride (e.g. the three
    column blocks of one fused [B*T, 3C] buffer, so the projection dgrad / wgrad run as single GEMMs)."""
    B, Tq, H, D = q.shape
    Tk = k.shape[1]
    if out is not None:
        dq, dk, dv = out
    else:
        dq = torch.empty((B, Tq, H, D), dtype=BF16, device=q.device)
        dk = torch.empty((B, Tk, H, D), dtype=BF16, device=q.device)
        dv = torch.empty((B, Tk, H, D), dtype=BF16, device=q.device)
    ws = workspace(_lib.query("aoz_attn_bwd_workspace_floats", B, H, Tq), q.device)
    _lib.call("aoz_attn_bwd", q.data_ptr(), q.stride(1), k.data_ptr(), k.stride(1), v.data_ptr(), v.stride(1),
              o.data_ptr(), o.stride(1), do.data_ptr(), do.stride(1), lse.data_ptr(), dq.data_ptr(), dq.stride(1),
              dk.data_ptr(), dk.stride(1), dv.data_ptr(), dv.stride(1), B, H, Tq, Tk, float(scale), ws.data_ptr(), _stream())
    _count(3)
    return dq, dk, dv


# ------------------------------------------------------------------------------------------------------------
# norms
# ------------------------------------------------------------------------------------------------------------
def groupnorm_fwd(x, gamma, beta, eps, silu):
    """x: [NB, HW, C] (or [NB,H,W,C]) bf16 -> (y, mean[NB,32], rstd[NB,32])."""
    _chk(x, "groupnorm x")
    NB, C = x.shape[0], x.shape[-1]
    HW = x.numel() // (NB * C)
    y = torch.empty_like(x)
    mean = torch.empty((NB, 32), dtype=torch.float32, device=x.device)
    rstd = torch.empty((NB, 32), dtype=torch.float32, device=x.device)
    ws = workspace(_lib.query("aoz_groupnorm_workspace_floats", NB, HW, C), x.device)
    _lib.call("aoz_groupnorm_fwd", x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), NB, HW, C, float(eps), int(silu),
              y.data_ptr(), mean.data_ptr(), rstd.data_ptr(), ws.data_ptr(), _stream())
    _count(2)
    return y, mean, rstd


def groupnorm_bwd(dy, x, gamma, beta, mean, rstd, silu, need_param_grads=True, dres=None, dgamma=None, dbeta=None):
    """``dgamma`` / ``dbeta``: optional destinations (e.g. slices of a flat gradient buffer)."""
    _chk(dy, "groupnorm dy")
    NB, C = x.shape[0], x.shape[-1]
    HW = x.numel() // (NB * C)
    dx = torch.empty_like(x)
    if need_param_grads:
        dgamma = torch.empty_like(gamma) if dgamma is None else dgamma
        dbeta = torch.empty_like(beta) if dbeta is None else dbeta
    else:
        dgamma = dbeta = None
    ws = workspace(_lib.query("aoz_groupnorm_workspace_floats", NB, HW, C), x.device)
    _lib.call("aoz_groupnorm_bwd", dy.data_ptr(), x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), mean.data_ptr(),
              rstd.data_ptr(), NB, HW, C, int(silu), _p(dres), dx.data_ptr(), _p(dgamma), _p(dbeta), 0, ws.data_ptr(), _stream())
    _count(3)
    return dx, dgamma, dbeta


def layernorm_fwd(x, gamma, beta, eps=1e-5):
    _chk(x, "layernorm x")
    C = x.shape[-1]
    rows = x.numel() // C
    y = torch.empty_like(x)
    mean = torch.empty((rows,), dtype=torch.float32, device=x.device)
    rstd = torch.empty((rows,), dtype=torch.float32, device=x.device)
    _lib.call("aoz_layernorm_fwd", x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), rows, C, float(eps), y.data_ptr(),
              mean.data_ptr(), rstd.data_ptr(), _stream())
    _count()
    return y, mean, rstd


def layernorm_bwd(dy, x, gamma, mean, rstd, dres=None, dgamma=None, dbeta=None, dx_colsum=None):
    """``dgamma`` / ``dbeta``: optional destinations (e.g. slices of a flat gradient buffer).  ``dx_colsum``: a bf16 [C] destination
    for the column sums of dx (the bias gradient of the Linear that produced this LayerNorm's input), formed in the same pass."""
    _chk(dy, "layernorm dy")
    C = x.shape[-1]
    rows = x.numel() // C
    dx = torch.empty_like(x)
    dgamma = torch.empty_like(gamma) if dgamma is None else dgamma
    dbeta = torch.empty_like(gamma) if dbeta is None else dbeta
    ws = workspace(_lib.query("aoz_layernorm_bwd_workspace_floats", C), x.device)
    _lib.call("aoz_layernorm_bwd_colsum", dy.data_ptr(), x.data_ptr(), gamma.data_ptr(), mean.data_ptr(), rstd.data_ptr(), rows, C,
              _p(dres), dx.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), 0, _p(dx_colsum), ws.data_ptr(), _stream())
    _count(2)
    return dx, dgamma, dbeta


# ------------------------------------------------------------------------------------------------------------
# glue
# ------------------------------------------------------------------------------------------------------------
def nchw_to_nhwc(src, cpad=None):
    NB, C = src.shape[0], src.shape[1]
    HW = src.numel() // (NB * C)
    cpad = cpad or C
    _chk(src, "nchw_to_nhwc src", dtype=None)
    dst = torch.empty((NB,) + tuple(src.shape[2:]) + (cpad,), dtype=BF16, device=src.device)
    _lib.call("aoz_nchw_to_nhwc", src.data_ptr(), int(src.dtype == torch.float32), NB, C, HW, cpad, dst.data_ptr(), _stream())
    _count()
    return dst


def nhwc_to_nchw(src, c=None, out_dtype=BF16):
    _chk(src, "nhwc_to_nchw src")
    NB, ld = src.shape[0], src.shape[-1]
    c = c or ld
    HW = src.numel() // (NB * ld)
    dst = torch.empty((NB, c) + tuple(src.shape[1:-1]), dtype=out_dtype, device=src.device)
    _lib.call("aoz_nhwc_to_nchw", src.data_ptr(), NB, c, HW, ld, dst.data_ptr(), int(out_dtype == torch.float32), _stream())
    _count()
    return dst


MODE = {"epsilon": 0, "v_prediction": 1, "rectified_flow": 2}


def noise_target(latents, noise, tickets, alphas_cumprod, jitter, prediction_type, cpad=8):
    """train.py:2743-2758.  latents bf16 NCHW, noise fp32 NCHW, tickets int64[B] ->
    (xt NHWC bf16 [B,h,w,cpad], target fp32 NCHW, cond fp32 [B])."""
    _chk(latents, "noise_target latents")
    _chk(noise, "noise_target noise", dtype=torch.float32)
    _chk(tickets, "noise_target tickets", dtype=torch.int64)
    B, C, H, W = latents.shape
    xt = torch.empty((B, H, W, cpad), dtype=BF16, device=latents.device)
    target = torch.empty((B, C, H, W), dtype=torch.float32, device=latents.device)
    cond = torch.empty((B,), dtype=torch.float32, device=latents.device)
    _lib.call("aoz_noise_target", latents.data_ptr(), noise.data_ptr(), tickets.data_ptr(), _p(alphas_cumprod), _p(jitter),
              MODE[prediction_type], B, C, H * W, cpad, xt.data_ptr(), target.data_ptr(), cond.data_ptr(), _stream())
    _count()
    return xt, target, cond


def _strides3(t, nhwc, c):
    """(sample, channel, pixel) element strides of a [B,h,w,ld] (nhwc) or [B,C,h,w] (nchw) contiguous tensor."""
    if nhwc:
        ld = t.shape[-1]
        hw = t.numel() // (t.shape[0] * ld)
        return hw * ld, 1, ld
    hw = t.numel() // (t.shape[0] * c)
    return c * hw, hw, 1


def mse_loss(pred, target_nchw, tickets, table, denom, grad_scale=1.0, *, pred_nhwc=True, need_grad=True, dpred_ld=None,
             grad_scale_tensor=None):
    """weighted_sdxl_mse_loss (train.py:2408-2416) and dL/dpred in one pass.

    pred: bf16 [B,h,w,ld] (pred_nhwc) or [B,C,h,w]; target fp32 NCHW.  Returns (loss[1] fp32, per_sample[B], dpred|None);
    dpred has the layout of pred, with the last dim padded to ``dpred_ld`` channels (zeros) when given (NHWC only)."""
    _chk(pred, "mse_loss pred")
    _chk(target_nchw, "mse_loss target", dtype=torch.float32)
    B, C = target_nchw.shape[0], target_nchw.shape[1]
    HW = target_nchw.numel() // (B * C)
    dev = pred.device
    per = torch.empty((B,), dtype=torch.float32, device=dev)
    w = torch.empty((B,), dtype=torch.float32, device=dev)
    loss = torch.empty((1,), dtype=torch.float32, device=dev)
    dpred = None
    ds = (0, 0, 0)
    if need_grad:
        if pred_nhwc and dpred_ld and dpred_ld != pred.shape[-1]:
            dpred = torch.zeros(tuple(pred.shape[:-1]) + (dpred_ld,), dtype=BF16, device=dev)
        else:
            dpred = torch.zeros_like(pred) if (pred_nhwc and pred.shape[-1] != C) else torch.empty_like(pred)
        ds = _strides3(dpred, pred_nhwc, C)
    ps = _strides3(pred, pred_nhwc, C)
    _lib.call("aoz_mse_loss", pred.data_ptr(), ps[0], ps[1], ps[2], target_nchw.data_ptr(), _p(tickets), _p(table),
              0 if table is None else table.numel(), B, C, HW, float(denom), _p(grad_scale_tensor), float(grad_scale),
              per.data_ptr(), w.data_ptr(), loss.data_ptr(), _p(dpred), ds[0], ds[1], ds[2], _stream())
    _count(2)
    return loss, per, dpred


def geglu_bwd(dy, aux):
    """GEGLU backward: dy [.., half] and the saved pre-activation aux [.., 2 * half] -> daux [.., 2 * half]."""
    _chk(dy, "geglu_bwd dy")
    _chk(aux, "geglu_bwd aux")
    half = dy.shape[-1]
    M = dy.numel() // half
    daux = torch.empty_like(aux)
    _lib.call("aoz_geglu_bwd", dy.data_ptr(), aux.data_ptr(), M, half, daux.data_ptr(), _stream())
    _count()
    return daux


def silu_fwd(x):
    _chk(x, "silu x")
    y = torch.empty_like(x)
    _lib.call("aoz_silu_fwd", x.data_ptr(), x.numel(), y.data_ptr(), _stream())
    _count()
    return y


def silu_bwd(dy, x):
    _chk(dy, "silu dy")
    dx = torch.empty_like(x)
    _lib.call("aoz_silu_bwd", dy.data_ptr(), x.data_ptr(), x.numel(), dx.data_ptr(), _stream())
    _count()
    return dx


def add(a, b, out=None):
    _chk(a, "add a")
    _chk(b, "add b")
    if out is None:
        out = torch.empty_like(a)
    _lib.call("aoz_add", a.data_ptr(), b.data_ptr(), a.numel(), out.data_ptr(), _stream())
    _count()
    return out


def grad_accum_mt(ys, as_, bs, plan, stage, copy=False):
    """``ys[t] = bs[t]`` (``copy``) or ``as_[t] + bs[t]`` for every t, bf16, in ONE launch; each tensor is bit-identical to
    ``add``.  ``ys`` may alias ``as_`` or ``bs``.  ``plan`` is the caller's ``MultiTensorPlan`` and ``stage`` its ``_Staging``
    (optimizers/raven.py): the pointer tables go through ``stage``, so a call under CUDA-graph capture bakes its own tables in."""
    n = len(ys)
    if n == 0 or len(bs) != n or (not copy and len(as_) != n):
        raise _lib.AozoraError("grad_accum_mt: need the same, non-zero number of tensors in every list")
    for i in range(n):
        for t, name in ((ys[i], "grad_accum_mt y"), (bs[i], "grad_accum_mt b")) + (() if copy else ((as_[i], "grad_accum_mt a"),)):
            _chk(t, name)
            if t.numel() != ys[i].numel():
                raise _lib.AozoraError(f"{name}: tensor {i} has {t.numel()} elements, y has {ys[i].numel()}")
    dev = ys[0].device
    plan.ensure([y.numel() for y in ys], dev)

    def table(name, ts):
        return stage.put(name, np.fromiter((t.data_ptr() for t in ts), dtype=np.uint64, count=n).view(np.int64), dev).data_ptr()

    yp, bp = table("acc_y", ys), table("acc_b", bs)
    ap = 0 if copy else table("acc_a", as_)
    _lib.call("aoz_grad_accum_mt", plan.n_tensors, plan.n_chunks, ap, bp, yp, plan.numel.data_ptr(), plan.chunk_start.data_ptr(),
              plan.chunk_tensor.data_ptr(), int(bool(copy)), _stream())
    _count()


def upsample2x_fwd(x):
    _chk(x, "upsample x")
    NB, H, W, C = x.shape
    y = torch.empty((NB, 2 * H, 2 * W, C), dtype=BF16, device=x.device)
    _lib.call("aoz_upsample2x_fwd", x.data_ptr(), NB, H, W, C, y.data_ptr(), _stream())
    _count()
    return y


def upsample2x_bwd(dy):
    _chk(dy, "upsample dy")
    NB, H2, W2, C = dy.shape
    dx = torch.empty((NB, H2 // 2, W2 // 2, C), dtype=BF16, device=dy.device)
    _lib.call("aoz_upsample2x_bwd", dy.data_ptr(), NB, H2 // 2, W2 // 2, C, dx.data_ptr(), _stream())
    _count()
    return dx


def zero_insert2x(x, hout, wout):
    """y[n, 2h, 2w, :] = x[n, h, w, :], zeros elsewhere (adjoint helper of the stride-2 convolution)."""
    _chk(x, "zero_insert x")
    NB, H, W, C = x.shape
    y = torch.empty((NB, hout, wout, C), dtype=BF16, device=x.device)
    _lib.call("aoz_zero_insert2x", x.data_ptr(), NB, H, W, C, hout, wout, y.data_ptr(), _stream())
    _count()
    return y


def copy_channels(src, src_off, dst, dst_off, ch, accumulate=False):
    """dst[..., dst_off:dst_off+ch] (+)= src[..., src_off:src_off+ch] over all rows (channels-last)."""
    rows = src.numel() // src.shape[-1]
    _lib.call("aoz_copy_channels", src.data_ptr(), src.shape[-1], src_off, dst.data_ptr(), dst.shape[-1], dst_off, rows, ch,
              int(accumulate), _stream())
    _count()
    return dst


def concat_channels(a, b):
    _chk(a, "concat a")
    _chk(b, "concat b")
    out = torch.empty(tuple(a.shape[:-1]) + (a.shape[-1] + b.shape[-1],), dtype=BF16, device=a.device)
    copy_channels(a, 0, out, 0, a.shape[-1])
    copy_channels(b, 0, out, a.shape[-1], b.shape[-1])
    return out


def colsum(x2d, out=None, accumulate=False):
    """out[c] = sum_r x[r, c]; x: [M, N] bf16 (row stride allowed)."""
    _chk(x2d, "colsum x", contiguous=False)
    M, N = x2d.shape
    if out is None:
        out = torch.empty((N,), dtype=BF16, device=x2d.device)
    ws = workspace(_lib.query("aoz_colsum_workspace_floats", 1, N), x2d.device)
    _lib.call("aoz_colsum", x2d.data_ptr(), 1, M, N, x2d.stride(0), 0, out.data_ptr(), int(accumulate), ws.data_ptr(), _stream())
    _count(2)
    return out


def colsum_grouped(x3d):
    """out[g, c] = sum_r x[g, r, c]; x: [G, M, N] contiguous bf16 -> [G, N] (per-image sums: time-embedding gradient)."""
    _chk(x3d, "colsum_grouped x")
    G, N = x3d.shape[0], x3d.shape[-1]
    M = x3d.numel() // (G * N)
    out = torch.empty((G, N), dtype=BF16, device=x3d.device)
    ws = workspace(_lib.query("aoz_colsum_workspace_floats", G, N), x3d.device)
    _lib.call("aoz_colsum", x3d.data_ptr(), G, M, N, N, M * N, out.data_ptr(), 0, ws.data_ptr(), _stream())
    _count(2)
    return out


def timestep_embedding(t, dim):
    """diffusers Timesteps(dim, flip_sin_to_cos=True, downscale_freq_shift=0): t fp32 [n] -> bf16 [n, dim]."""
    _chk(t, "timestep_embedding t", dtype=torch.float32)
    out = torch.empty((t.numel(), dim), dtype=BF16, device=t.device)
    _lib.call("aoz_timestep_embedding", t.data_ptr(), t.numel(), dim, out.data_ptr(), _stream())
    _count()
    return out
