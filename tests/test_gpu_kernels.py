"""GPU parity tests of every kernel family, called through the C ABI (ops -> ctypes -> libaozora_b200.so).

Floating-point kernels are compared with plain PyTorch fp32 references of the same op (tolerances stated per test);
the Raven update is compared with the CPU oracle (oracle/host_ref.py, pinned to the reference's own trajectories)."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16
# bf16 stores round at 2^-9 relative: rms relative error of a correctly rounded result is ~1.7e-3
REL_TOL = 4e-3
COS_TOL = 0.9999


def _ops():
    from aozora_sdxl_training_b200 import ops
    return ops


def check(got, ref, rel=REL_TOL, cos=COS_TOL):
    got, ref = got.float().flatten(), ref.float().flatten()
    assert not torch.isnan(got).any()
    r = ((got - ref).norm() / (ref.norm() + 1e-30)).item()
    c = torch.nn.functional.cosine_similarity(got, ref, dim=0).item()
    assert r <= rel and c >= cos, (r, c)


def gen(seed=0):
    return torch.Generator(device="cuda").manual_seed(seed)


@pytest.mark.parametrize("a_mn,b_mn,M,N,K", [
    (False, False, 128, 128, 64), (False, False, 1000, 640, 320), (False, False, 4096, 1280, 1280),
    (False, False, 4, 1280, 320), (True, False, 256, 256, 256), (False, True, 1000, 320, 640),
    (True, True, 640, 320, 1000), (False, False, 308, 1280, 2048), (True, True, 1280, 2048, 308),
])
def test_gemm_all_operand_majors(a_mn, b_mn, M, N, K):
    ops = _ops()
    g = gen(1)
    A = torch.randn((K, M) if a_mn else (M, K), device="cuda", generator=g).to(BF16)
    B = torch.randn((K, N) if b_mn else (N, K), device="cuda", generator=g).to(BF16)
    out = ops.gemm(A, B, a_mn=a_mn, b_mn=b_mn)
    ref = (A.float().t() if a_mn else A.float()) @ (B.float() if b_mn else B.float().t())
    check(out, ref)


def test_gemm_epilogues_bias_residual_rowgroup_splitk_accumulate():
    ops = _ops()
    g = gen(2)
    M, N, K = 512, 384, 256
    A = torch.randn(M, K, device="cuda", generator=g).to(BF16)
    B = torch.randn(N, K, device="cuda", generator=g).to(BF16)
    bias = torch.randn(N, device="cuda", generator=g).to(BF16)
    res = torch.randn(M, N, device="cuda", generator=g).to(BF16)
    rgb = torch.randn(4, N, device="cuda", generator=g).to(BF16)
    base = A.float() @ B.float().t()
    check(ops.gemm(A, B, bias=bias, residual=res), (base + bias.float()).to(BF16).float() + res.float())
    ref = (base + bias.float()).to(BF16).float() + rgb.float().repeat_interleave(128, dim=0)
    check(ops.gemm(A, B, bias=bias, rowgroup_bias=rgb, rows_per_group=128), ref)
    check(ops.gemm(A, B, splits=4), base)
    acc = res.clone()
    ops.gemm(A, B, out=acc, accumulate=True, splits=1)
    check(acc, base.to(BF16).float() + res.float())


@pytest.mark.parametrize("pair_mode", [0, 2])
@pytest.mark.parametrize("M,N,K,b_mn", [(4096, 1280, 1280, False), (4096, 1280, 5120, False), (4096, 1280, 10240, True),
                                         (308, 2560, 2048, False), (1000, 640, 320, False), (16384, 640, 640, True)])
def test_gemm_tail_split_matches_plain_tiles(pair_mode, M, N, K, b_mn):
    """The last, partly filled wave cut along K (fp32 slices + fix-up kernel with the fused epilogue) must give the same
    result as whole tiles; forced on (tail mode 2) so every shape exercises it, with bias + residual in the fix-up."""
    from aozora_sdxl_training_b200 import _lib
    ops = _ops()
    g = gen(11)
    A = torch.randn(M, K, device="cuda", generator=g).to(BF16)
    B = (torch.randn((K, N) if b_mn else (N, K), device="cuda", generator=g) * 0.05).to(BF16)
    bias = torch.randn(N, device="cuda", generator=g).to(BF16)
    res = torch.randn(M, N, device="cuda", generator=g).to(BF16)
    ref = ((A.float() @ (B.float() if b_mn else B.float().t())) + bias.float()).to(BF16).float() + res.float()
    try:
        _lib.call("aoz_gemm_set_pair_mode", pair_mode)
        outs = []
        for tail in (0, 2):
            _lib.call("aoz_gemm_set_tail_mode", tail)
            l0 = _lib.query("aoz_launch_count")
            outs.append(ops.gemm(A, B, b_mn=b_mn, bias=bias, residual=res, splits=1))
            launches = _lib.query("aoz_launch_count") - l0
            check(outs[-1], ref)
        assert launches == 2 or M * N <= 128 * 64          # GEMM + fix-up: the forced mode really took the tail path
        check(outs[1], outs[0].float(), rel=2e-3)
    finally:
        _lib.call("aoz_gemm_set_pair_mode", 1)
        _lib.call("aoz_gemm_set_tail_mode", 1)


@pytest.mark.parametrize("pair_mode,tail_mode", [(0, 0), (2, 0), (1, 1), (0, 2), (2, 2)])
def test_grouped_weight_gradient_gemm(pair_mode, tail_mode):
    """One persistent launch for several dW = dy^T x problems sharing the token count (a transformer block's weight
    gradients); every problem must match its own plain fp32 reference, for every tile / tail configuration."""
    from aozora_sdxl_training_b200 import _lib
    ops = _ops()
    g = gen(13)
    T = 1000                                                   # tokens: not a multiple of the 64-row K step
    shapes = [(768, 256), (256, 256), (256, 256), (2048, 256), (256, 1024), (200, 136)]      # (out features, in features)
    probs, refs = [], []
    for of, inf in shapes:
        dy = torch.randn(T, of, device="cuda", generator=g).to(BF16)
        x = torch.randn(T, inf, device="cuda", generator=g).to(BF16)
        probs.append((dy, x, None))
        refs.append(dy.float().t() @ x.float())
    try:
        _lib.call("aoz_gemm_set_pair_mode", pair_mode)
        _lib.call("aoz_gemm_set_tail_mode", tail_mode)
        l0 = _lib.query("aoz_launch_count")
        outs = ops.gemm_grouped(probs, a_mn=True, b_mn=True)
        assert _lib.query("aoz_launch_count") - l0 <= 2          # one GEMM (+ at most the tail fix-up)
        for o, r in zip(outs, refs):
            check(o, r)
        # strided output views (row blocks of a stacked gradient) and > 8 problems (split into two launches)
        big = torch.zeros(1024, 256, device="cuda", dtype=BF16)
        more = [(probs[1][0], probs[1][1], big[i * 256:(i + 1) * 256]) for i in range(4)] + probs[:5]
        outs = ops.gemm_grouped(more, a_mn=True, b_mn=True)
        for i in range(4):
            check(big[i * 256:(i + 1) * 256], refs[1])
        for o, r in zip(outs[4:], refs[:5]):
            check(o, r)
    finally:
        _lib.call("aoz_gemm_set_pair_mode", 1)
        _lib.call("aoz_gemm_set_tail_mode", 1)


def test_conv_tail_split_with_time_embedding_and_residual():
    from aozora_sdxl_training_b200 import _lib
    ops = _ops()
    g = gen(12)
    NB, H, W, Cin, Cout = 4, 32, 32, 256, 320
    x = torch.randn(NB, H, W, Cin, device="cuda", generator=g).to(BF16)
    w = (torch.randn(Cout, Cin, 3, 3, device="cuda", generator=g) * 0.05).to(BF16)
    b = torch.randn(Cout, device="cuda", generator=g).to(BF16)
    temb = torch.randn(NB, Cout, device="cuda", generator=g).to(BF16)
    res = torch.randn(NB, H, W, Cout, device="cuda", generator=g).to(BF16)
    wf, _ = ops.pack_conv_weight(w, need_dgrad=False)
    conv = torch.nn.functional.conv2d(x.float().permute(0, 3, 1, 2), w.float(), b.float(), padding=1).permute(0, 2, 3, 1)
    ref_t = conv.to(BF16).float() + temb.float()[:, None, None, :]
    ref_r = conv.to(BF16).float() + res.float()
    try:
        for pair in (0, 2):
            _lib.call("aoz_gemm_set_pair_mode", pair)
            for tail in (0, 2):
                _lib.call("aoz_gemm_set_tail_mode", tail)
                check(ops.conv_fwd(x, wf, Cout, 3, bias=b, rowgroup_bias=temb), ref_t)
                check(ops.conv_fwd(x, wf, Cout, 3, bias=b, residual=res), ref_r)
    finally:
        _lib.call("aoz_gemm_set_pair_mode", 1)
        _lib.call("aoz_gemm_set_tail_mode", 1)


def test_conv_wide_plan_equals_ordinary_tiles():
    """The 320-wide plan on the implicit-GEMM convolution (forward with bias + time embedding = general epilogue, bias + residual =
    fast epilogue, and the flipped dgrad pack): same K order per output element, so the bits equal the ordinary tiles', and both
    match the fp32 convolution."""
    from aozora_sdxl_training_b200 import _lib
    ops = _ops()
    g = gen(60)
    for NB, H, W, Cin, Cout in ((4, 32, 32, 256, 320), (2, 32, 32, 128, 640), (1, 18, 14, 320, 192), (4, 32, 32, 128, 1280)):
        x = torch.randn(NB, H, W, Cin, device="cuda", generator=g).to(BF16)
        w = (torch.randn(Cout, Cin, 3, 3, device="cuda", generator=g) * 0.05).to(BF16)
        b = torch.randn(Cout, device="cuda", generator=g).to(BF16)
        temb = torch.randn(NB, Cout, device="cuda", generator=g).to(BF16)
        res = torch.randn(NB, H, W, Cout, device="cuda", generator=g).to(BF16)
        dy = torch.randn(NB, H, W, Cout, device="cuda", generator=g).to(BF16)
        wf, wd = ops.pack_conv_weight(w)
        runs = {}
        for mode in (0, 2):
            try:
                _lib.call("aoz_gemm_set_wide_mode", mode)
                _lib.call("aoz_gemm_set_wide_max_rounds", 3)
                _lib.call("aoz_gemm_set_tail_mode", 0)
                runs[mode] = (ops.conv_fwd(x, wf, Cout, 3, bias=b, rowgroup_bias=temb), ops.conv_fwd(x, wf, Cout, 3, bias=b, residual=res),
                              ops.conv_fwd(dy, wd, Cin, 3, stride=1, pad=1, flip=True))
            finally:
                _lib.call("aoz_gemm_set_wide_mode", 1)
                _lib.call("aoz_gemm_set_wide_max_rounds", 2)
                _lib.call("aoz_gemm_set_tail_mode", 1)
        conv = torch.nn.functional.conv2d(x.float().permute(0, 3, 1, 2), w.float(), b.float(), padding=1).permute(0, 2, 3, 1)
        check(runs[2][0], conv.to(BF16).float() + temb.float()[:, None, None, :])
        check(runs[2][1], conv.to(BF16).float() + res.float())
        dx = torch.nn.functional.conv_transpose2d(dy.float().permute(0, 3, 1, 2), w.float(), padding=1).permute(0, 2, 3, 1)
        check(runs[2][2], dx)
        for got, ref in zip(runs[2], runs[0]):
            assert torch.equal(got, ref), (NB, H, W, Cin, Cout)


def test_conv_wgrad_wide_plan_equals_ordinary_tiles():
    """Weight gradients (both operands MN-major through 4-D TMA pixel tiles, fp32 partials + permuting reduce) on 320-wide tiles:
    the third 64-channel chunk of a CTA's x tile is half used and the second MMA reads half a swizzle atom; with and without split-K,
    stride 2, and an output-channel count that leaves the second CTA of the last pair partly empty."""
    from aozora_sdxl_training_b200 import _lib
    ops = _ops()
    g = gen(61)
    for NB, H, W, Cin, Cout, stride in ((1, 32, 32, 640, 320, 1), (2, 16, 16, 320, 256, 1), (1, 16, 16, 960, 640, 1), (2, 16, 16, 320, 640, 2)):
        x = torch.randn(NB, H, W, Cin, device="cuda", generator=g).to(BF16)
        Ho, Wo = H // stride, W // stride
        dy = torch.randn(NB, Ho, Wo, Cout, device="cuda", generator=g).to(BF16)
        runs = {}
        for mode in (0, 2):
            try:
                _lib.call("aoz_gemm_set_wide_mode", mode)
                runs[mode] = [ops.conv_wgrad(dy, x, 3, stride=stride, pad=1, splits=sp) for sp in (1, 2, None)]
            finally:
                _lib.call("aoz_gemm_set_wide_mode", 1)
        xr = x.float().permute(0, 3, 1, 2)
        wr = torch.zeros(Cout, Cin, 3, 3, device="cuda", requires_grad=True)
        torch.nn.functional.conv2d(xr, wr, None, stride=stride, padding=1).backward(dy.float().permute(0, 3, 1, 2))
        for got, ref in zip(runs[2], runs[0]):
            check(got, wr.grad)
            assert torch.equal(got, ref), (NB, H, W, Cin, Cout, stride)


@pytest.mark.parametrize("M,C", [(512, 128), (4096, 640), (300, 64)])
def test_geglu_fused_epilogue_and_backward(M, C):
    ops = _ops()
    g = gen(3)
    x = torch.randn(M, C, device="cuda", generator=g).to(BF16)
    w = (torch.randn(8 * C, C, device="cuda", generator=g) * 0.05).to(BF16)
    b = torch.randn(8 * C, device="cuda", generator=g).to(BF16)
    aux = torch.empty(M, 8 * C, device="cuda", dtype=BF16)
    out = ops.gemm(x, w, bias=b, epi=ops.EPI_GEGLU, aux=aux)
    proj = (x.float() @ w.float().t() + b.float()).to(BF16)
    check(aux, proj)
    h, gate = proj.float().chunk(2, dim=-1)
    check(out, h * torch.nn.functional.gelu(gate).to(BF16).float())
    dy = torch.randn(M, 4 * C, device="cuda", generator=g).to(BF16)
    pr = proj.float().requires_grad_(True)
    hh, gg = pr.chunk(2, dim=-1)
    (hh * torch.nn.functional.gelu(gg)).backward(dy.float())
    check(ops.geglu_bwd(dy, aux), pr.grad, rel=8e-3)


def test_gemm_wide_one_wave_plan_equals_two_round_plan():
    """The 320-wide one-wave plan (one 256 x 320 tile per CTA pair, two MMAs per K step into a single accumulator, permuted column
    chunks in the epilogue) against the ordinary plans: every output element is the same K-ordered fp32 sum, so the bits agree; both
    operand majors of B, with and without the fused bias / residual, accumulate, and a shape with fewer tiles than SM pairs."""
    from aozora_sdxl_training_b200 import _lib
    ops = _ops()
    g = gen(59)
    for M, N, K, b_mn in ((4096, 1280, 1280, False), (4096, 1280, 1280, True), (4096, 1280, 5120, False), (4096, 1280, 3840, True),
                          (512, 640, 320, False), (300, 320, 72, True), (4096, 1280, 10240, True),
                          (16384, 640, 640, False), (16384, 640, 640, True)):          # two and three tiles per CTA pair
        x = torch.randn(M, K, device="cuda", generator=g).to(BF16)
        w = ((torch.randn(K, N, device="cuda", generator=g) if b_mn else torch.randn(N, K, device="cuda", generator=g)) * 0.05).to(BF16)
        b = torch.randn(N, device="cuda", generator=g).to(BF16)
        res = torch.randn(M, N, device="cuda", generator=g).to(BF16)
        acc0 = torch.randn(M, N, device="cuda", generator=g).to(BF16)
        runs = {}
        for mode in (0, 2):
            try:
                _lib.call("aoz_gemm_set_wide_mode", mode)
                _lib.call("aoz_gemm_set_wide_max_rounds", 3)
                _lib.call("aoz_gemm_set_tail_mode", 0)              # a tail split sums K slices in another order: not the reference here
                plain = ops.gemm(x, w, b_mn=b_mn, splits=1)
                fused = ops.gemm(x, w, b_mn=b_mn, bias=b, residual=res)
                acc = acc0.clone()
                ops.gemm(x, w, b_mn=b_mn, out=acc, accumulate=True, splits=1)
            finally:
                _lib.call("aoz_gemm_set_wide_mode", 1)
                _lib.call("aoz_gemm_set_wide_max_rounds", 2)
                _lib.call("aoz_gemm_set_tail_mode", 1)
            runs[mode] = (plain, fused, acc)
        wf = w.float() if b_mn else w.float().t()
        check(runs[2][0], x.float() @ wf)
        check(runs[2][1], x.float() @ wf + b.float() + res.float())
        for got, ref in zip(runs[2], runs[0]):
            assert torch.equal(got, ref), (M, N, K, b_mn, (got.float() - ref.float()).abs().max().item())


def test_layernorm_backward_with_column_sums_of_dx():
    """ln_bwd_kernel's third accumulator: the column sums of the dx it stores (bf16-rounded) = the bias gradient of the Linear that
    produced the LayerNorm's input.  dx / dgamma / dbeta must not change; the sums must equal colsum(dx) up to fp32 summation order."""
    ops = _ops()
    g = gen(57)
    for rows, C, with_res in ((4096, 1280, True), (16384, 640, True), (1000, 320, False), (7, 64, True)):
        x = torch.randn(rows, C, device="cuda", generator=g).to(BF16)
        dy = torch.randn(rows, C, device="cuda", generator=g).to(BF16)
        dres = torch.randn(rows, C, device="cuda", generator=g).to(BF16) if with_res else None
        ga = (1 + 0.1 * torch.randn(C, device="cuda", generator=g)).to(BF16)
        be = torch.zeros(C, device="cuda", dtype=BF16)
        _, mean, rstd = ops.layernorm_fwd(x, ga, be)
        dx0, dg0, db0 = ops.layernorm_bwd(dy, x, ga, mean, rstd, dres=dres)
        col = torch.empty(C, device="cuda", dtype=BF16)
        dx1, dg1, db1 = ops.layernorm_bwd(dy, x, ga, mean, rstd, dres=dres, dx_colsum=col)
        assert torch.equal(dx0, dx1) and torch.equal(dg0, dg1) and torch.equal(db0, db1)
        want = dx1.float().sum(0)
        err = (col.float() - want).abs()
        assert bool((err <= 2 ** -7 * want.abs() + 2e-2).all()), float(err.max())


@pytest.mark.parametrize("NB,H,W,Cin,Cout,ks,stride", [
    (2, 16, 16, 64, 128, 3, 1), (1, 18, 14, 320, 192, 3, 1), (2, 16, 16, 64, 64, 3, 2), (1, 13, 19, 128, 64, 3, 2),
    (2, 16, 16, 128, 64, 1, 1), (2, 16, 16, 8, 320, 3, 1), (2, 16, 16, 320, 8, 3, 1), (1, 32, 32, 640, 320, 3, 1),
])
def test_conv_fwd_dgrad_wgrad(NB, H, W, Cin, Cout, ks, stride):
    ops = _ops()
    g = gen(4)
    pad = ks // 2
    x = torch.randn(NB, H, W, Cin, device="cuda", generator=g).to(BF16)
    w = (torch.randn(Cout, Cin, ks, ks, device="cuda", generator=g) * 0.05).to(BF16)
    b = torch.randn(Cout, device="cuda", generator=g).to(BF16)
    wf, wd = ops.pack_conv_weight(w)
    y = ops.conv_fwd(x, wf, Cout, ks, stride=stride, pad=pad, bias=b)
    xr = x.float().permute(0, 3, 1, 2).requires_grad_(True)
    wr = w.float().requires_grad_(True)
    yr = torch.nn.functional.conv2d(xr, wr, b.float(), stride=stride, padding=pad)
    check(y, yr.permute(0, 2, 3, 1))
    dy = torch.randn(y.shape, device="cuda", generator=g).to(BF16)
    yr.backward(dy.float().permute(0, 3, 1, 2))
    dyi = dy if stride == 1 else ops.zero_insert2x(dy, H, W)
    check(ops.conv_fwd(dyi, wd, Cin, ks, stride=1, pad=pad, flip=True), xr.grad.permute(0, 2, 3, 1))
    check(ops.conv_wgrad(dy, x, ks, stride=stride, pad=pad), wr.grad)


def test_conv_fused_time_embedding_and_residual():
    ops = _ops()
    g = gen(5)
    NB, H, W, C = 2, 16, 16, 128
    x = torch.randn(NB, H, W, C, device="cuda", generator=g).to(BF16)
    w = (torch.randn(C, C, 3, 3, device="cuda", generator=g) * 0.05).to(BF16)
    b = torch.randn(C, device="cuda", generator=g).to(BF16)
    temb = torch.randn(NB, C, device="cuda", generator=g).to(BF16)
    res = torch.randn(NB, H, W, C, device="cuda", generator=g).to(BF16)
    wf, _ = ops.pack_conv_weight(w, need_dgrad=False)
    conv = torch.nn.functional.conv2d(x.float().permute(0, 3, 1, 2), w.float(), b.float(), padding=1).permute(0, 2, 3, 1)
    check(ops.conv_fwd(x, wf, C, 3, bias=b, rowgroup_bias=temb), conv.to(BF16).float() + temb.float()[:, None, None, :])
    check(ops.conv_fwd(x, wf, C, 3, bias=b, residual=res), conv.to(BF16).float() + res.float())


@pytest.mark.parametrize("xs", [1.0, 1.5])
@pytest.mark.parametrize("B,H,Tq,Tk", [(1, 2, 128, 128), (2, 5, 1024, 1024), (2, 10, 1024, 1024), (1, 3, 1008, 1008), (2, 10, 1024, 77),
                                        (1, 5, 988, 154), (1, 2, 64, 64), (1, 1, 16, 77), (1, 10, 4096, 77), (2, 3, 200, 77),
                                        (1, 2, 300, 128), (1, 2, 300, 40)])
def test_attention_fwd_bwd(B, H, Tq, Tk, xs):
    """Forward and backward against fp32 SDPA.  With Q and K scaled by xs = 1.5 the scores are wide enough that in a few rows of the
    larger shapes a later key tile's P exceeds 2^8 against the running reference (never at 1.0), so the forward's exact-maximum
    rescale of O and the row sum runs as well."""
    ops = _ops()
    g = gen(6)
    q = (torch.randn(B, Tq, H, 64, device="cuda", generator=g) * xs).to(BF16)
    k = (torch.randn(B, Tk, H, 64, device="cuda", generator=g) * xs).to(BF16)
    v = torch.randn(B, Tk, H, 64, device="cuda", generator=g).to(BF16)
    do = torch.randn(B, Tq, H, 64, device="cuda", generator=g).to(BF16)
    o, lse = ops.attn_fwd(q, k, v, 0.125)
    qr, kr, vr = [t.float().permute(0, 2, 1, 3).requires_grad_(True) for t in (q, k, v)]
    orf = torch.nn.functional.scaled_dot_product_attention(qr, kr, vr)
    check(o, orf.permute(0, 2, 1, 3), rel=6e-3)
    lse_ref = torch.logsumexp(torch.einsum("bhqd,bhkd->bhqk", qr, kr) * 0.125, dim=-1)
    assert (lse - lse_ref).abs().max().item() < 1e-4
    orf.backward(do.float().permute(0, 2, 1, 3))
    dq, dk, dv = ops.attn_bwd(q, k, v, o, do, lse, 0.125)
    check(dq, qr.grad.permute(0, 2, 1, 3), rel=8e-3)
    check(dk, kr.grad.permute(0, 2, 1, 3), rel=8e-3)
    check(dv, vr.grad.permute(0, 2, 1, 3), rel=8e-3)


@pytest.mark.parametrize("B,H,Tq,Tk", [(2, 10, 1024, 1024), (1, 3, 1008, 1008), (2, 10, 1024, 77), (1, 10, 4096, 77), (1, 2, 64, 64),
                                        (1, 2, 300, 40), (1, 5, 988, 154), (1, 2, 300, 128), (2, 3, 200, 77), (1, 2, 333, 200),
                                        (2, 2, 130, 129), (1, 1, 4, 300)])
def test_attention_backward_variants_agree(B, H, Tq, Tk):
    """The one-kernel backward (key-major scores, P^T / dS^T in tensor memory, dQ -- and with a single KV tile dK / dV -- summed over
    CTAs by bulk reduce-add in fp32; default; Tq = 333 is not a multiple of 4 and takes the two-kernel path in both modes, 130 x 129
    has one-row / one-key partial tiles) against the bit-reproducible dK/dV + dQ kernel pair: the same five products with
    different rounding points (dS is formed from the unrounded P in both) -> equal within bf16 rounding of the results; both against
    fp32 autograd."""
    from aozora_sdxl_training_b200 import _lib
    ops = _ops()
    g = gen(36)
    q, do = [torch.randn(B, Tq, H, 64, device="cuda", generator=g).to(BF16) for _ in range(2)]
    k, v = [torch.randn(B, Tk, H, 64, device="cuda", generator=g).to(BF16) for _ in range(2)]
    o, lse = ops.attn_fwd(q, k, v, 0.125)
    res = {}
    try:
        for mode in (2, 0):
            _lib.call("aoz_attn_set_bwd_mode", mode)
            res[mode] = [t.clone() for t in ops.attn_bwd(q, k, v, o, do, lse, 0.125)]
    finally:
        _lib.call("aoz_attn_set_bwd_mode", 2)
    qr, kr, vr = [t.float().permute(0, 2, 1, 3).requires_grad_(True) for t in (q, k, v)]
    torch.nn.functional.scaled_dot_product_attention(qr, kr, vr, scale=0.125).backward(do.float().permute(0, 2, 1, 3))
    for a, b, ref in zip(res[2], res[0], (qr.grad, kr.grad, vr.grad)):
        check(a, b, rel=6e-3)
        check(a, ref.permute(0, 2, 1, 3), rel=8e-3)
        check(b, ref.permute(0, 2, 1, 3), rel=8e-3)


@pytest.mark.parametrize("NB,HW,C,silu", [(2, 64, 320, True), (2, 256, 1280, False), (1, 100, 960, True), (4, 4096, 320, True),
                                           (1, 16, 2560, True), (2, 1, 64, False), (4, 1024, 1280, True), (2, 1024, 2560, True),
                                           (3, 1000, 1280, False), (2, 4096, 640, True), (1, 16384, 960, True)])
def test_groupnorm_silu_fwd_bwd(NB, HW, C, silu):
    ops = _ops()
    g = gen(7)
    x = (torch.randn(NB, HW, C, device="cuda", generator=g) * 2 + 0.5).to(BF16)
    ga = (1 + 0.1 * torch.randn(C, device="cuda", generator=g)).to(BF16)
    be = (0.1 * torch.randn(C, device="cuda", generator=g)).to(BF16)
    dres = torch.randn(NB, HW, C, device="cuda", generator=g).to(BF16)
    y, mean, rstd = ops.groupnorm_fwd(x, ga, be, 1e-5, silu)
    xr = x.float().requires_grad_(True)
    gr, br = ga.float().requires_grad_(True), be.float().requires_grad_(True)
    yr = torch.nn.functional.group_norm(xr.permute(0, 2, 1), 32, gr, br, 1e-5)
    yr = (torch.nn.functional.silu(yr) if silu else yr).permute(0, 2, 1)
    check(y, yr)
    dy = torch.randn(y.shape, device="cuda", generator=g).to(BF16)
    yr.backward(dy.float())
    dx, dg, db = ops.groupnorm_bwd(dy, x, ga, be, mean, rstd, silu)
    check(dx, xr.grad)
    check(dg, gr.grad)
    check(db, br.grad)
    dx2, _, _ = ops.groupnorm_bwd(dy, x, ga, be, mean, rstd, silu, dres=dres)
    check(dx2, xr.grad.to(BF16).float() + dres.float())


def test_groupnorm_slab_kernels_agree_with_the_two_pass_path():
    """The single-launch slab kernels (a group's pixels held in shared memory) against the statistics + apply kernels on the
    same inputs: same math, different summation order -> equal within fp32 reduction noise after the bf16 rounding."""
    from aozora_sdxl_training_b200 import _lib
    ops = _ops()
    g = gen(17)
    NB, HW, C = 4, 1024, 1280
    x = (torch.randn(NB, HW, C, device="cuda", generator=g) * 2 + 0.5).to(BF16)
    dy = torch.randn(NB, HW, C, device="cuda", generator=g).to(BF16)
    dres = torch.randn(NB, HW, C, device="cuda", generator=g).to(BF16)
    ga = (1 + 0.1 * torch.randn(C, device="cuda", generator=g)).to(BF16)
    be = (0.1 * torch.randn(C, device="cuda", generator=g)).to(BF16)
    res = {}
    try:
        for slab in (1, 0):
            _lib.call("aoz_groupnorm_set_slab", slab)
            y, mean, rstd = ops.groupnorm_fwd(x, ga, be, 1e-5, True)
            dx, dg, db = ops.groupnorm_bwd(dy, x, ga, be, mean, rstd, True, dres=dres)
            res[slab] = (y, mean, rstd, dx, dg, db)
    finally:
        _lib.call("aoz_groupnorm_set_slab", 1)
    torch.testing.assert_close(res[1][1], res[0][1], rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(res[1][2], res[0][2], rtol=1e-5, atol=1e-6)
    for i in (0, 3, 4, 5):
        check(res[1][i], res[0][i], rel=2e-3)
    # run-to-run reproducible
    y2, _, _ = ops.groupnorm_fwd(x, ga, be, 1e-5, True)
    assert torch.equal(y2, res[1][0])


@pytest.mark.parametrize("rows,C", [(300, 640), (1000, 1280), (7, 64), (4096, 2048), (16384, 640), (4096, 1280), (33, 320), (1, 8),
                                    (2049, 1536), (613, 1024)])
def test_layernorm_fwd_bwd(rows, C):
    ops = _ops()
    g = gen(8)
    x = (torch.randn(rows, C, device="cuda", generator=g) * 2 + 0.5).to(BF16)
    ga = (1 + 0.1 * torch.randn(C, device="cuda", generator=g)).to(BF16)
    be = (0.1 * torch.randn(C, device="cuda", generator=g)).to(BF16)
    y, mean, rstd = ops.layernorm_fwd(x, ga, be)
    xr = x.float().requires_grad_(True)
    gr, br = ga.float().requires_grad_(True), be.float().requires_grad_(True)
    yr = torch.nn.functional.layer_norm(xr, (C,), gr, br, 1e-5)
    check(y, yr)
    xf = x.float()
    torch.testing.assert_close(mean, xf.mean(1), rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(rstd, torch.rsqrt(xf.var(1, unbiased=False) + 1e-5), rtol=1e-4, atol=1e-5)
    dy = torch.randn(y.shape, device="cuda", generator=g).to(BF16)
    yr.backward(dy.float())
    dx, dg, db = ops.layernorm_bwd(dy, x, ga, mean, rstd)
    check(dx, xr.grad)
    check(dg, gr.grad)
    check(db, br.grad)
    dres = torch.randn(rows, C, device="cuda", generator=g).to(BF16)      # residual-stream gradient added in the same pass
    dx2, dg2, db2 = ops.layernorm_bwd(dy, x, ga, mean, rstd, dres=dres)
    check(dx2, xr.grad.to(BF16).float() + dres.float())
    assert torch.equal(dg2, dg) and torch.equal(db2, db)                  # fixed summation order: bit-reproducible


def test_column_sums_of_strided_wide_and_tiny_tensors():
    """Bias gradients by colsum (different heights and widths, strided rows, a caller's destination) against fp32 sums, and
    bit-equal from run to run (fixed summation order, no atomics on data; the finalize tickets reset after every launch)."""
    ops = _ops()
    g = gen(21)
    big = torch.randn(4096, 3840, device="cuda", generator=g).to(BF16)
    xs = [torch.randn(4096, 1280, device="cuda", generator=g).to(BF16), big[:, 1280:2560], torch.randn(4096, 10240, device="cuda", generator=g).to(BF16),
          torch.randn(308, 640, device="cuda", generator=g).to(BF16), torch.randn(1, 8, device="cuda", generator=g).to(BF16)]
    dest = torch.zeros(1280, device="cuda", dtype=BF16)
    outs = [ops.colsum(xs[0], out=dest)] + [ops.colsum(x) for x in xs[1:]]
    assert outs[0].data_ptr() == dest.data_ptr()
    for x, o in zip(xs, outs):
        check(o, x.float().sum(0))
    outs2 = [ops.colsum(x) for x in xs]
    for a, b in zip(outs, outs2):
        assert torch.equal(a, b)


def test_glue_kernels():
    ops = _ops()
    g = gen(9)
    x = torch.randn(2, 6, 10, 64, device="cuda", generator=g).to(BF16)
    up = ops.upsample2x_fwd(x)
    ref = torch.nn.functional.interpolate(x.float().permute(0, 3, 1, 2), scale_factor=2.0, mode="nearest").permute(0, 2, 3, 1)
    assert torch.equal(up.float(), ref)
    dy = torch.randn(up.shape, device="cuda", generator=g).to(BF16)
    check(ops.upsample2x_bwd(dy), dy.float().view(2, 6, 2, 10, 2, 64).sum(dim=(2, 4)))
    a = torch.randn(2, 5, 7, 64, device="cuda", generator=g).to(BF16)
    b = torch.randn(2, 5, 7, 128, device="cuda", generator=g).to(BF16)
    assert torch.equal(ops.concat_channels(a, b), torch.cat([a, b], dim=-1))
    m = torch.randn(1000, 320, device="cuda", generator=g).to(BF16)
    check(ops.colsum(m), m.float().sum(0))
    m3 = torch.randn(3, 500, 64, device="cuda", generator=g).to(BF16)
    check(ops.colsum_grouped(m3), m3.float().sum(1))
    v = torch.randn(777, device="cuda", generator=g).to(BF16)
    check(ops.silu_fwd(v), torch.nn.functional.silu(v.float()))
    src = torch.randn(2, 4, 8, 8, device="cuda", generator=g)
    nhwc = ops.nchw_to_nhwc(src, cpad=8)
    assert torch.equal(nhwc[..., :4].float(), src.to(BF16).float().permute(0, 2, 3, 1)) and nhwc[..., 4:].abs().sum() == 0
    assert torch.equal(ops.nhwc_to_nchw(nhwc, c=4).float(), src.to(BF16).float())
    t = torch.tensor([0.0, 1.0, 500.5, 999.0], device="cuda")
    emb = ops.timestep_embedding(t, 320)
    freqs = torch.exp(-torch.log(torch.tensor(10000.0)) * torch.arange(160, device="cuda") / 160)
    ang = t[:, None] * freqs[None]
    check(emb, torch.cat([ang.cos(), ang.sin()], -1), rel=5e-3)


@pytest.mark.parametrize("mode", ["epsilon", "v_prediction", "rectified_flow"])
def test_noise_target_matches_scheduler_semantics(mode):
    """aoz_noise_target vs the ORACLE's restatement of train.py:2743-2758 (oracle.train_step_ref.make_targets over
    oracle.scheduler_ref.RefDDPMScheduler, identical rounding points); the product's own scheduler class must agree too."""
    ops = _ops()
    from aozora_sdxl_training_b200.scheduler import DDPMScheduler
    from oracle.scheduler_ref import RefDDPMScheduler
    g = gen(10)
    lat = (torch.randn(3, 4, 16, 16, device="cuda", generator=g) * 0.8).to(BF16)
    noise = torch.randn(3, 4, 16, 16, device="cuda", generator=g)
    tickets = torch.tensor([3, 500, 999], device="cuda")
    jitter = torch.rand(3, device="cuda", generator=g)
    sch = RefDDPMScheduler(prediction_type=mode)
    assert torch.equal(DDPMScheduler(prediction_type=mode).alphas_cumprod, sch.alphas_cumprod)
    assert torch.equal(DDPMScheduler().add_noise(lat, noise, tickets), sch.add_noise(lat, noise, tickets))
    acp = sch.alphas_cumprod.cuda()
    xt8, target, cond = ops.noise_target(lat, noise, tickets, None if mode == "rectified_flow" else acp,
                                         jitter if mode == "rectified_flow" else None, mode)
    if mode == "rectified_flow":
        t = ((tickets.float() + jitter) / 1000.0).clamp(0, 1)
        te = t.view(-1, 1, 1, 1)
        noisy, tgt, c = (1 - te) * lat + te * noise, noise - lat, t * 1000.0
    else:
        noisy = sch.add_noise(lat, noise, tickets)
        tgt = sch.get_velocity(lat, noise, tickets) if mode == "v_prediction" else noise
        c = tickets.float()
    assert (xt8[..., :4].float() - noisy.to(BF16).float().permute(0, 2, 3, 1)).abs().max().item() <= 2e-2
    check(xt8[..., :4], noisy.to(BF16).permute(0, 2, 3, 1), rel=2e-3)
    assert xt8[..., 4:].abs().sum() == 0
    check(target, tgt, rel=1e-5, cos=0.999999)
    assert torch.allclose(cond, c, rtol=1e-6)


def test_weighted_mse_loss_and_gradient():
    ops = _ops()
    from aozora_sdxl_training_b200.loss import weighted_sdxl_mse_loss
    g = gen(11)
    pred = torch.randn(3, 4, 16, 16, device="cuda", generator=g).to(BF16).requires_grad_(True)
    target = torch.randn(3, 4, 16, 16, device="cuda", generator=g)
    ts = torch.tensor([0, 495, 2000], device="cuda")
    table = torch.linspace(0.5, 2.0, 1000, device="cuda")
    loss = weighted_sdxl_mse_loss(pred, target, ts, table)
    (loss / 4).backward()
    pr = pred.detach().float().requires_grad_(True)
    per = (pr - target).pow(2).flatten(1).mean(1)
    ref = (per * table[ts.clamp(0, 999)]).mean()
    (ref / 4).backward()
    assert abs(loss.item() - ref.item()) <= 1e-6 * abs(ref.item()) + 1e-7      # fp32 loss: 1e-6 relative
    check(pred.grad, pr.grad)
    loss2, per2, d8 = ops.mse_loss(ops.nchw_to_nhwc(pred.detach(), cpad=4), target, ts, None, denom=3, grad_scale=1 / 3, dpred_ld=8)
    assert abs(loss2.item() - per.mean().item()) <= 1e-6 * per.mean().item() + 1e-7
    assert d8.shape[-1] == 8 and d8[..., 4:].abs().sum() == 0


def _run_raven(cls, pdt, mdt, lr, steps=4, clip=None):
    from oracle import host_ref
    torch.manual_seed(0)
    shapes = [(257,), (64, 33), (3, 3, 16, 16), (40000,), (5,)]
    ps = [torch.nn.Parameter(torch.randn(s).to(pdt).cuda()) for s in shapes]
    ref_p = [p.detach().cpu().clone() for p in ps]
    ref_m = [torch.zeros_like(p, dtype=mdt) for p in ref_p]
    ref_v = [torch.zeros_like(p, dtype=mdt) for p in ref_p]
    hp = dict(lr=lr, betas=(0.9, 0.999), weight_decay=0.01, eps=1e-8, debias_strength=0.3)
    opt = cls(ps, momentum_dtype=mdt, **hp)
    for step in range(1, steps + 1):
        gs = []
        for i, p in enumerate(ps):
            g = (torch.randn(p.shape, generator=torch.Generator().manual_seed(100 * step + i)) * 1e-2).to(pdt)
            gs.append(g)
        if clip is not None:
            host_ref.clip_grad_norm_ref(gs, clip)        # torch.nn.utils.clip_grad_norm_ on CPU (in place)
        for i, p in enumerate(ps):
            p.grad = (torch.randn(p.shape, generator=torch.Generator().manual_seed(100 * step + i)) * 1e-2).to(pdt).cuda()
            host_ref.raven_update_(ref_p[i], gs[i], ref_m[i], ref_v[i], step=step, **hp)
        if clip is None:
            opt.step()
        else:
            opt.clip_and_step(clip)
        opt.zero_grad(set_to_none=True)
    return ps, opt, ref_p, ref_m, ref_v


@pytest.mark.parametrize("pdt,mdt", [(torch.float32, torch.float32), (torch.float32, torch.bfloat16),
                                      (torch.float32, torch.float16), (torch.bfloat16, torch.bfloat16),
                                      (torch.bfloat16, torch.float32)])
def test_raven_step_matches_oracle(pdt, mdt):
    """fp32 parameters: within 1e-6 relative (north_star); bf16 parameters: identical after RNE rounding except where
    the fp32 result sits on a rounding boundary (<= 1 bf16 ulp on a vanishing fraction of elements)."""
    from aozora_sdxl_training_b200.optimizers import RavenAdamW
    ps, opt, ref_p, ref_m, ref_v = _run_raven(RavenAdamW, pdt, mdt, lr=1e-3)
    for i, p in enumerate(ps):
        got, ref = p.detach().cpu().float(), ref_p[i].float()
        if pdt == torch.float32 and mdt == torch.float32:
            assert torch.allclose(got, ref, rtol=1e-6, atol=1e-9), (got - ref).abs().max()       # north_star: 1e-6 relative
        elif pdt == torch.float32:
            # 16-bit moments: a 1-ulp fp32 difference can flip the moment's rounding (2^-8 relative), which moves the
            # update by at most lr * 2^-7
            assert torch.allclose(got, ref, rtol=1e-6, atol=1e-3 * 2 ** -7), (got - ref).abs().max()
        else:
            bad = (got != ref).float().mean().item()
            assert bad < 2e-3 and (got - ref).abs().max() <= ref.abs().max() * 2 ** -7
        m = opt.state[p]["exp_avg"].cpu().float()
        tol = 1e-6 if mdt == torch.float32 else 2 ** -7
        assert torch.allclose(m, ref_m[i].float(), rtol=tol, atol=1e-12)
        assert opt.state[p]["exp_avg"].dtype == mdt and opt.state[p]["exp_avg"].is_cuda and opt.state[p]["step"] == 4


def test_raven_bf16_small_lr_updates_vanish_like_reference():
    """SURVEY.md M6: bf16 parameters, lr 8e-7 -> the update is below half an ulp and the stored weights do not move."""
    from aozora_sdxl_training_b200.optimizers import RavenAdamW
    torch.manual_seed(0)
    p = torch.nn.Parameter(torch.randn(4096).to(torch.bfloat16).cuda())
    before = p.detach().clone()
    opt = RavenAdamW([p], lr=8e-7, betas=(0.9, 0.999), weight_decay=0.01, eps=1e-8, debias_strength=0.3)
    for s in range(3):
        p.grad = (torch.randn(4096, generator=torch.Generator().manual_seed(s)) * 1e-3).to(torch.bfloat16).cuda()
        opt.step()
    assert (p.detach() != before).float().mean().item() < 0.02


def test_raven_golden_trajectories_from_reference_code():
    """Product optimizers vs trajectories recorded from the reference's RavenAdamW / TitanAdamW (tests/golden)."""
    from aozora_sdxl_training_b200.optimizers import RavenAdamW, TitanAdamW
    blob = torch.load(os.path.join(os.path.dirname(__file__), "golden", "raven_golden.pt"))
    hp = blob["hparams"]
    for tag, tr in blob["traj"].items():
        cls = TitanAdamW if tag.startswith("titan") else RavenAdamW
        torch.manual_seed(tr["p0_seed"])
        p = torch.nn.Parameter(torch.randn(257).to(tr["p"].dtype).cuda())
        opt = cls([p], lr=tr["lr"], betas=hp["betas"], weight_decay=hp["weight_decay"], eps=hp["eps"],
                  debias_strength=hp["debias_strength"], momentum_dtype=tr["m"].dtype)
        for g in tr["grads"]:
            (p * g.cuda()).sum().backward()
            if cls is TitanAdamW:
                assert p.grad is None                      # offloaded by the hook, like the reference
            opt.step()
            opt.zero_grad(set_to_none=True)
        got = p.detach().cpu().float()
        ref = tr["p"].float()
        if tr["p"].dtype == torch.float32:
            assert torch.allclose(got, ref, rtol=1e-6, atol=1e-9), tag
        else:
            assert (got != ref).float().mean().item() < 0.02 and (got - ref).abs().max() <= ref.abs().max() * 2 ** -7, tag
        assert torch.allclose(opt.state[p]["exp_avg"].cpu().float(), tr["m"].float(), rtol=2 ** -7 if tr["m"].dtype != torch.float32 else 1e-6, atol=1e-12), tag
        if hasattr(opt, "close"):
            opt.close()


@pytest.mark.parametrize("pdt", [torch.float32, torch.bfloat16])
def test_fused_clip_and_step_matches_torch_clip_grad_norm(pdt):
    """clip_and_step == torch.nn.utils.clip_grad_norm_ (incl. its bf16 rounding, SURVEY.md a7) followed by step()."""
    from aozora_sdxl_training_b200.optimizers import RavenAdamW
    ps, opt, ref_p, _, _ = _run_raven(RavenAdamW, pdt, torch.float32, lr=1e-3, steps=2, clip=0.05)
    for i, p in enumerate(ps):
        got, ref = p.detach().cpu().float(), ref_p[i].float()
        if pdt == torch.float32:
            assert torch.allclose(got, ref, rtol=2e-6, atol=1e-9)
        else:
            assert (got != ref).float().mean().item() < 0.02


def test_grad_norm_and_cpu_state_roundtrip():
    from aozora_sdxl_training_b200.optimizers import RavenAdamW
    torch.manual_seed(1)
    ps = [torch.nn.Parameter(torch.randn(n).cuda()) for n in (1000, 33, 70000)]
    for p in ps:
        p.grad = torch.randn_like(p)
    opt = RavenAdamW(ps, lr=1e-3)
    n = opt.grad_norm(1.0)
    ref = torch.sqrt(sum((p.grad.double() ** 2).sum() for p in ps)).item()
    assert abs(n[0].item() - ref) <= 1e-5 * ref
    assert abs(n[1].item() - min(1.0, 1.0 / (ref + 1e-6))) <= 1e-5
    opt.step()
    st = opt.save_cpu_state()
    assert st["_momentum_dtype"] == torch.bfloat16 and set(st) == {"_momentum_dtype", 0, 1, 2}
    assert st[0]["step"] == 1 and st[0]["exp_avg_cpu"].device.type == "cpu" and st[0]["exp_avg_cpu"].dtype == torch.bfloat16
    opt2 = RavenAdamW(ps, lr=1e-3)
    opt2.load_cpu_state(st)
    for p in ps:
        assert torch.equal(opt2.state[p]["exp_avg"], opt.state[p]["exp_avg"]) and opt2.state[p]["exp_avg"].is_cuda
        assert opt2.state[p]["step"] == 1


def test_no_cpu_fallback():
    from aozora_sdxl_training_b200 import _lib
    ops = _ops()
    with pytest.raises(_lib.AozoraError):
        ops.gemm(torch.zeros(8, 8, dtype=BF16), torch.zeros(8, 8, dtype=BF16))
