"""Per-element float64 bounds and guard bands around every kernel output.

test_gpu_kernels.py compares each kernel with an fp32 reference through a global metric (relative L2 error and cosine over the
whole tensor).  That metric passes one element that is completely wrong, or a whole 8-column store segment that is off by about
its own scale, and it cannot see a store that lands outside the output tensor.  Those are the failure shapes of tile-edge,
tail-tile and epilogue bugs, and the training step writes most of its results into views of larger buffers (fused q/k/v
gradients, stacked weight gradients, the flat data-parallel gradient buffer), where a stray store corrupts another tensor.

Every test here therefore:
  * writes each output into a view of a guarded buffer whose other elements hold a NaN payload that arithmetic never produces
    (bf16 0x7FA5, fp32 0x7FA5A5A5) and checks every bit outside the view afterwards (``assert_untouched``);
  * checks that every input's bytes are unchanged (``Frozen``);
  * compares every element with a float64 reference computed on the GPU from the exact bf16 inputs, against a bound derived
    per op from the kernel's rounding points (``assert_within``; the derivation is in each test's docstring);
  * runs each call twice and requires bit-identical buffers (guards included): these paths promise a fixed summation order.
    The one-kernel attention backward (mode 2) sums dQ with fp32 reduce-adds in arrival order and is exempt.

Bound conventions (u = 2^-8, the largest relative error of one round-to-nearest into bf16):
  * a contraction of length K accumulated in fp32: K * 2^-22 * mag, mag = the same contraction over absolute values in fp64;
  * each bf16 rounding point adds u * |value at that point| (the fp64 value; second-order terms are covered by SLACK).
The worst err/bound ratio per group is printed at the end of the module (run with -s to see it).
"""
import collections
import importlib.util
import itertools
import math
import os
import random

import pytest
import torch

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16
F64 = torch.float64
U = 2.0 ** -8            # bf16 round-to-nearest: |rd(x) - x| <= 2^-8 |x|
FA = 2.0 ** -22          # fp32 accumulation allowance per term of a sum (4x the unit roundoff 2^-24)
SLACK = 1.0 + 2.0 ** -6  # products of two first-order error terms
SCALE = 0.125            # attention softmax scale (head dim 64)

_SENTINEL = {torch.bfloat16: (torch.int16, 0x7FA5), torch.float32: (torch.int32, 0x7FA5A5A5)}
WORST = collections.defaultdict(float)          # group letter -> worst err / bound seen


def _ops():
    from aozora_sdxl_training_b200 import ops
    return ops


def _lib():
    from aozora_sdxl_training_b200 import _lib
    return _lib


def _stream():
    return torch.cuda.current_stream().cuda_stream


def gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def randn(*shape, g, scale=1.0, dtype=BF16):
    return (torch.randn(shape, device="cuda", generator=g) * scale).to(dtype)


@pytest.fixture(scope="module", autouse=True)
def _report_worst_ratios():
    yield
    if WORST:
        print("\nworst err/bound per group: " + ", ".join(f"{k} {v:.3f}" for k, v in sorted(WORST.items())))


# ------------------------------------------------------------------------------------------------------------
# harness
# ------------------------------------------------------------------------------------------------------------
def _bits(t):
    return t.view({2: torch.int16, 4: torch.int32, 8: torch.int64, 1: torch.uint8}[t.element_size()])


def guarded(shape, dtype=BF16, ld=None, col_off=0):
    """(buf, view): ``view`` has ``shape`` and lives inside the flat sentinel-filled ``buf`` with two rows and 64 elements of
    margin on both sides.  ``ld``: row stride of the view (columns ld - cols of every row stay guarded); ``col_off``: shift of
    the view's first element (1 = unaligned, which takes the scalar store paths)."""
    shape = tuple(int(s) for s in shape)
    cols = shape[-1]
    rows = math.prod(shape[:-1])
    ld = cols if ld is None else ld
    assert ld >= cols
    pad = (2 * ld + 64 + 7) // 8 * 8               # keeps an unshifted view 16-byte aligned
    itype, sentinel = _SENTINEL[dtype]
    buf = torch.empty(pad + rows * ld + pad, dtype=dtype, device="cuda")
    _bits(buf).fill_(sentinel)
    strides = [1] * len(shape)
    if len(shape) > 1:
        strides[-2] = ld
        for i in range(len(shape) - 3, -1, -1):
            strides[i] = strides[i + 1] * shape[i + 1]
    return buf, buf.as_strided(shape, strides, pad + col_off)


def _cover(buf, views):
    mask = torch.zeros(buf.numel(), dtype=torch.bool, device=buf.device)
    for v in views:
        off = (v.data_ptr() - buf.data_ptr()) // buf.element_size()
        mask.as_strided(v.shape, v.stride(), off).fill_(True)
    return mask


def assert_untouched(buf, *views):
    """Every element of ``buf`` outside ``views`` still holds the sentinel bits."""
    sentinel = _SENTINEL[buf.dtype][1]
    outside = ~_cover(buf, views)
    bad = outside & (_bits(buf) != sentinel)
    n = int(bad.sum())
    if n:
        idx = torch.nonzero(bad).flatten()
        raise AssertionError(f"{n} element(s) written outside the output view; first at flat offset {int(idx[0])} "
                             f"(buffer of {buf.numel()})")


class Frozen:
    """Snapshot of the inputs' bytes; ``check()`` asserts that the call changed none of them."""

    def __init__(self, *tensors):
        self.items = [(t, _bits(t).clone()) for t in tensors if t is not None]

    def check(self):
        for i, (t, snap) in enumerate(self.items):
            assert torch.equal(_bits(t), snap), f"input {i} ({tuple(t.shape)}) was modified"


def assert_within(got, ref, bound, group, what=""):
    """|got - ref| <= bound elementwise (NaN fails); reports the count, the worst index and its err / bound."""
    got = got.to(F64)
    ref = ref.to(F64).expand_as(got)
    bound = (bound.to(F64) * SLACK).expand_as(got)
    err = (got - ref).abs()
    ratio = torch.where(bound > 0, err / bound, torch.where(err > 0, torch.full_like(err, math.inf), torch.zeros_like(err)))
    ratio = torch.nan_to_num(ratio, nan=math.inf)
    worst = float(ratio.max()) if ratio.numel() else 0.0
    if not worst <= 1.0:
        bad = int((ratio > 1.0).sum())
        flat = int(ratio.flatten().argmax())
        idx = tuple(int(i) for i in torch.unravel_index(torch.tensor(flat), got.shape))
        raise AssertionError(f"{what}: {bad} of {got.numel()} elements outside the bound; worst at {idx}: got "
                             f"{float(got[idx]):.6g}, ref {float(ref[idx]):.6g}, bound {float(bound[idx]):.3g}, "
                             f"err/bound {worst:.3g}")
    WORST[group] = max(WORST[group], worst)
    return worst


def twice(run):
    """run() -> tuple of buffers; called twice, every buffer must be bit-identical (guards included)."""
    first = run()
    second = run()
    for i, (a, b) in enumerate(zip(first, second)):
        assert torch.equal(_bits(a), _bits(b)), f"buffer {i} differs between two identical calls"
    return first


def epilogue(acc, mag, K, bias=None, later=()):
    """(ref, bound) of rd(...rd(rd(acc + bias) + later[0]) + later[1]...) for an fp32 accumulator of a length-K contraction:
    the bias is added to the accumulator, every later addend after a bf16 rounding of the running value (epi_store8's order:
    bias -> time embedding -> residual -> accumulate)."""
    v = acc if bias is None else acc + bias
    bound = K * FA * mag
    for a in later:
        bound = bound + U * v.abs()
        v = v + a
    return v, bound + U * v.abs()


# ------------------------------------------------------------------------------------------------------------
# self-test of the harness
# ------------------------------------------------------------------------------------------------------------
def _old_check():
    spec = importlib.util.spec_from_file_location("_kernel_suite", os.path.join(os.path.dirname(__file__), "test_gpu_kernels.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.check


def test_harness_rejects_what_the_global_metric_accepts():
    """A correct 1000 x 640 GEMM passes; one element off by 2 % of its magnitude and one zeroed 8-column store segment fail
    assert_within but pass test_gpu_kernels.check (global relative L2 <= 4e-3, cosine >= 0.9999); one sentinel overwritten
    just outside the view fails assert_untouched."""
    ops = _ops()
    check = _old_check()
    g = gen(100)
    M, N, K = 1000, 640, 320
    A, B = randn(M, K, g=g), randn(N, K, g=g)
    buf, out = guarded((M, N), ld=N + 8)
    ops.gemm(A, B, out=out, splits=1)
    a64, b64 = A.to(F64), B.to(F64)
    ref, bound = epilogue(a64 @ b64.t(), a64.abs() @ b64.abs().t(), K)
    assert_within(out, ref, bound, "self")
    assert_untouched(buf, out)
    check(out, ref.float())

    bumped = out.clone()
    r, c = divmod(int(ref.abs().argmax()), N)
    bumped[r, c] = (ref[r, c] * 1.02).to(BF16)
    check(bumped, ref.float())
    with pytest.raises(AssertionError):
        assert_within(bumped, ref, bound, "self")

    zeroed = out.clone()
    zeroed[(r + 1) % M, 128:136] = 0
    check(zeroed, ref.float())
    with pytest.raises(AssertionError):
        assert_within(zeroed, ref, bound, "self")

    # one past the last column of row 12: a guard element (ld = N + 8)
    buf.view(torch.int16)[(out[12, N - 1:].data_ptr() - buf.data_ptr()) // 2 + 1] = 0
    with pytest.raises(AssertionError):
        assert_untouched(buf, out)


# ------------------------------------------------------------------------------------------------------------
# A. GEMM
# ------------------------------------------------------------------------------------------------------------
def _pairwise(params, valid, seed=7):
    """Greedy all-pairs cover of the parameter lists (a deterministic subset of the product in which every valid pair of
    values of two parameters appears at least once)."""
    names = list(params)
    rng = random.Random(seed)

    def pairs_of(case):
        return {(i, case[i], j, case[j]) for i, j in itertools.combinations(range(len(names)), 2)}

    wanted = set()
    for i, j in itertools.combinations(range(len(names)), 2):
        for a in params[names[i]]:
            for b in params[names[j]]:
                probe = [None] * len(names)
                probe[i], probe[j] = a, b
                if valid(dict(zip(names, probe)), partial=True):
                    wanted.add((i, a, j, b))
    cases = []
    while wanted:
        best, gain = None, -1
        seed_pair = next(iter(sorted(wanted, key=repr)))
        for _ in range(60):
            case = [rng.choice(params[n]) for n in names]
            case[seed_pair[0]], case[seed_pair[2]] = seed_pair[1], seed_pair[3]
            if not valid(dict(zip(names, case)), partial=False):
                continue
            gn = len(pairs_of(case) & wanted)
            if gn > gain:
                best, gain = case, gn
        if best is None:                       # the seed pair cannot be completed: drop it
            wanted.discard(seed_pair)
            continue
        wanted -= pairs_of(best)
        cases.append(tuple(best))
    return names, cases


_GEMM_PARAMS = {
    "M": [1, 127, 129, 257, 1000],
    "N": [4, 8, 24, 72, 136, 328],
    "K": [8, 72, 1000, 5120],
    "majors": [(False, False), (True, False), (False, True), (True, True)],
    "epi": ["store", "bias", "bias_res", "rowgroup", "acc"],
    "splits": [1, 2, 3, 7],
    "out": ["ld", "block3", "off1"],
    "mode": ["default", "pair0", "pair2", "tail0", "tail2", "wide0", "wide2", "budget-8", "budget100"],
}


def _gemm_valid(c, partial):
    N, majors, epi, splits = c.get("N"), c.get("majors"), c.get("epi"), c.get("splits")
    if N is not None and majors is not None and N % 8 and majors[1]:
        return False                                            # [K, N] B needs a 16-byte row stride
    if epi is not None and splits is not None and splits > 1 and epi not in ("store", "acc"):
        return False                                            # split-K fuses no bias / residual
    return True


_GEMM_NAMES, _GEMM_CASES = _pairwise(_GEMM_PARAMS, _gemm_valid)
_GEMM_CASES += [(4096, 1280, 1280, (False, False), "store", 1, "ld", "wide2"),      # the 320-wide one-wave plan
                (4096, 1280, 1280, (False, True), "acc", 1, "block3", "wide2"),
                (1000, 328, 5120, (False, False), "acc", 7, "off1", "default"),     # scalar split-K reduce with accumulate
                (257, 24, 1000, (True, False), "store", 3, "off1", "budget100")]


def _set_mode(mode):
    lib = _lib()
    if mode.startswith("pair"):
        lib.call("aoz_gemm_set_pair_mode", int(mode[4:]))
    elif mode.startswith("tail"):
        lib.call("aoz_gemm_set_tail_mode", int(mode[4:]))
    elif mode.startswith("wide"):
        lib.call("aoz_gemm_set_wide_mode", int(mode[4:]))
    elif mode == "budget-8":
        lib.call("aoz_gemm_set_sm_budget", lib.query("aoz_sm_count") - 8)
    elif mode == "budget100":
        lib.call("aoz_gemm_set_sm_budget", 100)


def _reset_modes():
    lib = _lib()
    lib.call("aoz_gemm_set_pair_mode", 1)
    lib.call("aoz_gemm_set_tail_mode", 1)
    lib.call("aoz_gemm_set_wide_mode", 1)
    lib.call("aoz_gemm_set_sm_budget", 0)


def _operand(rows, cols, g, scale=1.0):
    """[rows, cols] bf16 operand; a row length that is not a multiple of 8 gets a padded row stride (TMA needs 16-byte strides)."""
    ld = (cols + 7) // 8 * 8
    return randn(rows, ld, g=g, scale=scale)[:, :cols]


def _out_view(M, N, kind):
    if kind == "ld":
        buf, v = guarded((M, N), ld=N + 8)
        return buf, v
    if kind == "block3":
        buf, full = guarded((M, 3 * N), ld=3 * N + 8)
        return buf, full[:, N:2 * N]
    return guarded((M, N), col_off=1)


@pytest.mark.parametrize(",".join(_GEMM_NAMES), _GEMM_CASES)
def test_gemm_elementwise_bounds_and_guards(M, N, K, majors, epi, splits, out, mode):
    """C = A·Bᵀ (+ bias (+ time-embedding row groups) (+ residual) (+ accumulate)) into a guarded view.

    Bound: K·2^-22·(|A|·|B|ᵀ) for the fp32 accumulation (split-K and tail slices add partials of the same terms), then
    2^-8·|v| at every bf16 rounding point v of epi_store8 / the split-K reduce: after bias (+ time embedding), after the
    residual, after the accumulate.  rows_per_group = 100 is not a multiple of the 128-row tile."""
    ops = _ops()
    a_mn, b_mn = majors
    g = gen(1000 + M + 7 * N + 13 * K)
    A = _operand(K, M, g) if a_mn else _operand(M, K, g)
    B = _operand(K, N, g, 0.5) if b_mn else _operand(N, K, g, 0.5)
    bias = randn(N, g=g) if epi in ("bias", "bias_res", "rowgroup") else None
    res = randn(M, N, g=g) if epi == "bias_res" else None
    rpg = 100
    rgb = randn((M + rpg - 1) // rpg, N, g=g) if epi == "rowgroup" else None
    old = randn(M, N, g=g, scale=4.0) if epi == "acc" else None
    frozen = Frozen(A, B, bias, res, rgb)

    def run():
        buf, view = _out_view(M, N, out)
        if old is not None:
            view.copy_(old)
        try:
            _set_mode(mode)
            ops.gemm(A, B, a_mn=a_mn, b_mn=b_mn, bias=bias, residual=res, rowgroup_bias=rgb, rows_per_group=rpg if rgb is not None else 0,
                     out=view, accumulate=old is not None, splits=splits)
        finally:
            _reset_modes()
        assert_untouched(buf, view)
        return buf, view

    buf, view = twice(run)
    frozen.check()
    a64 = (A.t() if a_mn else A).to(F64)
    b64 = (B if b_mn else B.t()).to(F64)
    later = []
    if rgb is not None:
        later.append(rgb.to(F64).repeat_interleave(rpg, dim=0)[:M])
    if res is not None:
        later.append(res.to(F64))
    if old is not None:
        later.append(old.to(F64))
    ref, bound = epilogue(a64 @ b64, a64.abs() @ b64.abs(), K + splits, None if bias is None else bias.to(F64), later)
    assert_within(view, ref, bound, "A", f"gemm {M}x{N}x{K} {majors} {epi} splits={splits} {out} {mode}")


# ------------------------------------------------------------------------------------------------------------
# B. GEGLU
# ------------------------------------------------------------------------------------------------------------
def _gelu64(x):
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


@pytest.mark.parametrize("half", [12, 20])
def test_geglu_rejects_a_half_width_that_is_not_a_multiple_of_8(half):
    """The GEGLU epilogue stores 8-column vectors with no scalar tail: N/2 % 8 != 0 must be refused before any launch."""
    ops, lib = _ops(), _lib()
    g = gen(200)
    x, w = randn(64, 64, g=g), randn(2 * half, 64, g=g)
    buf, out = guarded((64, half), ld=half + 4)
    l0 = lib.query("aoz_launch_count")
    with pytest.raises(lib.AozoraError, match="multiple of 8"):
        ops.gemm(x, w, epi=ops.EPI_GEGLU, out=out)
    assert lib.query("aoz_launch_count") == l0
    assert_untouched(buf)


@pytest.mark.parametrize("what", ["out", "aux", "bias", "ldc", "ld_aux"])
def test_geglu_rejects_misaligned_outputs_and_bias(what):
    """16-byte vector loads / stores of C, aux and bias need 16-byte aligned pointers and row strides that are multiples of 8."""
    ops, lib = _ops(), _lib()
    g = gen(201)
    M, half, K = 64, 64, 64
    x, w = randn(M, K, g=g), randn(2 * half, K, g=g)
    bbuf, bias = guarded((2 * half,), col_off=1 if what == "bias" else 0)
    bias.copy_(randn(2 * half, g=g))
    obuf, out = guarded((M, half), ld=half + 4 if what == "ldc" else half + 8, col_off=1 if what == "out" else 0)
    abuf, aux = guarded((M, 2 * half), ld=2 * half + 4 if what == "ld_aux" else 2 * half + 8, col_off=1 if what == "aux" else 0)
    l0 = lib.query("aoz_launch_count")
    with pytest.raises(lib.AozoraError, match="16-byte aligned"):
        ops.gemm(x, w, bias=bias, epi=ops.EPI_GEGLU, aux=aux, out=out)
    assert lib.query("aoz_launch_count") == l0
    assert_untouched(obuf)
    assert_untouched(abuf)


@pytest.mark.parametrize("M,half,K", [(129, 64, 72), (1000, 640, 320), (257, 5120, 1280)])
def test_geglu_epilogue_elementwise_bounds_and_guards(M, half, K):
    """out = rd(rd(h)·rd(gelu(rd(g)))), aux = [rd(h) | rd(g)] with h, g = x·Wᵀ + b, written into views with ld > row length.

    Bounds: aux: K·2^-22·mag + 2^-8·|h| (resp. g).  out: with e_h, e_g the aux bounds and |gelu'| <= 1.13,
    e_h·G + H·(1.13·e_g + 2^-8·G) + 2^-8·H·G, where H = |h| + e_h and G = |gelu(g)| + 1.13·e_g."""
    ops = _ops()
    g = gen(202 + half)
    x, w, b = randn(M, K, g=g), randn(2 * half, K, g=g, scale=0.05), randn(2 * half, g=g)
    frozen = Frozen(x, w, b)

    def run():
        obuf, out = guarded((M, half), ld=half + 8)
        abuf, aux = guarded((M, 2 * half), ld=2 * half + 16)
        ops.gemm(x, w, bias=b, epi=ops.EPI_GEGLU, aux=aux, out=out)
        assert_untouched(obuf, out)
        assert_untouched(abuf, aux)
        return obuf, abuf, out, aux

    _, _, out, aux = twice(run)
    frozen.check()
    x64, w64 = x.to(F64), w.to(F64)
    pre = x64 @ w64.t() + b.to(F64)
    mag = x64.abs() @ w64.abs().t()
    e = K * FA * mag + U * pre.abs()
    assert_within(aux, pre, e, "B", f"geglu aux {M}x{half}x{K}")
    h, gt = pre[:, :half], pre[:, half:]
    e_h, e_g = e[:, :half], e[:, half:]
    ge = _gelu64(gt)
    H, G = h.abs() + e_h, ge.abs() + 1.13 * e_g
    bound = e_h * G + H * (1.13 * e_g + U * G) + U * H * G
    assert_within(out, h * ge, bound, "B", f"geglu out {M}x{half}x{K}")


# ------------------------------------------------------------------------------------------------------------
# C. grouped GEMM
# ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [77, 1000])
@pytest.mark.parametrize("pair_mode,tail_mode", [(0, 0), (2, 0), (1, 1), (0, 2), (2, 2)])
def test_grouped_gemm_row_and_column_blocks(K, pair_mode, tail_mode):
    """Ten weight-gradient problems dW = dyᵀ·x (K = tokens: 77 for the cross-attention k/v weights) whose outputs are row blocks
    and column blocks of ONE guarded buffer, with M and N off the 128-row / 64-column tile edges (multiples of 8: the operands
    are [K, M] and [K, N] with 16-byte row strides).
    Bound per problem: K·2^-22·(|dy|ᵀ·|x|) + 2^-8·|ref|."""
    ops, lib = _ops(), _lib()
    g = gen(300 + K)
    shapes = [(136, 72), (200, 136), (72, 328), (136, 64), (264, 24), (8, 136), (328, 8), (104, 200), (64, 64), (160, 120)]
    probs = [(randn(K, m, g=g), randn(K, n, g=g)) for m, n in shapes]
    frozen = Frozen(*[t for p in probs for t in p])
    # layout: problems 0-4 stacked as row blocks in columns [0, 328); problems 5-9 side by side as column blocks below them
    row_h = sum(m for m, _ in shapes[:5])
    width = 328 + 8 + sum(n for _, n in shapes[5:]) + 8 * 5

    def views(full):
        vs, r = [], 0
        for m, n in shapes[:5]:
            vs.append(full[r:r + m, :n])
            r += m
        c = 0
        for m, n in shapes[5:]:
            vs.append(full[row_h:row_h + m, c:c + n])
            c += n + 8
        return vs

    def run():
        buf, full = guarded((row_h + max(m for m, _ in shapes[5:]), width), ld=width + 8)
        vs = views(full)
        try:
            lib.call("aoz_gemm_set_pair_mode", pair_mode)
            lib.call("aoz_gemm_set_tail_mode", tail_mode)
            ops.gemm_grouped([(a, b, v) for (a, b), v in zip(probs, vs)], a_mn=True, b_mn=True)
        finally:
            _reset_modes()
        assert_untouched(buf, *vs)
        return buf, full

    _, full = twice(run)
    frozen.check()
    for (a, b), v, (m, n) in zip(probs, views(full), shapes):
        a64, b64 = a.to(F64), b.to(F64)
        ref, bound = epilogue(a64.t() @ b64, a64.abs().t() @ b64.abs(), K)
        assert_within(v, ref, bound, "C", f"grouped {m}x{n}x{K} pair {pair_mode} tail {tail_mode}")


# ------------------------------------------------------------------------------------------------------------
# D. convolution
# ------------------------------------------------------------------------------------------------------------
def _nchw(t):
    return t.permute(0, 3, 1, 2)


def _nhwc(t):
    return t.permute(0, 2, 3, 1)


_CONV_CASES = [
    # NB, H, W, Cin, Cout, stride, epilogue, cin_real, out col_off
    (2, 13, 19, 64, 4, 1, "bias", None, 0),               # conv_out's shape class: Cout = 4 takes the scalar epilogue
    (1, 128, 128, 320, 4, 1, "bias", None, 0),            # conv_out at 128 x 128
    (1, 128, 128, 8, 320, 1, "bias", 4, 0),               # conv_in: 4 real input channels of 8
    (2, 17, 33, 64, 8, 1, "temb_res", None, 0),
    (2, 13, 19, 128, 72, 1, "bias_res", None, 1),         # unaligned output: scalar epilogue with a residual
    (1, 17, 33, 72, 136, 2, "temb", None, 0),             # stride 2 at odd H
    (2, 13, 19, 136, 136, 2, "bias", None, 0),
    (1, 17, 33, 320, 72, 1, "temb_res", None, 1),
]


@pytest.mark.parametrize("NB,H,W,Cin,Cout,stride,epi,cin_real,col_off", _CONV_CASES)
def test_conv_fwd_dgrad_wgrad_elementwise_bounds_and_guards(NB, H, W, Cin, Cout, stride, epi, cin_real, col_off):
    """Forward (bias / time embedding / residual epilogue), dgrad (flipped pack; zero-inserted dy for stride 2) and wgrad
    (accumulated into a grad_w view of a guarded flat buffer, splits 1, 2 and automatic) against an fp64 conv2d.

    Bounds: forward K = 9·Cin, mag = conv2d(|x|, |w|), then the epilogue's rounding points (bias + time embedding, residual);
    dgrad K = 9·Cout over conv_transpose2d(|dy|, |w|); wgrad K = NB·Ho·Wo pixels (+ splits) over the weight gradient of
    (|x|, |dy|), then rd(partial sum) + old, rounded."""
    ops = _ops()
    g = gen(400 + H * W + Cin + Cout)
    cr = cin_real or Cin
    x = randn(NB, H, W, Cin, g=g)
    if cr < Cin:
        x[..., cr:] = 0
    w = randn(Cout, Cin, 3, 3, g=g, scale=0.05)
    if cr < Cin:
        w[:, cr:] = 0
    b = randn(Cout, g=g)
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    temb = randn(NB, Cout, g=g) if "temb" in epi else None
    res = randn(NB, Ho, Wo, Cout, g=g) if "res" in epi else None
    wf, wd = ops.pack_conv_weight(w)
    cpad = (Cout + 7) // 8 * 8                         # dy channels seen by dgrad / wgrad (conv_out: 4 real of 8)
    dy = torch.zeros(NB, Ho, Wo, cpad, device="cuda", dtype=BF16)
    dy[..., :Cout] = randn(NB, Ho, Wo, Cout, g=g)
    old = randn(cpad, cr, 3, 3, g=g, scale=0.5)
    frozen = Frozen(x, wf, wd, b, temb, res, dy)
    x64, w64 = _nchw(x.to(F64)), w.to(F64)
    conv = torch.nn.functional.conv2d
    ref_y = _nhwc(conv(x64, w64, None, stride=stride, padding=1))
    mag_y = _nhwc(conv(x64.abs(), w64.abs(), None, stride=stride, padding=1))
    later = [t for t in (None if temb is None else temb.to(F64)[:, None, None, :], None if res is None else res.to(F64)) if t is not None]
    ref_y, bound_y = epilogue(ref_y, mag_y, 9 * Cin, b.to(F64), later)

    def run_fwd():
        buf, y = guarded((NB, Ho, Wo, Cout), col_off=col_off)
        ops.conv_fwd(x, wf, Cout, 3, stride=stride, pad=1, bias=b, rowgroup_bias=temb, residual=res, out=y)
        assert_untouched(buf, y)
        return buf, y

    buf, y = twice(run_fwd)
    assert_within(y, ref_y, bound_y, "D", f"conv fwd {NB}x{H}x{W} {Cin}->{Cout} s{stride} {epi}")

    dy64 = _nchw(dy[..., :Cout].to(F64))
    ref_dx = _nhwc(torch.nn.grad.conv2d_input(x64.shape, w64, dy64, stride=stride, padding=1))
    mag_dx = _nhwc(torch.nn.grad.conv2d_input(x64.shape, w64.abs(), dy64.abs(), stride=stride, padding=1))
    ref_dx, bound_dx = epilogue(ref_dx, mag_dx, 9 * cpad)
    dyi = dy if stride == 1 else ops.zero_insert2x(dy, H, W)

    def run_dgrad():
        buf, dx = guarded((NB, H, W, Cin))
        ops.conv_fwd(dyi, wd, Cin, 3, stride=1, pad=1, flip=True, out=dx)
        assert_untouched(buf, dx)
        return buf, dx

    buf, dx = twice(run_dgrad)
    assert_within(dx, ref_dx, bound_dx, "D", f"conv dgrad {NB}x{H}x{W} {Cin}->{Cout} s{stride}")

    dy64p = _nchw(dy.to(F64))
    gw = torch.nn.grad.conv2d_weight(x64[:, :cr], (cpad, cr, 3, 3), dy64p, stride=stride, padding=1)
    mag_w = torch.nn.grad.conv2d_weight(x64[:, :cr].abs(), (cpad, cr, 3, 3), dy64p.abs(), stride=stride, padding=1)
    for splits in (1, 2, None):
        def run_wgrad():
            buf, flat = guarded((cpad * cr * 9 + 24,))
            gview = flat[16:16 + cpad * cr * 9].view(cpad, cr, 3, 3)
            gview.copy_(old)
            ops.conv_wgrad(dy, x, 3, stride=stride, pad=1, grad_w=gview, accumulate=True, cin_real=cr, splits=splits)
            assert_untouched(buf, gview)
            return buf, gview

        buf, gview = twice(run_wgrad)
        sp = splits or 16
        ref_w, bound_w = epilogue(gw, mag_w, NB * Ho * Wo + sp, None, [old.to(F64)])
        assert_within(gview, ref_w, bound_w, "D", f"conv wgrad {NB}x{H}x{W} {Cin}->{Cout} s{stride} splits={splits}")
    frozen.check()


# ------------------------------------------------------------------------------------------------------------
# E. attention
# ------------------------------------------------------------------------------------------------------------
def _heads(t, B, T, H):
    """[B*T, ...] column block -> [B, T, H, 64] view.  The kernels take the row stride of the [B*T, ...] block (t.stride(0)):
    with T = 1 the stride of the size-1 T dimension of the 4-D view is arbitrary."""
    return t.view(B, T, H, 64) if t.is_contiguous() else t.unflatten(0, (B, T)).unflatten(-1, (H, 64))


_ATTN_CASES = [(2, 3, 1, 1, True), (2, 3, 3, 3, True), (2, 2, 63, 63, True), (2, 2, 65, 65, True), (1, 5, 127, 127, True),
               (2, 2, 129, 129, True), (1, 2, 4032, 4032, True),
               (2, 2, 1, 77, False), (2, 3, 63, 77, False), (1, 5, 129, 77, False), (1, 2, 4032, 77, False),
               (2, 2, 65, 154, False), (1, 2, 127, 154, False), (2, 3, 3, 154, False)]


@pytest.mark.parametrize("mode", [0, 2])
@pytest.mark.parametrize("B,H,Tq,Tk,self_attn", _ATTN_CASES)
def test_attention_elementwise_bounds_and_guards(B, H, Tq, Tk, self_attn, mode):
    """q / k / v are column blocks of guarded fused buffers in the UNet layout (self: [B·T, 3C], cross: q [B·Tq, C] and
    k / v [B·77, 2C]); o and lse go into guarded views, dq / dk / dv into column blocks of guarded [B·Tq, 3C] / [B·Tk, 2C]
    buffers.  The backward's reference is the explicit fp64 formula on the kernel's own o and lse.

    Bounds (per score: e_S = 64·2^-22·scale·(|q|·|k|ᵀ) + 2^-21·(|scale·s| + |lse|) + 2^-20 for the fp32 scores, the exp and the
    log-sum; P's relative error e_P = e_S, plus 2^-8 where P is rounded to bf16 for an MMA):
      o:   (e_P + 2^-8)·(P·|V| + |o|) + Tk·2^-22·P·|V| + 2^-8·|o|;   lse: max_j e_S + (Tk + 8)·2^-22
      dV:  (e_P + 2^-8)·Pᵀ·|dO| + Tq·2^-22·Pᵀ·|dO| + 2^-8·|dV|
      dS = P∘(dP − D): E = e_P·|dS| + P∘(64·2^-22·(|dO|·|V|ᵀ + Σ|dO∘o|)) + 2^-8·|dS| (dS rounded for the MMAs)
      dQ:  scale·(E·|K| + Tk·2^-22·|dS|·|K|) + 2^-8·|dQ|;   dK: scale·(Eᵀ·|Q| + Tq·2^-22·|dS|ᵀ·|Q|) + 2^-8·|dK|"""
    lib = _lib()
    g = gen(500 + Tq + 3 * Tk + H)
    C = H * 64
    if self_attn:
        qbuf, qkv = guarded((B * Tq, 3 * C), ld=3 * C + 8)
        qkv.copy_(randn(B * Tq, 3 * C, g=g))
        q2, k2, v2 = qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:]
        kbuf = None
    else:
        qbuf, q2 = guarded((B * Tq, C), ld=C + 8)
        q2.copy_(randn(B * Tq, C, g=g))
        kbuf, kv = guarded((B * Tk, 2 * C), ld=2 * C + 8)
        kv.copy_(randn(B * Tk, 2 * C, g=g))
        k2, v2 = kv[:, :C], kv[:, C:]
    q, k, v = _heads(q2, B, Tq, H), _heads(k2, B, Tk, H), _heads(v2, B, Tk, H)
    do = randn(B, Tq, H, 64, g=g)
    frozen = Frozen(qbuf, kbuf, do)

    def run_fwd():
        obuf, o2 = guarded((B * Tq, C), ld=C + 8)
        lbuf, lse = guarded((B, H, Tq), dtype=torch.float32)
        o = _heads(o2, B, Tq, H)
        lib.call("aoz_attn_fwd", q.data_ptr(), q2.stride(0), k.data_ptr(), k2.stride(0), v.data_ptr(), v2.stride(0),
                 o.data_ptr(), o2.stride(0), lse.data_ptr(), B, H, Tq, Tk, SCALE, _stream())
        assert_untouched(obuf, o2)
        assert_untouched(lbuf, lse)
        return obuf, lbuf, o, lse, o2

    obuf, lbuf, o, lse, o2 = run_fwd()
    o_again, lse_again = run_fwd()[2:4]
    assert torch.equal(_bits(o), _bits(o_again)) and torch.equal(_bits(lse), _bits(lse_again))
    frozen.check()

    q64, k64, v64 = [t.to(F64).permute(0, 2, 1, 3) for t in (q, k, v)]          # [B, H, T, 64]
    s = q64 @ k64.transpose(-1, -2) * SCALE
    lse_ref = torch.logsumexp(s, dim=-1)
    P = torch.exp(s - lse_ref[..., None])
    ref_o = P @ v64
    e_S = 64 * FA * SCALE * (q64.abs() @ k64.abs().transpose(-1, -2)) + 2.0 ** -21 * (s.abs() + lse_ref.abs()[..., None]) + 2.0 ** -20
    assert_within(lse, lse_ref, e_S.amax(-1) + (Tk + 8) * FA, "E", f"attn lse B{B} H{H} {Tq}x{Tk}")
    PV = P @ v64.abs()
    e_P = e_S.amax(-1, keepdim=True)
    bound_o = (e_P + U) * (PV + ref_o.abs()) + Tk * FA * PV + U * ref_o.abs()
    assert_within(o.to(F64).permute(0, 2, 1, 3), ref_o, bound_o, "E", f"attn o B{B} H{H} {Tq}x{Tk}")

    # backward reference: the explicit formula on the kernel's o and lse
    o64, do64 = o.to(F64).permute(0, 2, 1, 3), do.to(F64).permute(0, 2, 1, 3)
    Pk = torch.exp(s - lse.to(F64)[..., None])
    dP = do64 @ v64.transpose(-1, -2)
    D = (do64 * o64).sum(-1, keepdim=True)
    dS = Pk * (dP - D)
    ref_dv = Pk.transpose(-1, -2) @ do64
    ref_dq = SCALE * dS @ k64
    ref_dk = SCALE * dS.transpose(-1, -2) @ q64
    e_Sk = 64 * FA * SCALE * (q64.abs() @ k64.abs().transpose(-1, -2)) + 2.0 ** -21 * (s.abs() + lse.to(F64).abs()[..., None]) + 2.0 ** -20
    PdO = Pk.transpose(-1, -2) @ do64.abs()
    bound_dv = ((e_Sk + U) * Pk).transpose(-1, -2) @ do64.abs() + Tq * FA * PdO + U * ref_dv.abs()
    E = e_Sk * dS.abs() + Pk * (64 * FA * (do64.abs() @ v64.abs().transpose(-1, -2) + (do64 * o64).abs().sum(-1, keepdim=True))) + U * dS.abs()
    bound_dq = SCALE * (E @ k64.abs() + Tk * FA * dS.abs() @ k64.abs()) + U * ref_dq.abs()
    bound_dk = SCALE * (E.transpose(-1, -2) @ q64.abs() + Tq * FA * dS.abs().transpose(-1, -2) @ q64.abs()) + U * ref_dk.abs()
    del s, P, Pk, dP, dS, E, e_S, e_Sk

    def run_bwd():
        qgbuf, qg = guarded((B * Tq, 3 * C if self_attn else C), ld=(3 * C if self_attn else C) + 8)
        if self_attn:
            kgbuf = None
            dq2, dk2, dv2 = qg[:, :C], qg[:, C:2 * C], qg[:, 2 * C:]
        else:
            kgbuf, kg = guarded((B * Tk, 2 * C), ld=2 * C + 8)
            dq2, dk2, dv2 = qg, kg[:, :C], kg[:, C:]
        dq, dk, dv = _heads(dq2, B, Tq, H), _heads(dk2, B, Tk, H), _heads(dv2, B, Tk, H)
        ws = _ops().workspace(lib.query("aoz_attn_bwd_workspace_floats", B, H, Tq), q.device)
        try:
            lib.call("aoz_attn_set_bwd_mode", mode)
            lib.call("aoz_attn_bwd", q.data_ptr(), q2.stride(0), k.data_ptr(), k2.stride(0), v.data_ptr(), v2.stride(0),
                     o.data_ptr(), o2.stride(0), do.data_ptr(), C, lse.data_ptr(), dq.data_ptr(), dq2.stride(0),
                     dk.data_ptr(), dk2.stride(0), dv.data_ptr(), dv2.stride(0), B, H, Tq, Tk, SCALE, ws.data_ptr(), _stream())
        finally:
            lib.call("aoz_attn_set_bwd_mode", 2)
        if self_attn:
            assert_untouched(qgbuf, qg)
        else:
            assert_untouched(qgbuf, qg)
            assert_untouched(kgbuf, kg)
        return [t for t in (qgbuf, kgbuf) if t is not None], (dq, dk, dv)

    inputs = Frozen(qbuf, kbuf, do, obuf, lbuf)
    bufs, (dq, dk, dv) = run_bwd()
    if mode == 0:                                   # the two-kernel backward is bit-reproducible
        bufs2, _ = run_bwd()
        for a, b2 in zip(bufs, bufs2):
            assert torch.equal(_bits(a), _bits(b2))
    inputs.check()
    tag = f"attn bwd mode {mode} B{B} H{H} {Tq}x{Tk}"
    assert_within(dv.to(F64).permute(0, 2, 1, 3), ref_dv, bound_dv, "E", tag + " dv")
    assert_within(dq.to(F64).permute(0, 2, 1, 3), ref_dq, bound_dq, "E", tag + " dq")
    assert_within(dk.to(F64).permute(0, 2, 1, 3), ref_dk, bound_dk, "E", tag + " dk")


# ------------------------------------------------------------------------------------------------------------
# F. norms
# ------------------------------------------------------------------------------------------------------------
STAT = 2.0 ** -12      # allowed error of the statistics: mean within STAT·sigma, rstd within STAT relative


def _norm_ref(x64, mean, rstd, gamma, beta, dy64, silu, red_dims):
    """fp64 y = silu?((x - mean)·rstd·γ + β) and its backward with the statistics over ``red_dims``, plus the magnitudes the
    bounds are built from: w = 1 + |x̂| (how far a statistics error moves x̂), adz = |dy|·(|silu'| + |γ|·w) (the SiLU slope and
    its change over a z error; |silu''| <= 1/2), dxmag = rstd·(adz·|γ| + mean(adz·|γ|) + w·mean(adz·|γ|·w))."""
    xh = (x64 - mean) * rstd
    z = xh * gamma + beta
    sg = torch.sigmoid(z)
    y = z * sg if silu else z
    dact = sg * (1 + z * (1 - sg)) if silu else torch.ones_like(z)
    dz = dy64 * dact
    n = math.prod(x64.shape[d] for d in red_dims)
    m1 = (dz * gamma).sum(red_dims, keepdim=True) / n
    m2 = (dz * gamma * xh).sum(red_dims, keepdim=True) / n
    dx = rstd * (dz * gamma - m1 - xh * m2)
    w = 1 + xh.abs()
    adz = dy64.abs() * (dact.abs() + (gamma.abs() * w if silu else 0))
    a = adz * gamma.abs()
    dxmag = rstd * (a + a.sum(red_dims, keepdim=True) / n + w * (a * w).sum(red_dims, keepdim=True) / n)
    return y, w, dz, xh, dx, adz, dxmag


@pytest.mark.parametrize("C,HW,slab,offset", [
    (1280, 1024, 1, 0.25), (1280, 1024, 1, 8), (1280, 1024, 1, 32), (1280, 1024, 1, 64), (1280, 1024, 1, 128),
    (2560, 1024, 1, 0.25), (2560, 1024, 1, 128),
    (320, 16384, 1, 0.25), (320, 16384, 1, 128),
    (640, 4096, 1, 0.25), (640, 4096, 1, 8), (640, 4096, 1, 32), (640, 4096, 1, 64), (640, 4096, 1, 128),
    (960, 4096, 1, 128), (1280, 4096, 1, 64),
    (1280, 1024, 0, 0.25), (1280, 1024, 0, 128)])
def test_groupnorm_offset_inputs_elementwise_bounds_and_guards(C, HW, slab, offset):
    """GroupNorm(32)(+SiLU) forward and backward on x = offset·σ + σ·z (σ = 2): slab kernels (C = 1280 / 2560 at 32 x 32) and
    the statistics + apply path (C = 320 / 640 / 960 at 64 x 64 and 128 x 128, and C = 1280 with the slab off).  dgamma / dbeta
    go into views of one guarded flat buffer, dx with dres into a guarded view.

    Bounds: the statistics may be off by STAT = 2^-12 (mean: STAT·σ_group, rstd: STAT relative) -- a fixed-order fp32 reduction
    of up to 2^20 terms x − pivot of size ~σ is within ~2^-16 of both, while E[x²] − mean² loses (offset/σ)²·2^-24·depth.
      y:      2^-8·|y| + 2^-20 + 2·STAT·1.1·|γ|·(1 + |x̂|)   (1.1 bounds the SiLU slope)
      mean:   STAT·σ + 2^-23·|mean|;  rstd: STAT·rstd
      dx:     2^-8·|dx| + 2^-8·|dx + dres| + 4·STAT·dxmag   (dxmag: see _norm_ref)
      dγ, dβ: 2^-8·|ref| + (NB·HW·2^-22 + 2·STAT)·Σ adz·(1 + |x̂|)  resp.  Σ adz"""
    ops, lib = _ops(), _lib()
    NB, silu = 2, True
    g = gen(600 + C + HW + int(offset))
    sigma = 2.0
    x = (torch.randn(NB, HW, C, device="cuda", generator=g) * sigma + offset * sigma).to(BF16)
    ga = (1 + 0.1 * torch.randn(C, device="cuda", generator=g)).to(BF16)
    be = (0.1 * torch.randn(C, device="cuda", generator=g)).to(BF16)
    dy = randn(NB, HW, C, g=g)
    dres = randn(NB, HW, C, g=g)
    frozen = Frozen(x, ga, be, dy, dres)

    def run():
        try:
            lib.call("aoz_groupnorm_set_slab", slab)
            y, mean, rstd = ops.groupnorm_fwd(x, ga, be, 1e-5, silu)
            pbuf, flat = guarded((2 * C + 16,))
            dg, db = flat[8:8 + C], flat[8 + C:8 + 2 * C]
            dx, _, _ = ops.groupnorm_bwd(dy, x, ga, be, mean, rstd, silu, dres=dres, dgamma=dg, dbeta=db)
        finally:
            lib.call("aoz_groupnorm_set_slab", 1)
        assert_untouched(pbuf, dg, db)
        return y, mean, rstd, pbuf, dx, dg, db

    y, mean, rstd, pbuf, dx, dg, db = twice(run)
    frozen.check()
    x64 = x.to(F64).view(NB, HW, 32, C // 32)
    mu = x64.mean((1, 3), keepdim=True)
    var = x64.var((1, 3), unbiased=False, keepdim=True)
    rs = 1.0 / torch.sqrt(var + 1e-5)
    gam, bet = ga.to(F64).view(32, C // 32), be.to(F64).view(32, C // 32)
    y64, w, dz, xh, dx64, adz, dxmag = _norm_ref(x64, mu, rs, gam, bet, dy.to(F64).view(NB, HW, 32, C // 32), silu, (1, 3))
    tag = f"groupnorm C{C} HW{HW} slab{slab} offset{offset}"
    assert_within(mean, mu.view(NB, 32), STAT * torch.sqrt(var).view(NB, 32) + 2.0 ** -23 * mu.abs().view(NB, 32), "F", tag + " mean")
    assert_within(rstd, rs.view(NB, 32), STAT * rs.view(NB, 32), "F", tag + " rstd")
    assert_within(y.view(NB, HW, 32, C // 32), y64, U * y64.abs() + 2.0 ** -20 + 2 * STAT * 1.1 * gam.abs() * w, "F", tag + " y")
    dsum = dx64 + dres.to(F64).view(NB, HW, 32, C // 32)
    assert_within(dx.view(NB, HW, 32, C // 32), dsum, U * (dx64.abs() + dsum.abs()) + 4 * STAT * dxmag, "F", tag + " dx")
    n = NB * HW
    ref_dg = (dz * xh).sum((0, 1)).flatten()
    ref_db = dz.sum((0, 1)).flatten()
    mag_dg = (adz * w).sum((0, 1)).flatten()
    mag_db = adz.sum((0, 1)).flatten()
    assert_within(dg, ref_dg, U * ref_dg.abs() + (n * FA + 2 * STAT) * mag_dg, "F", tag + " dgamma")
    assert_within(db, ref_db, U * ref_db.abs() + (n * FA + 2 * STAT) * mag_db, "F", tag + " dbeta")


@pytest.mark.parametrize("rows,C,offset", [(4096, 640, 0.25), (4096, 640, 128), (1000, 1280, 64), (7, 2048, 128), (77, 320, 8)])
def test_layernorm_offset_inputs_elementwise_bounds_and_guards(rows, C, offset):
    """LayerNorm forward and backward (with dres) on offset inputs: dgamma / dbeta / dx_colsum into views of one guarded flat
    buffer.  Bounds as for GroupNorm with the statistics over a row; dx_colsum is the column sum of the stored bf16 dx:
    Σ_rows bound(dx) + 2^-8·|ref| + rows·2^-22·Σ|dx|."""
    ops = _ops()
    g = gen(700 + rows + C)
    sigma = 2.0
    x = (torch.randn(rows, C, device="cuda", generator=g) * sigma + offset * sigma).to(BF16)
    ga = (1 + 0.1 * torch.randn(C, device="cuda", generator=g)).to(BF16)
    be = (0.1 * torch.randn(C, device="cuda", generator=g)).to(BF16)
    dy, dres = randn(rows, C, g=g), randn(rows, C, g=g)
    frozen = Frozen(x, ga, be, dy, dres)

    def run():
        y, mean, rstd = ops.layernorm_fwd(x, ga, be)
        pbuf, flat = guarded((3 * C + 24,))
        dg, db, col = flat[8:8 + C], flat[16 + C:16 + 2 * C], flat[24 + 2 * C:24 + 3 * C]
        dx, _, _ = ops.layernorm_bwd(dy, x, ga, mean, rstd, dres=dres, dgamma=dg, dbeta=db, dx_colsum=col)
        assert_untouched(pbuf, dg, db, col)
        return y, mean, rstd, pbuf, dx, dg, db, col

    y, mean, rstd, pbuf, dx, dg, db, col = twice(run)
    frozen.check()
    x64 = x.to(F64)
    mu = x64.mean(1, keepdim=True)
    var = x64.var(1, unbiased=False, keepdim=True)
    rs = 1.0 / torch.sqrt(var + 1e-5)
    y64, w, dz, xh, dx64, adz, dxmag = _norm_ref(x64, mu, rs, ga.to(F64), be.to(F64), dy.to(F64), False, (1,))
    tag = f"layernorm {rows}x{C} offset{offset}"
    assert_within(mean, mu.flatten(), STAT * torch.sqrt(var).flatten() + 2.0 ** -23 * mu.abs().flatten(), "F", tag + " mean")
    assert_within(rstd, rs.flatten(), STAT * rs.flatten(), "F", tag + " rstd")
    assert_within(y, y64, U * y64.abs() + 2.0 ** -20 + 2 * STAT * ga.to(F64).abs() * w, "F", tag + " y")
    dsum = dx64 + dres.to(F64)
    bound_dx = U * (dx64.abs() + dsum.abs()) + 4 * STAT * dxmag
    assert_within(dx, dsum, bound_dx, "F", tag + " dx")
    ref_dg, ref_db = (dz * xh).sum(0), dz.sum(0)
    assert_within(dg, ref_dg, U * ref_dg.abs() + (rows * FA + 2 * STAT) * (adz * w).sum(0), "F", tag + " dgamma")
    assert_within(db, ref_db, U * ref_db.abs() + (rows * FA + 2 * STAT) * adz.sum(0), "F", tag + " dbeta")
    ref_col = dsum.sum(0)
    bound_col = bound_dx.sum(0) + U * ref_col.abs() + rows * FA * dsum.abs().sum(0)
    assert_within(col, ref_col, bound_col, "F", tag + " dx_colsum")


# ------------------------------------------------------------------------------------------------------------
# G. glue
# ------------------------------------------------------------------------------------------------------------
def test_silu_bwd_odd_length():
    """dx = dy·silu'(x) for n = 8k + 5 into a guarded view.  Bound: 2^-8·|ref| + 2^-18·|dy|·(1 + |x|) (fp32 sigmoid with a fast
    exponential)."""
    lib = _lib()
    g = gen(800)
    n = 8 * 1000 + 5
    dy, x = randn(n, g=g), randn(n, g=g, scale=4.0)
    frozen = Frozen(dy, x)

    def run():
        buf, dx = guarded((n,))
        lib.call("aoz_silu_bwd", dy.data_ptr(), x.data_ptr(), n, dx.data_ptr(), _stream())
        assert_untouched(buf, dx)
        return buf, dx

    buf, dx = twice(run)
    frozen.check()
    xr = x.to(F64).requires_grad_(True)
    torch.nn.functional.silu(xr).backward(dy.to(F64))
    bound = U * xr.grad.abs() + 2.0 ** -18 * dy.to(F64).abs() * (1 + x.to(F64).abs())
    assert_within(dx, xr.grad, bound, "G", "silu_bwd")


@pytest.mark.parametrize("n", [8 * 7 + 5, 8 * 4099 + 5])
def test_add_in_place_with_scalar_tail(n):
    """out is a (GradSink.add, gradient accumulation): a += b over n = 8k + 5 elements, vector body and scalar tail.
    Bound: 2^-8·|a + b| (one rounding of an exact fp32 sum)."""
    ops = _ops()
    g = gen(801 + n)
    a0, b = randn(n, g=g), randn(n, g=g, scale=3.0)
    frozen = Frozen(b)

    def run():
        buf, a = guarded((n,))
        a.copy_(a0)
        ops.add(a, b, out=a)
        assert_untouched(buf, a)
        return buf, a

    buf, a = twice(run)
    frozen.check()
    ref = a0.to(F64) + b.to(F64)
    assert_within(a, ref, U * ref.abs(), "G", f"add n={n}")


@pytest.mark.parametrize("accumulate", [False, True])
def test_copy_channels_with_offsets(accumulate):
    """dst[..., 16:48] (+)= src[..., 8:40] over all rows; every other channel of dst and everything around it stays guarded."""
    ops = _ops()
    g = gen(802)
    rows = 2 * 13 * 19
    src = randn(2, 13, 19, 64, g=g)
    old = randn(rows, 32, g=g)
    frozen = Frozen(src)

    def run():
        buf, dst = guarded((2, 13, 19, 56))
        block = dst.view(rows, 56)[:, 16:48]
        if accumulate:
            block.copy_(old)
        ops.copy_channels(src, 8, dst, 16, 32, accumulate=accumulate)
        assert_untouched(buf, block)
        return buf, block

    buf, block = twice(run)
    frozen.check()
    ref = src.view(rows, 64)[:, 8:40].to(F64) + (old.to(F64) if accumulate else 0)
    assert_within(block, ref, U * ref.abs(), "G", f"copy_channels acc={accumulate}")


@pytest.mark.parametrize("H,W", [(7, 9), (13, 19)])
def test_upsample_and_zero_insert_at_odd_sizes(H, W):
    """Nearest 2x upsample (exact), its adjoint (sum of 4: 2^-8·|ref| + 4·2^-22·Σ|dy|) and zero insertion for Hout ∈ {2H−1, 2H}
    (exact), all into guarded outputs."""
    lib = _lib()
    g = gen(803 + H)
    NB, C = 2, 24
    x = randn(NB, H, W, C, g=g)
    dy = randn(NB, 2 * H, 2 * W, C, g=g)
    frozen = Frozen(x, dy)

    def run_up():
        buf, y = guarded((NB, 2 * H, 2 * W, C))
        lib.call("aoz_upsample2x_fwd", x.data_ptr(), NB, H, W, C, y.data_ptr(), _stream())
        assert_untouched(buf, y)
        return buf, y

    _, y = twice(run_up)
    assert torch.equal(_bits(y), _bits(x.repeat_interleave(2, 1).repeat_interleave(2, 2)))
    WORST["G"] = max(WORST["G"], 0.0)

    def run_down():
        buf, dx = guarded((NB, H, W, C))
        lib.call("aoz_upsample2x_bwd", dy.data_ptr(), NB, H, W, C, dx.data_ptr(), _stream())
        assert_untouched(buf, dx)
        return buf, dx

    _, dx = twice(run_down)
    d64 = dy.to(F64).view(NB, H, 2, W, 2, C)
    ref = d64.sum((2, 4))
    assert_within(dx, ref, U * ref.abs() + 4 * FA * d64.abs().sum((2, 4)), "G", "upsample2x_bwd")

    for hout, wout in ((2 * H - 1, 2 * W - 1), (2 * H, 2 * W), (2 * H - 1, 2 * W)):
        def run_zi():
            buf, z = guarded((NB, hout, wout, C))
            lib.call("aoz_zero_insert2x", x.data_ptr(), NB, H, W, C, hout, wout, z.data_ptr(), _stream())
            assert_untouched(buf, z)
            return buf, z

        _, z = twice(run_zi)
        want = torch.zeros(NB, hout, wout, C, device="cuda", dtype=BF16)
        want[:, ::2, ::2] = x[:, :(hout + 1) // 2, :(wout + 1) // 2]
        assert torch.equal(_bits(z), _bits(want)), (hout, wout)
    frozen.check()


def test_layout_conversions_with_padding_and_fp32():
    """nchw_to_nhwc from fp32 with cpad > C (values rounded once, pad channels exactly zero) and nhwc_to_nchw from a tensor
    with ld > C into fp32 (exact), both into guarded outputs."""
    lib = _lib()
    g = gen(804)
    NB, C, H, W, cpad = 2, 4, 13, 19, 8
    src = torch.randn(NB, C, H, W, device="cuda", generator=g) * 3
    frozen = Frozen(src)

    def run_in():
        buf, dst = guarded((NB, H, W, cpad))
        lib.call("aoz_nchw_to_nhwc", src.data_ptr(), 1, NB, C, H * W, cpad, dst.data_ptr(), _stream())
        assert_untouched(buf, dst)
        return buf, dst

    _, nhwc = twice(run_in)
    assert torch.equal(_bits(nhwc[..., :C]), _bits(src.to(BF16).permute(0, 2, 3, 1)))
    assert torch.equal(_bits(nhwc[..., C:]), torch.zeros_like(_bits(nhwc[..., C:])))
    frozen.check()
    nhwc = nhwc.contiguous()
    frozen2 = Frozen(nhwc)

    def run_out():
        buf, dst = guarded((NB, C, H, W), dtype=torch.float32)
        lib.call("aoz_nhwc_to_nchw", nhwc.data_ptr(), NB, C, H * W, cpad, dst.data_ptr(), 1, _stream())
        assert_untouched(buf, dst)
        return buf, dst

    _, nchw = twice(run_out)
    assert torch.equal(nchw, src.to(BF16).float())
    frozen2.check()


def test_column_sums_accumulate_into_views():
    """colsum (strided rows) and the per-image colsum_grouped with accumulate = True into views of one guarded flat buffer.
    Bound: M·2^-22·Σ|x| + 2^-8·|sum| + 2^-8·|sum + old|."""
    ops, lib = _ops(), _lib()
    g = gen(805)
    big = randn(1000, 3 * 320, g=g)
    x = big[:, 320:640]
    x3 = randn(3, 777, 136, g=g)
    old1, old3 = randn(320, g=g, scale=20.0), randn(3, 136, g=g, scale=20.0)
    frozen = Frozen(big, x3)

    def run():
        buf, flat = guarded((320 + 3 * 136 + 16,))
        v1 = flat[8:328]
        v3 = flat[336:336 + 3 * 136].view(3, 136)
        v1.copy_(old1)
        v3.copy_(old3)
        ops.colsum(x, out=v1, accumulate=True)
        ws = ops.workspace(lib.query("aoz_colsum_workspace_floats", 3, 136), x3.device)
        lib.call("aoz_colsum", x3.data_ptr(), 3, 777, 136, 136, 777 * 136, v3.data_ptr(), 1, ws.data_ptr(), _stream())
        assert_untouched(buf, v1, v3)
        return buf, v1, v3

    buf, v1, v3 = twice(run)
    frozen.check()
    for got, t, old, dim, M in ((v1, x, old1, 0, 1000), (v3, x3, old3, 1, 777)):
        s = t.to(F64).sum(dim)
        ref, bound = epilogue(s, t.to(F64).abs().sum(dim), M, None, [old.to(F64)])
        assert_within(got, ref, bound, "G", f"colsum M={M}")


def test_timestep_embedding_all_training_timesteps():
    """[cos | sin](t·10000^(-k/160)) for t = 0..999 (and fractional t) at dim 320.  Bound: 2^-8·|ref| + the fp32 angle error
    2^-21·(|θ| + 1) (frequency and product rounding, sin / cos accuracy)."""
    lib = _lib()
    t = torch.cat([torch.arange(1000, device="cuda", dtype=torch.float32), torch.tensor([0.5, 123.25, 998.75], device="cuda")])
    frozen = Frozen(t)

    def run_contig():
        buf, out = guarded((t.numel(), 320))
        lib.call("aoz_timestep_embedding", t.data_ptr(), t.numel(), 320, out.data_ptr(), _stream())
        assert_untouched(buf, out)
        return buf, out

    _, out = twice(run_contig)
    frozen.check()
    k = torch.arange(160, device="cuda", dtype=F64)
    ang = t.to(F64)[:, None] * torch.exp(-math.log(10000.0) * k / 160)[None]
    ref = torch.cat([ang.cos(), ang.sin()], -1)
    err = 2.0 ** -21 * (ang.abs() + 1)
    assert_within(out, ref, U * ref.abs() + torch.cat([err, err], -1), "G", "timestep_embedding")


def test_mse_loss_gradient_pad_channels_and_guard():
    """dL/dpred = 2·(pred − target)·w·grad_scale / (C·HW) into a guarded [B, h, w, 8] view whose 4 pad channels start at zero
    and must stay zero; loss within 2^-20 relative of fp64.  Bound on dpred: 2^-8·|ref| + 2^-20·|ref|."""
    lib = _lib()
    g = gen(806)
    B, C, H, W = 3, 4, 13, 19
    pred = randn(B, H, W, C, g=g)
    target = torch.randn(B, C, H, W, device="cuda", generator=g)
    tickets = torch.tensor([0, 495, 2000], device="cuda")
    table = torch.linspace(0.5, 2.0, 1000, device="cuda")
    gs = 1.0 / 3.0
    frozen = Frozen(pred, target, tickets, table)

    def run():
        buf, d = guarded((B, H, W, 8))
        d.zero_()
        per = torch.empty(B, device="cuda")
        w = torch.empty(B, device="cuda")
        loss = torch.empty(1, device="cuda")
        HWn = H * W
        lib.call("aoz_mse_loss", pred.data_ptr(), HWn * C, 1, C, target.data_ptr(), tickets.data_ptr(), table.data_ptr(), 1000,
                 B, C, HWn, float(B), 0, gs, per.data_ptr(), w.data_ptr(), loss.data_ptr(), d.data_ptr(), HWn * 8, 1, 8, _stream())
        assert_untouched(buf, d)
        return buf, d, loss

    buf, d, loss = twice(run)
    frozen.check()
    assert torch.equal(_bits(d[..., C:]), torch.zeros_like(_bits(d[..., C:])))
    wt = table.to(F64)[tickets.clamp(0, 999)]
    diff = pred.to(F64).permute(0, 3, 1, 2) - target.to(F64)
    ref_loss = ((diff ** 2).mean((1, 2, 3)) * wt).sum() / B
    assert_within(loss, ref_loss.view(1), 2.0 ** -20 * ref_loss.abs().view(1), "G", "mse loss")
    ref = (2 * diff * wt[:, None, None, None] * gs / (C * H * W)).permute(0, 2, 3, 1)
    assert_within(d[..., :C], ref, (U + 2.0 ** -20) * ref.abs(), "G", "mse dpred")
