"""Gradient accumulation (GRADIENT_ACCUMULATION_STEPS > 1) on one GPU: the multi-tensor bf16 accumulate kernel, the eager step that
uses it, and the captured step with its first / middle / last phases.

The reference accumulates ``(loss / GA).backward()`` into bf16 ``p.grad``: one fp32 add and one round to nearest even per
micro-step.  ``aoz_grad_accum_mt`` must therefore be bit-identical to ``aoz_add`` tensor by tensor, and the eager step that now
issues it once per micro-step must be bit-identical to the per-parameter ``ops.add`` loop it replaced."""
import gc

import pytest
import torch

pytestmark = pytest.mark.gpu
BF16 = torch.bfloat16
SENTINEL = 0x7FA5                    # bf16 NaN payload no arithmetic produces: marks the guard band around every output


# ---- harness (restated from tests/test_gpu_guarded.py) ------------------------------------------------------------
def _bits(t):
    return t.view(torch.int16)


def guarded(n, shift=0):
    """(buf, view): a length-n bf16 view inside a sentinel-filled buffer with 64 guard elements on both sides; ``shift`` = 1
    leaves the view's start off 16-byte alignment."""
    buf = torch.empty(64 + n + 64 + 8, dtype=BF16, device="cuda")
    _bits(buf).fill_(SENTINEL)
    return buf, buf[64 + shift:64 + shift + n]


def assert_untouched(buf, view):
    off = (view.data_ptr() - buf.data_ptr()) // 2
    bits = _bits(buf)
    assert bool((bits[:off] == SENTINEL).all()) and bool((bits[off + view.numel():] == SENTINEL).all()), "guard band written"


# ---- 1. the kernel -------------------------------------------------------------------------------------------------
SIZES = [1, 7, 8, 9, 16383, 16384, 16385, 3 * 16384 + 5, 4096 * 1280, 1001]
SHIFTED = {len(SIZES) - 1}           # this tensor's output starts off alignment: its chunks take the element-wise path


def _special_pairs(n, g):
    """bf16 operands: random values of mixed scale, with signed zeros, subnormals and exact ties of a + b planted through them."""
    a = (torch.randn(n, device="cuda", generator=g) * torch.exp2(torch.randint(-20, 8, (n,), device="cuda", generator=g).float()))
    b = torch.randn(n, device="cuda", generator=g)
    a, b = a.to(BF16), b.to(BF16)
    specials = [(0.0, -0.0), (-0.0, -0.0), (-0.0, 0.0),
                (2.0 ** -130, 2.0 ** -131), (-(2.0 ** -128), 2.0 ** -133),      # subnormal bf16 (and their sum)
                (1.0, 2.0 ** -8), (1.0 + 2.0 ** -7, 2.0 ** -8),                # halfway: rounds down to even / up to even
                (-3.0, -(2.0 ** -7)), (256.0, 1.0), (257.0 * 2 ** -8, -(2.0 ** -8))]
    for k, (x, y) in enumerate(specials):
        a[k::3 * len(specials) + 1] = x
        b[k::3 * len(specials) + 1] = y
    return a, b


def _tables():
    g = torch.Generator(device="cuda").manual_seed(11)
    return [_special_pairs(n, g) for n in SIZES]


def _run(pairs, mode, copy):
    """One launch over every pair.  mode: "out" (fresh guarded y), "a" (y is a), "b" (y is b).  Returns the guarded buffers and y."""
    from aozora_sdxl_training_b200 import ops
    from aozora_sdxl_training_b200.optimizers.raven import MultiTensorPlan, _Staging
    bufs, ys, as_, bs = [], [], [], []
    for i, (a0, b0) in enumerate(pairs):
        buf, v = guarded(a0.numel(), shift=1 if i in SHIFTED else 0)
        a, b = a0.clone(), b0.clone()
        if mode == "a":
            v.copy_(a0)
            a = v
        elif mode == "b":
            v.copy_(b0)
            b = v
        bufs.append(buf)
        ys.append(v)
        as_.append(a)
        bs.append(b)
    ops.grad_accum_mt(ys, as_, bs, MultiTensorPlan(), _Staging(), copy=copy)
    torch.cuda.synchronize()
    return bufs, ys


@pytest.mark.parametrize("copy", [False, True])
@pytest.mark.parametrize("mode", ["out", "a", "b"])
def test_grad_accum_mt_bit_identical_to_add_with_guards(mode, copy):
    from aozora_sdxl_training_b200 import ops
    if copy and mode == "a":
        pytest.skip("copy mode does not read a")
    pairs = _tables()
    snap = [(_bits(a).clone(), _bits(b).clone()) for a, b in pairs]
    bufs, ys = _run(pairs, mode, copy)
    for i, ((a0, b0), buf, y) in enumerate(zip(pairs, bufs, ys)):
        assert_untouched(buf, y)
        ref = b0 if copy else ops.add(a0, b0)
        assert torch.equal(_bits(y), _bits(ref)), f"tensor {i} (n={a0.numel()}) differs from aoz_add"
    torch.cuda.synchronize()
    for (a0, b0), (sa, sb) in zip(pairs, snap):                       # the inputs' bytes are unchanged
        assert torch.equal(_bits(a0), sa) and torch.equal(_bits(b0), sb)
    bufs2, _ = _run(pairs, mode, copy)                                # run to run: every buffer bit-identical, guards included
    for b1, b2 in zip(bufs, bufs2):
        assert torch.equal(_bits(b1), _bits(b2))


def test_grad_accum_mt_rejects_bad_arguments_before_any_launch():
    from aozora_sdxl_training_b200 import _lib
    from aozora_sdxl_training_b200.optimizers.raven import MultiTensorPlan
    t = torch.zeros(64, dtype=BF16, device="cuda")
    plan = MultiTensorPlan()
    plan.ensure([64], t.device)
    ptr = torch.tensor([t.data_ptr()], dtype=torch.int64, device="cuda")
    pp = torch.tensor([t.data_ptr()] * 2, dtype=torch.int64, device="cuda")
    lib = _lib.load()
    stream = torch.cuda.current_stream().cuda_stream

    def call(n_tensors, a, b, y, numel, copy=0):
        return lib.aoz_grad_accum_mt(n_tensors, plan.n_chunks, a, b, y, numel, plan.chunk_start.data_ptr(),
                                     plan.chunk_tensor.data_ptr(), copy, stream)

    good = ptr.data_ptr()
    l0 = _lib.query("aoz_launch_count")
    assert call(0, good, good, good, plan.numel.data_ptr()) == -1
    assert call(-1, good, good, good, plan.numel.data_ptr()) == -1
    assert call(1, good, 0, good, plan.numel.data_ptr()) == -1                        # null table
    assert call(1, 0, good, good, plan.numel.data_ptr()) == -1                        # a is read unless copy
    assert call(1, good, good, good, 0) == -1
    assert call(1, good, good, pp.data_ptr() + 4, plan.numel.data_ptr()) == -1       # misaligned pointer table
    assert call(1, good, good, good, plan.numel.data_ptr() + 2) == -1
    assert "aoz_grad_accum_mt" in _lib.last_error()
    assert _lib.query("aoz_launch_count") == l0
    assert call(1, 0, good, good, plan.numel.data_ptr(), copy=1) == 0                 # copy needs no a table
    torch.cuda.synchronize()
    assert _lib.query("aoz_launch_count") == l0 + 1


# ---- the step ------------------------------------------------------------------------------------------------------
class Cfg:
    SEED = 42
    BATCH_SIZE = 2
    MAX_TRAIN_STEPS = 40
    GRADIENT_ACCUMULATION_STEPS = 1
    CLIP_GRAD_NORM = 1.0
    PREDICTION_TYPE = "rectified_flow"
    TIMESTEP_ALLOCATION = None
    TIMESTEP_STRATIFIED_SAMPLING = False
    TIMESTEP_LOSS_WEIGHT_CURVE = [[0, 1], [0.49570201, 2], [1, 1]]
    LR_CUSTOM_CURVE = [[0.0, 1e-3], [1.0, 1e-4]]


def build_model(seed=42):
    from aozora_sdxl_training_b200.unet import UNet2DConditionModel, init_weights_, tiny_config
    return init_weights_(UNet2DConditionModel(tiny_config()), seed=seed, std=0.05).to(BF16).cuda()


def make_batch(B=2, h=16, w=16, L=77, seed=3):
    g = torch.Generator().manual_seed(seed)
    return dict(latents=(torch.randn(B, 4, h, w, generator=g) * 0.8).to(BF16), embeds=torch.randn(B, L, 128, generator=g).to(BF16),
                pooled=torch.randn(B, 64, generator=g).to(BF16), time_ids=[[1024, 1024, 0, 0, 1024, 1024]] * B)


def make_step(ga, use_graph, cls=None, **cfg):
    from aozora_sdxl_training_b200.optimizers import RavenAdamW
    from aozora_sdxl_training_b200.trainer import SDXLTrainStep
    prod = build_model()
    opt = RavenAdamW([{"params": list(prod.parameters()), "lr_scale": 1.0}], lr=1e-3, betas=(0.9, 0.999), weight_decay=0.01,
                     debias_strength=0.3)
    c = type("C", (Cfg,), dict(GRADIENT_ACCUMULATION_STEPS=ga, **cfg))
    return prod, opt, (cls or SDXLTrainStep)(prod, opt, c, use_cuda_graph=use_graph, graph_warmup=2)


@pytest.fixture
def reproducible_attention():
    """The fused attention backward sums dQ across CTAs in an unspecified order; the two-kernel form is bit-reproducible."""
    from aozora_sdxl_training_b200 import _lib
    _lib.call("aoz_attn_set_bwd_mode", 0)
    yield
    _lib.call("aoz_attn_set_bwd_mode", 2)


def _old_eager_step_class():
    """SDXLTrainStep.step as it was before the multi-tensor accumulate: one ``ops.add`` per parameter and micro-step."""
    from aozora_sdxl_training_b200 import ops
    from aozora_sdxl_training_b200.trainer import SDXLTrainStep, StepResult

    class OldLoop(SDXLTrainStep):
        @torch.no_grad()
        def step(self, batch, *, noise=None, jitter=None, taps=None):
            latents, embeds, pooled, time_ids, tickets, noise, jitter, global_len = self._host_inputs(batch, noise, jitter)
            loss, grads = self._device_step(latents, embeds, pooled, time_ids, tickets, noise, jitter, global_len)
            self.micro_step += 1
            if self._accum is None:
                self._accum = grads
            else:
                for p, g in grads.items():
                    ops.add(self._accum[p], g, out=self._accum[p])
            grads = self._accum
            if self.lr_scheduler is not None:
                self.lr_scheduler.step(self.micro_step)
            did = self.micro_step % self.grad_accum == 0
            norm = None
            if did:
                norm = self.optimizer.clip_and_step(self.clip, grads=grads)
                self._accum = None
                self.optimizer_steps += 1
            return StepResult(loss=loss, grad_norm=norm, timesteps=tickets, did_optimizer_step=did,
                              lr=self.optimizer.param_groups[0]["lr"])

    return OldLoop


def test_eager_accumulation_bit_identical_to_per_parameter_loop(reproducible_attention):
    """Two windows of GA = 3, eager: losses, gradient norms and every parameter bit-identical to the per-parameter loop."""
    runs = []
    for cls in (_old_eager_step_class(), None):
        prod, opt, step = make_step(3, False, cls)
        losses, norms = [], []
        for i in range(6):
            res = step.step(make_batch(seed=i))
            losses.append(res.loss.clone())
            norms.append(None if res.grad_norm is None else res.grad_norm.clone())
        runs.append((losses, norms, [p.detach().clone() for p in prod.parameters()]))
    (l0, n0, p0), (l1, n1, p1) = runs
    assert all(torch.equal(a, b) for a, b in zip(l0, l1))
    assert [n is None for n in n0] == [n is None for n in n1] == [True, True, False, True, True, False]
    assert all(torch.equal(a, b) for a, b in zip(n0, n1) if a is not None)
    assert all(torch.equal(a.view(torch.int16), b.view(torch.int16)) for a, b in zip(p0, p1))


def _count_accumulates(monkeypatch):
    from aozora_sdxl_training_b200 import ops
    calls = []
    real = ops.grad_accum_mt

    def counted(*a, **k):
        calls.append(k.get("copy", False))
        return real(*a, **k)

    monkeypatch.setattr(ops, "grad_accum_mt", counted)
    return calls


def _run_counting(step, n, calls):
    """n micro-steps; per step (result, library launches issued, accumulate calls)."""
    from aozora_sdxl_training_b200 import _lib
    out = []
    for i in range(n):
        c0, l0 = len(calls), _lib.query("aoz_launch_count")
        res = step.step(make_batch(seed=i))
        out.append((res, _lib.query("aoz_launch_count") - l0, len(calls) - c0))
    return out


@pytest.mark.parametrize("ga", [2, 3])
def test_captured_accumulation_matches_eager(ga, monkeypatch):
    """3 windows, graph against eager: the same optimizer-step pattern, Raven step counters = micro-steps / GA, losses and weights
    within the tolerances of test_cuda_graph_replay_matches_eager.  Captures are checked by their launches: graph replays bypass
    the library's launch sites, so the capturing step's launch count is what the graph holds."""
    n = 3 * ga
    calls = _count_accumulates(monkeypatch)
    results = []
    for use_graph in (False, True):
        prod, opt, step = make_step(ga, use_graph)
        rows = _run_counting(step, n, calls)
        results.append(([r.did_optimizer_step for r, _, _ in rows], [r.loss_value() for r, _, _ in rows],
                        [p.detach().float().cpu() for p in prod.parameters()], {opt.state[p]["step"] for p in prod.parameters()}, rows,
                        step))
    (d0, l0, p0, s0, _, _), (d1, l1, p1, s1, rows, gstep) = results
    assert d0 == d1 == [(i + 1) % ga == 0 for i in range(n)]
    assert s0 == s1 == {n // ga}
    for a, b in zip(l0, l1):
        assert abs(a - b) <= 2e-3 * abs(a), (l0, l1)
    moved = sum(float((a - b).abs().sum()) for a, b in zip(p0, p1)) / sum(float(a.abs().sum()) for a in p0)
    assert moved < 2e-3
    # window 3 is captured: micro-steps 2*ga+1 .. 3*ga
    assert len(gstep._graphs) == ga and len(gstep._pools) == 1
    ga1_capture = _run_counting(make_step(1, True)[2], 3, calls)[2][1]
    cap = [launches for _, launches, _ in rows[2 * ga:]]
    assert all(acc == 1 for _, _, acc in rows[2 * ga:])
    assert cap[-1] == ga1_capture + 1                      # the last phase: GA = 1's launches plus one accumulate
    for c in cap[:-1]:
        assert c == ga1_capture - 3 + 1                    # first / middle: no norm (2 launches) or Raven (1) launch, one accumulate
    for r, _, _ in rows:
        assert (r.grad_norm is not None) == r.did_optimizer_step


def test_ga1_capture_unchanged(monkeypatch):
    """GA = 1: the capture issues exactly the launches of one eager step, no accumulate call, no accumulator, no shared pool."""
    prod, opt, step = make_step(1, True)
    rows = _run_counting(step, 4, _count_accumulates(monkeypatch))
    (_, eager2, acc2), (_, capture, acc3) = rows[1], rows[2]
    assert capture == eager2 and acc2 == acc3 == 0 and all(a == 0 for _, _, a in rows)
    assert step._acc is None and step._pools == {} and len(step._graphs) == 1
    assert all(r.did_optimizer_step for r, _, _ in rows)
    assert list(step._graphs) == [((2, 4, 16, 16), (2, 77, 128), 2)]


def _reserved_peak(ga):
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_reserved()
    prod, opt, step = make_step(ga, True)
    trace = []
    for i in range(3 * ga):
        step.step(make_batch(h=64, w=64, seed=i))
        torch.cuda.synchronize()
        trace.append(f"{(torch.cuda.memory_reserved() - base) / 2**20:.0f}/{(torch.cuda.max_memory_reserved() - base) / 2**20:.0f}")
    print(f"\nGA={ga} reserved/peak MiB after each micro-step: {' '.join(trace)}")
    peak = torch.cuda.max_memory_reserved() - base
    acc = 0 if step._acc is None else step._acc.numel() * 2
    del prod, opt, step
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return peak, acc


def test_captured_phases_share_one_memory_pool():
    """GA = 3 captures three graphs of one shape into one shared pool.  The reserved peak must stay within GA = 1's plus the
    accumulator plus SLACK.  SLACK is allocator fragmentation, not a second copy of the activations: the pool reuses the blocks
    the first capture freed, but the caching allocator does not lay the second capture's blocks out exactly over them (on a B200
    the tiny UNet at 64 x 64 reserved 404 MiB after the warm-ups, +126 MiB at the first capture, +80 at the second, +0 at the
    third).  A pool per phase would add two more captures of ~126 MiB each, which this bound rejects."""
    SLACK = 96 << 20
    peak1, acc1 = _reserved_peak(1)
    peak3, acc3 = _reserved_peak(3)
    print(f"\nreserved peak GA=1 {peak1 / 2**20:.1f} MiB, GA=3 {peak3 / 2**20:.1f} MiB, accumulator {acc3 / 2**20:.1f} MiB")
    assert acc1 == 0 and acc3 > 0
    assert peak3 <= peak1 + acc3 + SLACK
