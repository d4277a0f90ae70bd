"""CPU tests of gradient accumulation under data parallel (world size 2, gloo): every micro-step is reduce-scattered exactly as with
GRADIENT_ACCUMULATION_STEPS = 1, the reduced shard is accumulated, and the last micro-step of a window clips and steps.  After two
windows the parameters and moments must equal one process that sums the same global-batch gradients over each window and then
steps -- also when one rank holds no rows in a middle or in the last micro-step (its step goes through
``SDXLTrainStep._rank_without_rows``, which must follow the same phase rule, or the ranks' collectives fall out of step).  The
device math is injected from the CPU oracle, as in test_parallel_cpu.py."""
import datetime
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

HP = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01, debias_strength=0.3)
CLIP = 0.5
SHAPES = [(5,), (40, 25), (17,), (3, 3, 8, 8), (3,), (701,)]


class _OracleBackend:
    """CPU stand-in for the CUDA kernels, built from the oracle (tests only)."""

    @staticmethod
    def sumsq(seg_g, numels, plan, out3, gdt):
        out3[2] = sum(float((g.double() ** 2).sum()) for g in seg_g)

    @staticmethod
    def clip_coef(sumsq, max_norm, out2):
        nrm = float(sumsq[0]) ** 0.5
        out2[0] = nrm
        out2[1] = min(1.0, max_norm / (nrm + 1e-6))

    @staticmethod
    def raven(seg_p, seg_g, seg_m, seg_v, plan, hyper, clip_coef, pdt, gdt, mdt):
        from oracle import host_ref
        c = 1.0 if clip_coef is None else float(clip_coef[0])
        for p, g, m, v in zip(seg_p, seg_g, seg_m, seg_v):
            host_ref.raven_update_(p, g * c, m, v, **HP, step=_OracleBackend.step)

    @staticmethod
    def add(a, b, out):
        out.copy_(a + b)


class _Cfg:
    SEED = 42
    BATCH_SIZE = 4
    MAX_TRAIN_STEPS = 100
    CLIP_GRAD_NORM = CLIP
    PREDICTION_TYPE = "epsilon"
    TIMESTEP_ALLOCATION = None
    TIMESTEP_STRATIFIED_SAMPLING = False
    TIMESTEP_LOSS_WEIGHT_CURVE = None
    LR_CUSTOM_CURVE = None


def _grad(window, micro, rank, i):
    return torch.randn(SHAPES[i], generator=torch.Generator().manual_seed(100000 * window + 1000 * micro + 10 * rank + i))


def _worker(rank, world, port, q, ga, empty_at):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=datetime.timedelta(seconds=60))
    try:
        from aozora_sdxl_training_b200.parallel import DataParallel
        from aozora_sdxl_training_b200.trainer import SDXLTrainStep
        from oracle import host_ref
        torch.manual_seed(0)
        model = torch.nn.ParameterList([torch.nn.Parameter(torch.randn(s)) for s in SHAPES])
        ref_p = [p.detach().clone() for p in model]
        ref_m = [torch.zeros_like(p) for p in ref_p]
        ref_v = [torch.zeros_like(p) for p in ref_p]
        dp = DataParallel(model, momentum_dtype=torch.float32, backend=_OracleBackend, flat_dtype=torch.float32, bucket_elems=256)
        opt = dp.make_optimizer(**HP)
        assert len(dp.layout.buckets) >= 4 and any(len(b) > 1 for b in dp.param_buckets)     # parameters straddle buckets
        step = SDXLTrainStep(model, opt, type("C", (_Cfg,), dict(GRADIENT_ACCUMULATION_STEPS=ga)), device="cpu", dp=dp)
        empty_rank = world - 1
        for window in (1, 2):
            _OracleBackend.step = window
            acc = None
            for micro in range(1, ga + 1):
                last = micro == ga
                if micro == empty_at and rank == empty_rank:
                    res = step._rank_without_rows({"global_batch_len": 2, "global_row_offset": 2})
                    assert res.did_optimizer_step == last and (res.grad_norm is None) == (not last)
                else:
                    for i in reversed(range(len(SHAPES))):
                        g = _grad(window, micro, rank, i)
                        if i % 2 == 0:
                            dp.grad_ready(dp.params[i], g)                               # staged by copy
                        else:
                            dp.grad_view(dp.params[i]).copy_(g)                          # produced in place
                            dp.grad_ready(dp.params[i], dp.grad_view(dp.params[i]))
                    step.micro_step += 1
                    if last:
                        dp.reduce_clip_step(opt, CLIP, accumulated=True)
                    else:
                        dp.reduce_accumulate(first=micro == 1)
                summed = [sum(_grad(window, micro, r, i) for r in range(world) if not (micro == empty_at and r == empty_rank))
                          for i in range(len(SHAPES))]
                acc = summed if acc is None else [a + s for a, s in zip(acc, summed)]
            assert step.micro_step == window * ga and opt.step_count == window
            norm = torch.sqrt(sum((g.double() ** 2).sum() for g in acc)).item()
            coef = min(1.0, CLIP / (norm + 1e-6))
            for i in range(len(SHAPES)):
                host_ref.raven_update_(ref_p[i], acc[i] * coef, ref_m[i], ref_v[i], **HP, step=window)
            for i, p in enumerate(dp.params):
                assert torch.allclose(p.detach(), ref_p[i], rtol=1e-6, atol=1e-8), (window, i)
        st = opt.save_cpu_state()
        for i in range(len(SHAPES)):
            assert st[i]["step"] == 2
            assert torch.allclose(st[i]["exp_avg_cpu"], ref_m[i], rtol=1e-6, atol=1e-9), i
            assert torch.allclose(st[i]["exp_avg_sq_cpu"], ref_v[i], rtol=1e-6, atol=1e-12), i
        q.put((rank, "ok"))
    except Exception:
        import traceback
        q.put((rank, traceback.format_exc()))
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.timeout(180)
@pytest.mark.parametrize("ga,empty_at", [(2, None), (3, None), (3, 2), (3, 3)],
                         ids=["ga2", "ga3", "ga3-no-rows-middle", "ga3-no-rows-last"])
def test_accumulated_data_parallel_matches_one_process_world2_gloo(ga, empty_at):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q, ga, empty_at)) for r in range(2)]
    for p in procs:
        p.start()
    results = [q.get(timeout=150) for _ in procs]
    for p in procs:
        p.join(timeout=30)
    for rank, msg in results:
        assert msg == "ok", f"rank {rank}: {msg}"
