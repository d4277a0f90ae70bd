"""Gradient accumulation on one GPU: the multi-tensor accumulate kernel alone, and the captured step at bench.py's workload with
GRADIENT_ACCUMULATION_STEPS = 1 against 4.

    python tools/grad_accum_bench.py [--steps 16] [--rounds 2] [--batch 4] [--res 1024]

1. ``aoz_grad_accum_mt`` over the SDXL UNet's 1680 trainable tensors (2.57 G elements; every operand is GBs, far beyond the
   126 MB L2): time per launch, GB/s at 6 B per element (add: two bf16 reads, one write) or 4 B (copy), and the fraction of the
   HBM bandwidth measured here by a device-to-device copy of 4 GiB.  ``aoz_add`` over one flat tensor of the same size is the
   single-tensor yardstick with the same arithmetic.
2. The captured step (one SDXLTrainStep per configuration, graphs captured, then timed), GA = 1 and GA = 4 alternated ``--rounds``
   times: images/s and ms per micro-step, split into the last micro-step of a window (norm + Raven) and the others.
The card's name, power limit and SM clock limit are printed first, from the same process.
"""
import argparse
import gc
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

BF16 = torch.bfloat16


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def events_ms(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def kernel_alone(reps):
    from aozora_sdxl_training_b200 import ops
    from aozora_sdxl_training_b200.optimizers.raven import MultiTensorPlan, _Staging
    from aozora_sdxl_training_b200.unet import UNet2DConditionModel, sdxl_config
    with torch.device("meta"):
        numels = [p.numel() for p in UNet2DConditionModel(sdxl_config()).parameters()]
    offs, off = [], 0
    for n in numels:
        offs.append(off)
        off += (n + 7) // 8 * 8
    total = sum(numels)
    flat = [torch.randn(off, device="cuda").to(BF16) for _ in range(3)]
    a, b, y = ([f[o:o + n] for o, n in zip(offs, numels)] for f in flat)
    plan, stage = MultiTensorPlan(), _Staging()
    ms_add = events_ms(lambda: ops.grad_accum_mt(y, a, b, plan, stage), reps)
    ms_inplace = events_ms(lambda: ops.grad_accum_mt(a, a, b, plan, stage), reps)
    ms_copy = events_ms(lambda: ops.grad_accum_mt(y, None, b, plan, stage, copy=True), reps)
    ms_flat = events_ms(lambda: ops.add(flat[0], flat[1], out=flat[2]), reps)
    del flat, a, b, y
    src = torch.empty(1 << 31, dtype=BF16, device="cuda")
    dst = torch.empty_like(src)
    ms_cp = events_ms(lambda: dst.copy_(src), reps)
    hbm = 2 * src.numel() * 2 / ms_cp / 1e6
    del src, dst
    torch.cuda.empty_cache()
    print(f"kernel alone: {len(numels)} tensors, {total / 1e9:.3f} G elements, {plan.n_chunks} chunks; measured HBM "
          f"(4 GiB device copy) {hbm:.0f} GB/s")
    for what, ms, bpe in (("grad_accum_mt add, y separate", ms_add, 6), ("grad_accum_mt add, in place", ms_inplace, 6),
                          ("grad_accum_mt copy", ms_copy, 4), ("aoz_add, one flat tensor", ms_flat, 6)):
        gbs = bpe * total / ms / 1e6
        print(f"  {what:32s} {ms:8.3f} ms  {gbs:7.0f} GB/s  {gbs / hbm:.3f} of measured HBM")


def step_ab(args):
    import bench
    from aozora_sdxl_training_b200.optimizers import RavenAdamW
    from aozora_sdxl_training_b200.trainer import SDXLTrainStep
    from aozora_sdxl_training_b200.unet import UNet2DConditionModel, init_weights_fast_, sdxl_config
    with torch.device("cuda"):
        unet = UNet2DConditionModel(sdxl_config()).to(BF16)
    init_weights_fast_(unet, seed=bench.Cfg.SEED)
    opt = RavenAdamW([{"params": [p for p in unet.parameters() if p.requires_grad], "lr_scale": 1.0}], lr=8e-7,
                     momentum_dtype=BF16, **bench.Cfg.RAVEN)
    batch = {k: v.cuda() for k, v in bench.synth_batch(args.batch, (args.res, args.res), 100).items()}
    rows = []
    for rnd in range(args.rounds):
        for ga in (1, 4):
            cfg = type("C", (bench.Cfg,), dict(BATCH_SIZE=args.batch, GRADIENT_ACCUMULATION_STEPS=ga, MAX_TRAIN_STEPS=10 ** 6,
                                                   PREDICTION_TYPE="epsilon", TIMESTEP_ALLOCATION=None))
            step = SDXLTrainStep(unet, opt, cfg, use_cuda_graph=True)
            for _ in range(3 * ga + 4):                     # per phase: two eager warm-ups, the capture, replays
                step.step(batch)
            while step.micro_step % 4:                      # start the timed run on a window boundary
                step.step(batch)
            n = args.steps
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(n + 1)]
            last = []
            torch.cuda.synchronize()
            ev[0].record()
            for i in range(n):
                last.append(step.step(batch).did_optimizer_step)
                ev[i + 1].record()
            torch.cuda.synchronize()
            ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(n)]
            tot = sum(ms)
            ms_last = [m for m, d in zip(ms, last) if d]
            ms_other = [m for m, d in zip(ms, last) if not d]
            line = (f"round {rnd} GA={ga}: {args.batch * n / tot * 1e3:.3f} imgs/s, {tot / n:.2f} ms per micro-step; last "
                    f"{sum(ms_last) / len(ms_last):.2f} ms (n={len(ms_last)})")
            if ms_other:
                line += f", non-last {sum(ms_other) / len(ms_other):.2f} ms (n={len(ms_other)})"
            print(line, flush=True)
            rows.append((ga, tot / n))
            step._graphs.clear()
            del step
            gc.collect()
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--batch", type=int, default=4)
    ap.add_argument("--res", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--no-step", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("grad_accum_bench.py needs a CUDA device")
    print("card:", card(), flush=True)
    kernel_alone(args.reps)
    if not args.no_step:
        step_ab(args)


if __name__ == "__main__":
    main()
