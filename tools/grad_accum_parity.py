"""Gradient accumulation under data parallel on real GPUs (run under torchrun, 2+ ranks): N ranks x b samples with
GRADIENT_ACCUMULATION_STEPS = 2 must reproduce ONE process with BATCH_SIZE = N*b and the same accumulation (tools/dp_parity.py does
the same for GA = 1).  Every micro-step's loss is compared, the gradient norm on every optimizer step, the weights at the end.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29512 \
        tools/grad_accum_parity.py [--graph] [--defer]
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

BF16 = torch.bfloat16


class Cfg:
    SEED = 42
    MAX_TRAIN_STEPS = 10
    GRADIENT_ACCUMULATION_STEPS = 2
    CLIP_GRAD_NORM = 1.0
    PREDICTION_TYPE = "rectified_flow"
    TIMESTEP_ALLOCATION = None
    TIMESTEP_STRATIFIED_SAMPLING = False
    TIMESTEP_LOSS_WEIGHT_CURVE = None
    LR_CUSTOM_CURVE = [[0.0, 2e-5], [1.0, 1e-5]]        # small enough that bf16 summation-order noise is not amplified step to step


def batch_for(seed, B):
    g = torch.Generator().manual_seed(seed)
    return dict(latents=(torch.randn(B, 4, 16, 16, generator=g) * 0.8).to(BF16), embeds=torch.randn(B, 77, 128, generator=g).to(BF16),
                pooled=torch.randn(B, 64, generator=g).to(BF16), time_ids=[[1024, 1024, 0, 0, 1024, 1024]] * B)


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    from aozora_sdxl_training_b200.optimizers import RavenAdamW
    from aozora_sdxl_training_b200.parallel import DataParallel
    from aozora_sdxl_training_b200.trainer import SDXLTrainStep
    from aozora_sdxl_training_b200.unet import UNet2DConditionModel, init_weights_, tiny_config
    b = 2
    B = b * world
    hp = dict(lr=2e-5, betas=(0.9, 0.999), weight_decay=0.01, eps=1e-8, debias_strength=0.3)
    cfg = type("C", (Cfg,), dict(BATCH_SIZE=B))
    # data-parallel run
    m_dp = init_weights_(UNet2DConditionModel(tiny_config()), seed=7, std=0.05).to(BF16).to(dev)
    defer = "--defer" in sys.argv            # all-gather of the updated parameters deferred into the next step's forward pass
    dp = DataParallel(m_dp, momentum_dtype=torch.float32, defer_all_gather=defer)
    opt_dp = dp.make_optimizer(**hp)
    use_graph = "--graph" in sys.argv
    step_dp = SDXLTrainStep(m_dp, opt_dp, cfg, device=dev, dp=dp, use_cuda_graph=use_graph, graph_warmup=2)
    # single-process run with the global batch (every rank does the same thing; rank 0 reports)
    m_1 = init_weights_(UNet2DConditionModel(tiny_config()), seed=7, std=0.05).to(BF16).to(dev)
    opt_1 = RavenAdamW([{"params": list(m_1.parameters()), "lr_scale": 1.0}], momentum_dtype=torch.float32, **hp)
    step_1 = SDXLTrainStep(m_1, opt_1, cfg, device=dev)
    ok = True
    for i in range(12 if use_graph else 6):      # graph: per phase two eager warm-ups, the capture, then replays
        full = batch_for(100 + i, B)
        mine = {k: (v[rank * b:(rank + 1) * b] if torch.is_tensor(v) else v[rank * b:(rank + 1) * b]) for k, v in full.items()}
        r_dp = step_dp.step(mine)
        r_1 = step_1.step(full)
        l_dp = r_dp.loss.clone()
        dist.all_reduce(l_dp)                               # per-rank losses are normalised by the global count: they add up
        rel = abs(l_dp.item() - r_1.loss.item()) / abs(r_1.loss.item())
        ok = ok and rel < 3e-3 and r_dp.did_optimizer_step == r_1.did_optimizer_step == (i % 2 == 1)
        msg = f"micro-step {i}: loss dp {l_dp.item():.6f} single {r_1.loss.item():.6f} rel {rel:.2e}"
        if r_1.did_optimizer_step:
            gn_rel = abs(r_dp.grad_norm[0].item() - r_1.grad_norm[0].item()) / r_1.grad_norm[0].item()
            ok = ok and gn_rel < 3e-2
            msg += f" | optimizer step, grad norm rel {gn_rel:.2e}"
        if rank == 0:
            print(msg, flush=True)
    dp.gather_params()                        # deferred mode: the last update's slices are gathered on demand
    num = sum(float((a.detach().float() - c.detach().float()).abs().sum()) for a, c in zip(m_dp.parameters(), m_1.parameters()))
    den = sum(float(c.detach().float().abs().sum()) for c in m_1.parameters())
    moved = sum(float((c.detach().float() - init_weights_(UNet2DConditionModel(tiny_config()), seed=7, std=0.05).to(BF16).state_dict()[n].to(dev).float()).abs().sum())
                for n, c in m_1.named_parameters())
    if rank == 0:
        print(f"param diff / |param| = {num / den:.3e}; update size / |param| = {moved / den:.3e}", flush=True)
    ok = ok and num / den < 0.15 * max(moved / den, 1e-6)      # Adam-style updates: sign flips of near-zero gradients dominate
    t = torch.tensor([1.0 if ok else 0.0], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("GA=2 DP PARITY", "(deferred all-gather)" if defer else "", "(graph)" if use_graph else "(eager)", "OK" if t.item() == 1.0 else "FAILED", flush=True)
    dist.barrier()
    torch.cuda.synchronize()
    code = 0 if t.item() == 1.0 else 1
    sys.stdout.flush()
    os._exit(code)            # captured NCCL graphs make destroy_process_group hang at exit; the processes have nothing left to do


if __name__ == "__main__":
    main()
