"""How far do two VALID variants of the product drift apart over the 50-step loss curve of tests/test_gpu_fullsize.py?  The same
training run (tiny config, lr 1e-4, bf16 weights, fp32 moments) is executed with the default kernels and with the round-1 attention
backward (two-kernel form, aoz_attn_set_bwd_mode(0)): the two differ only in rounding order, and both pass every parity test.
Their mutual deviation is the noise floor of any free-running comparison at this learning rate.  profiles/r02_loss_curve_variants.txt
was recorded when the round-1 variant also ran the split-statistics attention forward, since removed.
    python tools/loss_curve_variants.py [epsilon|v_prediction|rectified_flow]"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from aozora_sdxl_training_b200 import _lib  # noqa: E402
from aozora_sdxl_training_b200.optimizers import RavenAdamW  # noqa: E402
from aozora_sdxl_training_b200.trainer import SDXLTrainStep  # noqa: E402
from aozora_sdxl_training_b200.unet import UNet2DConditionModel, init_weights_, tiny_config  # noqa: E402
from oracle import host_ref  # noqa: E402

BF16 = torch.bfloat16


def run(mode, bwd_mode, steps=50):
    _lib.call("aoz_attn_set_bwd_mode", bwd_mode)
    prod = init_weights_(UNet2DConditionModel(tiny_config()), seed=42, std=0.05).to(BF16).cuda()

    class Cfg:
        SEED = 42
        BATCH_SIZE = 2
        MAX_TRAIN_STEPS = steps
        GRADIENT_ACCUMULATION_STEPS = 1
        CLIP_GRAD_NORM = 1.0
        PREDICTION_TYPE = mode
        TIMESTEP_ALLOCATION = None
        TIMESTEP_STRATIFIED_SAMPLING = False
        TIMESTEP_LOSS_WEIGHT_CURVE = None
        LR_CUSTOM_CURVE = [[0.0, 1e-4], [1.0, 1e-4]]

    hp = dict(lr=1e-4, betas=(0.9, 0.999), weight_decay=0.01, eps=1e-8, debias_strength=0.3, momentum_dtype=torch.float32)
    opt = RavenAdamW([{"params": list(prod.parameters()), "lr_scale": 1.0}], **hp)
    step = SDXLTrainStep(prod, opt, Cfg)
    batches = []
    for s in range(4):
        g = torch.Generator().manual_seed(100 + s)
        batches.append(dict(latents=(torch.randn(2, 4, 16, 16, generator=g) * 0.8).to(BF16), embeds=torch.randn(2, 77, 128, generator=g).to(BF16),
                            pooled=torch.randn(2, 64, generator=g).to(BF16), time_ids=[[1024, 1024, 0, 0, 1024, 1024]] * 2))
    out = []
    for micro in range(1, steps + 1):
        b = batches[micro % 4]
        res = step.step(b, noise=host_ref.step_noise(b["latents"].shape, Cfg.SEED, micro), jitter=host_ref.rf_jitter(2, Cfg.SEED, micro))
        out.append(res.loss_value())
    return torch.tensor(out)


def main():
    mode = sys.argv[1] if len(sys.argv) > 1 else "epsilon"
    a = run(mode, 2)
    b = run(mode, 0)
    a2 = run(mode, 2)
    rel = (a - b).abs() / b
    win = (a.view(5, 10).mean(1) / b.view(5, 10).mean(1) - 1).abs()
    rel2 = (a - a2).abs() / a
    print(f"[{mode}] default kernels vs round-1 attention backward: step max {rel.max():.3f}, mean {rel.mean():.4f}, window max {win.max():.4f}; "
          f"default vs default again (fp32 reduce-add order only): step max {rel2.max():.3f}, mean {rel2.mean():.4f}")
    print("default :", [round(x, 3) for x in a.tolist()])
    print("round-1 :", [round(x, 3) for x in b.tolist()])
    _lib.call("aoz_attn_set_bwd_mode", 2)


if __name__ == "__main__":
    main()
