"""Attention forward / backward: correctness against fp32 SDPA and CUDA-event timing at the SDXL shapes; --bwd-modes times the
backward forms of aoz_attn_set_bwd_mode (2 = one kernel, 0 = dK/dV + dQ kernels).
    python tools/attn_bench.py [--bwd-modes 2,0] [--out PATH]"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from aozora_sdxl_training_b200 import _lib, ops  # noqa: E402

BF = torch.bfloat16
SHAPES = [("self_4096x10", 4, 10, 4096, 4096), ("self_1024x20", 4, 20, 1024, 1024), ("cross_4096x10", 4, 10, 4096, 77),
          ("cross_1024x20", 4, 20, 1024, 77), ("tail_4032x10", 1, 10, 4032, 4032), ("tail_988x20", 1, 20, 988, 988)]


def timeit(fn, n=20):
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bwd-modes", default="")
    ap.add_argument("--out", default=os.path.join(ROOT, "gpurun_out", "attn_bench.json"))
    args = ap.parse_args()
    bwd_modes = [int(m) for m in args.bwd_modes.split(",") if m != ""]
    res = {}
    g = torch.Generator(device="cuda").manual_seed(7)
    for name, B, H, T, Tk in SHAPES:
        q, do = [torch.randn(B, T, H, 64, device="cuda", generator=g).to(BF) for _ in range(2)]
        k, v = [torch.randn(B, Tk, H, 64, device="cuda", generator=g).to(BF) for _ in range(2)]
        qr, kr, vr = [t.float().permute(0, 2, 1, 3).requires_grad_(True) for t in (q, k, v)]
        ref = torch.nn.functional.scaled_dot_product_attention(qr, kr, vr, scale=0.125)
        ref.backward(do.float().permute(0, 2, 1, 3))
        ref = ref.detach().permute(0, 2, 1, 3)
        f = 4.0 * B * H * T * Tk * 64
        o, lse = ops.attn_fwd(q, k, v, 0.125)
        torch.cuda.synchronize()
        err = (o.float() - ref).abs().max().item() / ref.abs().max().item()
        cos = torch.nn.functional.cosine_similarity(o.float().flatten(), ref.flatten(), dim=0).item()
        ms = timeit(lambda: ops.attn_fwd(q, k, v, 0.125))
        res[f"{name}_fwd"] = dict(us=round(ms * 1e3, 1), tflops=round(f / ms / 1e9, 1), rel_err=round(err, 5), cos=round(cos, 6))
        print(name, "fwd", res[f"{name}_fwd"], flush=True)
        for m in (bwd_modes or [None]):
            if m is not None:
                _lib.call("aoz_attn_set_bwd_mode", m)
            try:
                dq, dk, dv = ops.attn_bwd(q, k, v, o, do, lse, 0.125)
                torch.cuda.synchronize()
                errs = []
                for got, want in ((dq, qr.grad), (dk, kr.grad), (dv, vr.grad)):
                    want = want.permute(0, 2, 1, 3)
                    errs.append(round((got.float() - want).abs().max().item() / want.abs().max().item(), 5))
                ms = timeit(lambda: ops.attn_bwd(q, k, v, o, do, lse, 0.125))
                res[f"{name}_bwd_mode{m}"] = dict(us=round(ms * 1e3, 1), tflops=round(2.5 * f / ms / 1e9, 1), rel_err_dq_dk_dv=errs)
            except Exception as e:
                res[f"{name}_bwd_mode{m}"] = dict(error=str(e)[:200])
            print(name, "bwd mode", m, res[f"{name}_bwd_mode{m}"], flush=True)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
