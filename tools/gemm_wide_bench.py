"""The 320-wide one-wave plan against the ordinary plans on the 4096 x 1280 x K projection shapes of the step: device time of every
kernel a call launches (GEMM + tail fix-up), median over calls, L2-warm and with a 256 MB flush between calls (weights cold, as in
the step).      python tools/gemm_wide_bench.py"""
import collections
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

from aozora_sdxl_training_b200 import _lib, ops  # noqa: E402

BF = torch.bfloat16


def call_us(fn, n=8, interleave=None):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as p:
        for _ in range(n):
            if interleave is not None:
                interleave()
            fn()
        torch.cuda.synchronize()
    tot = collections.defaultdict(float)
    for ev in p.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA and ("gemm_bf16" in ev.name or "tail_fixup" in ev.name or "splitk" in ev.name):
            tot[ev.name.split("(")[0]] += ev.device_time
    return round(sum(tot.values()) / n, 1)


def main():
    big = torch.empty(64 << 20, device="cuda", dtype=torch.float32)
    flush = lambda: big.zero_()
    rows = []
    _lib.call("aoz_gemm_set_wide_max_rounds", 2)
    for M, N, K, b_mn, fused in ((4096, 1280, 1280, False, True), (4096, 1280, 1280, True, False), (4096, 1280, 5120, False, True),
                                 (4096, 1280, 3840, True, False), (4096, 1280, 10240, True, False), (4096, 1280, 320, False, True),
                                 # two rounds of wide tiles (aoz_gemm_set_wide_max_rounds(2)): the 640-channel level and batch 8
                                 (16384, 640, 640, False, True), (16384, 640, 640, True, False), (16384, 640, 2560, False, True),
                                 (16384, 640, 5120, True, False), (16384, 640, 1920, True, False), (8192, 1280, 1280, False, True),
                                 (8192, 1280, 1280, True, False), (8192, 1280, 5120, False, True)):
        x = torch.randn(M, K, device="cuda").to(BF)
        w = ((torch.randn(K, N, device="cuda") if b_mn else torch.randn(N, K, device="cuda")) * 0.02).to(BF)
        bias = torch.zeros(N, device="cuda", dtype=BF)
        res = torch.randn(M, N, device="cuda").to(BF)
        out = torch.empty(M, N, device="cuda", dtype=BF)
        fn = (lambda: ops.gemm(x, w, b_mn=b_mn, bias=bias, residual=res, out=out)) if fused else (lambda: ops.gemm(x, w, b_mn=b_mn, out=out))
        row = {"M": M, "N": N, "K": K, "b_mn": int(b_mn), "fused": int(fused)}
        for mode in (0, 2):
            _lib.call("aoz_gemm_set_wide_mode", mode)
            row[f"wide{mode}_warm_us"] = call_us(fn)
            row[f"wide{mode}_cold_us"] = call_us(fn, interleave=flush)
        _lib.call("aoz_gemm_set_wide_mode", 1)
        row["tflops_cold"] = [round(2.0 * M * N * K / row[f"wide{m}_cold_us"] * 1e-6, 1) for m in (0, 2)]
        rows.append(row)
        print(row, flush=True)
    _lib.call("aoz_gemm_set_wide_max_rounds", 2)
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    json.dump(rows, open(os.path.join(ROOT, "gpurun_out", "gemm_wide_bench.json"), "w"), indent=1)


if __name__ == "__main__":
    main()
