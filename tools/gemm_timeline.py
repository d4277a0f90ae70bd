"""Where one GEMM launch spends its time: clock64 stamps of CTA 0 (debug flag 64) -- kernel entry, prologue done, dependency wait
done, first TMA issued, first operands landed, last MMA committed, accumulator complete (epilogue starts), each epilogue warp done,
teardown -- next to the kernel duration CUPTI reports.      python tools/gemm_timeline.py"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from aozora_sdxl_training_b200 import _lib, ops  # noqa: E402
from tools.gemm_wide_bench import call_us  # noqa: E402

BF = torch.bfloat16
NAMES = ["entry", "prologue", "dep_wait", "tma0", "data0", "mma_done_issue", "acc_ready"]


def main():
    M, N = 4096, 1280
    lines = []
    for K, b_mn, fused, wide in ((1280, False, True, 2), (1280, False, True, 0), (1280, True, False, 2), (320, False, True, 2),
                                 (320, False, False, 2), (5120, False, True, 2)):
        x = torch.randn(M, K, device="cuda").to(BF)
        w = ((torch.randn(K, N, device="cuda") if b_mn else torch.randn(N, K, device="cuda")) * 0.02).to(BF)
        bias = torch.zeros(N, device="cuda", dtype=BF)
        res = torch.randn(M, N, device="cuda").to(BF)
        out = torch.empty(M, N, device="cuda", dtype=BF)
        fn = (lambda: ops.gemm(x, w, b_mn=b_mn, bias=bias, residual=res, out=out)) if fused else (lambda: ops.gemm(x, w, b_mn=b_mn, out=out, splits=1))
        _lib.call("aoz_gemm_set_wide_mode", wide)
        _lib.call("aoz_gemm_set_tail_mode", 0)
        us = call_us(fn)
        scratch = ops._gemm_scratch[torch.cuda.current_device()]
        scratch[:512].zero_()
        _lib.call("aoz_gemm_debug_flags", 64)
        fn()
        torch.cuda.synchronize()
        _lib.call("aoz_gemm_debug_flags", 0)
        t = scratch[:512].view(torch.int64).cpu().tolist()
        t0 = t[0]
        parts = [f"{n}={t[i] - t0}" for i, n in enumerate(NAMES) if t[i]]
        epi = [t[8 + wp] - t0 for wp in range(2, 10) if t[8 + wp]]
        plan = _lib.query("aoz_gemm_describe_plan", M, N, K, int(b_mn), 1)
        line = (f"K={K} b_mn={int(b_mn)} fused={int(fused)} wide={wide} plan={plan} kernel {us} us | cycles from entry: " + " ".join(parts) +
                f" epilogue_warps_done={min(epi)}..{max(epi)} teardown={t[7] - t0}")
        print(line, flush=True)
        lines.append(line)
    _lib.call("aoz_gemm_set_wide_mode", 1)
    _lib.call("aoz_gemm_set_tail_mode", 1)
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    open(os.path.join(ROOT, "gpurun_out", "gemm_timeline.txt"), "w").write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
