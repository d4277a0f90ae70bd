#!/usr/bin/env python
"""bench.py -- SDXL 1024x1024 UNet training-step throughput on N B200s (BASELINE.json metric), one JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--batch B] [--mode v_prediction] [--dump-outputs DIR]

Own arm: ``SDXLTrainStep.step`` (aozora_sdxl_training_b200/trainer.py) on synthetic SDXL-shaped batches and random-init
weights of the exact SDXL UNet layout: noising -> UNet fwd -> weighted MSE -> reverse sweep -> clip -> Raven update,
every step, nothing skipped.  ``value`` = imgs/s with inputs resident in HBM; ``e2e`` = the same call fed from pinned
HOST buffers (H2D of latents / text embeddings inside the timed region) with the loss read back to the host each step.
``roofline`` = the dominant kernel (the tcgen05 GEMM, at the GEGLU feed-forward shape) timed live with CUDA events.
``cpu_baseline`` / ``--impl reference`` = the reference's step semantics on the box's host cores through the CPU oracle
(oracle/train_step_ref.py; the UNet arithmetic is diffusers', restated -- kind "port") at BASELINE config 1 (512x512, batch 1,
epsilon, fp32), split into fwd+bwd / clip / Raven, best of >= 3 steps, no rescaling.  ``--workload 3 | 4`` select BASELINE
configs 3 (rectified flow, logit-normal tickets, batch 8/GPU) and 4 (layer exclusion over three aspect-ratio buckets).
``--dump-outputs DIR`` writes what the own arm's last timed step computed as DIR/<name>.npy (see ``dump_outputs``); inputs and
weights are seeded, so two builds run with the same arguments can be compared output for output.  Compare with a tolerance: the
attention backward adds dQ partial tiles into fp32 in arrival order, so two runs of one build agree to rounding, not bit for bit.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NCCL_CTAS_DEFAULT = 0                # data parallel: CTAs (and SMs) reserved for NCCL; see --nccl-ctas
TRAIN_TFLOP_PER_IMG = 20.28          # fwd + dgrad + wgrad at 1024x1024, SURVEY.md 8d (recompute not counted)


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf_sust=p["bf16_tflops_sustained"], src="measured")
    except Exception:
        return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


class Cfg:
    SEED = 42
    MAX_TRAIN_STEPS = 1000
    GRADIENT_ACCUMULATION_STEPS = 1
    CLIP_GRAD_NORM = 1.0
    TIMESTEP_STRATIFIED_SAMPLING = False
    TIMESTEP_LOSS_WEIGHT_CURVE = None
    LR_CUSTOM_CURVE = [[0.0, 0.0], [0.05, 8.0e-7], [0.85, 8.0e-7], [1.0, 1.0e-7]]
    RAVEN = dict(betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01, debias_strength=0.3)


def synth_batch(b, res, seed, device="cpu", pin=False):
    """``res``: side of a square image or a (width, height) bucket; latents [b, 4, height/8, width/8], time_ids as train.py:2726-2731."""
    import torch
    g = torch.Generator().manual_seed(seed)
    wpx, hpx = (res, res) if isinstance(res, int) else res
    out = dict(latents=(torch.randn(b, 4, hpx // 8, wpx // 8, generator=g) * 0.8).to(torch.bfloat16),
               embeds=torch.randn(b, 77, 2048, generator=g).to(torch.bfloat16),
               pooled=torch.randn(b, 1280, generator=g).to(torch.bfloat16),
               time_ids=torch.tensor([[hpx, wpx, 0, 0, hpx, wpx]] * b, dtype=torch.bfloat16))
    if device != "cpu":
        out = {k: v.to(device) for k, v in out.items()}
    elif pin:
        out = {k: v.pin_memory() for k, v in out.items()}
    return out


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], None, set()
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return dict(sm_mhz=(sm[len(sm) // 2] if sm else None), sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))


def gemm_roofline(torch, peaks, iters=20):
    """Dominant kernel timed live: gemm_bf16_kernel at the GEGLU feed-forward shape (M = 4 x 32 x 32 tokens, C = 1280)."""
    from aozora_sdxl_training_b200 import ops
    M, K, N = 4096, 1280, 10240
    x = torch.randn(M, K, device="cuda").to(torch.bfloat16)
    w = (torch.randn(N, K, device="cuda") * 0.02).to(torch.bfloat16)
    b = torch.zeros(N, device="cuda", dtype=torch.bfloat16)
    aux = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    out = torch.empty(M, N // 2, device="cuda", dtype=torch.bfloat16)
    flush = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
    for _ in range(3):
        ops.gemm(x, w, bias=b, epi=ops.EPI_GEGLU, aux=aux, out=out)
    torch.cuda.synchronize()
    evs = []
    for _ in range(iters):
        # L2 flush (1 GiB memset) in front of every timed launch; everything is queued before the single synchronize so
        # the GPU never waits for the host between the start event and the kernel
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ops.gemm(x, w, bias=b, epi=ops.EPI_GEGLU, aux=aux, out=out)
        e1.record()
        evs.append((e0, e1))
    torch.cuda.synchronize()
    times = [a.elapsed_time(c) for a, c in evs]
    ms = sum(times) / len(times)
    flops = 2.0 * M * N * K
    ach = flops / (ms * 1e-3) / 1e12
    return dict(bound="tensor", kernel="gemm_bf16_kernel<256> (GEGLU epilogue) M=4096 K=1280 N=10240", achieved=round(ach, 1),
                peak=peaks["tf_burst"], unit="TFLOP/s", frac=round(ach / peaks["tf_burst"], 4),
                # dram__bytes_read.sum + dram__bytes_write.sum of this exact launch from the committed `ncu --set full` capture
                # (algorithmic bytes: 36.7 MB operands + 125.8 MB outputs, part of the output still in L2 when the kernel ends)
                traffic=113185536, traffic_source="profiles/r02_gemm_geglu_ncu_v2.txt (dram__bytes_read 36.92 MB + dram__bytes_write 76.26 MB)",
                peak_source=f"{peaks['src']} bf16_tflops (burst: kernel timed alone)", ms_per_launch=round(ms, 4),
                flops_per_launch=flops,
                # the whole GEMM / conv family inside the step (1211 launches, FLOP-weighted): tools/gemm_in_step.py, recorded once per round
                family_in_step=dict(tflops=946.8, frac_of_burst=round(946.8 / peaks["tf_burst"], 4), ms=75.73, launches=1211,
                                    source="profiles/r02_gemm_in_step_v3.txt (71.70 TFLOP of GEMM / conv work per step in 75.73 ms)"))


def kernel_table(torch, peaks, param_numels=None):
    """Side metrics BASELINE.json names: attention TFLOPS (4096 tok x 10 heads x 64) and Raven step HBM GB/s."""
    from aozora_sdxl_training_b200 import ops
    from aozora_sdxl_training_b200.optimizers import RavenAdamW
    out = {}

    def timeit(fn, n=10):
        for _ in range(2):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    B, H, T = 4, 10, 4096
    q, k, v, do = [torch.randn(B, T, H, 64, device="cuda").to(torch.bfloat16) for _ in range(4)]
    ms = timeit(lambda: ops.attn_fwd(q, k, v, 0.125))
    f = 4.0 * B * H * T * T * 64
    out["attn_fwd_tflops"] = round(f / ms / 1e9, 1)
    o, lse = ops.attn_fwd(q, k, v, 0.125)
    ms = timeit(lambda: ops.attn_bwd(q, k, v, o, do, lse, 0.125))
    out["attn_bwd_tflops"] = round(2.5 * f / ms / 1e9, 1)
    # cross-attention (attn2): 4096 queries x 77 keys x 10 heads x 64 (BASELINE config 5); latency / occupancy bound, one KV tile
    kc, vc = [torch.randn(B, 77, H, 64, device="cuda").to(torch.bfloat16) for _ in range(2)]
    fc = 4.0 * B * H * T * 77 * 64
    ms = timeit(lambda: ops.attn_fwd(q, kc, vc, 0.125), n=20)
    out["cross_attn_fwd_tflops"] = round(fc / ms / 1e9, 1)
    out["cross_attn_fwd_us"] = round(ms * 1e3, 1)
    oc, lsec = ops.attn_fwd(q, kc, vc, 0.125)
    ms = timeit(lambda: ops.attn_bwd(q, kc, vc, oc, do, lsec, 0.125), n=20)
    out["cross_attn_bwd_tflops"] = round(2.5 * fc / ms / 1e9, 1)
    out["cross_attn_bwd_us"] = round(ms * 1e3, 1)
    del q, k, v, do, o, lse, kc, vc, oc, lsec
    if param_numels:
        # Raven over the REAL table: 1680 tensors / 2,567,463,684 parameters, bf16 p, g, m, v (14 B per parameter = 35.9 GB per step)
        ps = [torch.nn.Parameter(torch.zeros(nn_, device="cuda", dtype=torch.bfloat16)) for nn_ in param_numels]
        for p in ps:
            p.grad = torch.full_like(p, 1e-3)
        opt = RavenAdamW(ps, lr=8e-7, **Cfg.RAVEN)
        ms = timeit(lambda: opt.step(), n=5)
        tot = sum(param_numels)
        out["raven_sdxl_table_gbs"] = round(14.0 * tot / ms / 1e6, 1)
        out["raven_sdxl_table_ms"] = round(ms, 3)
        out["raven_sdxl_table_frac_of_hbm"] = round(out["raven_sdxl_table_gbs"] / peaks["hbm"], 4)
        out["raven_sdxl_table"] = f"{len(param_numels)} tensors, {tot} parameters"
        del ps, opt
        torch.cuda.empty_cache()
    n = 512 * 1024 * 1024                                    # 0.5 G parameters in 16 tensors (bounded memory, > L2)
    ps = [torch.nn.Parameter(torch.zeros(n // 16, device="cuda", dtype=torch.bfloat16)) for _ in range(16)]
    for p in ps:
        p.grad = torch.full_like(p, 1e-3)
    opt = RavenAdamW(ps, lr=8e-7, **Cfg.RAVEN)
    ms = timeit(lambda: opt.step(), n=5)
    out["raven_step_gbs"] = round(14.0 * n / ms / 1e6, 1)
    out["raven_frac_of_hbm"] = round(out["raven_step_gbs"] / peaks["hbm"], 4)
    def timeit_graph(fn, n=10):
        """Device time of small kernels: n calls captured in a CUDA graph and replayed (an eager Python loop measures the host:
        three allocations + a ctypes call cost more than a 10-microsecond kernel)."""
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(n):
                fn()
        g.replay()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    # GroupNorm+SiLU forward, 4 B / element: 1280 channels at 32x32 (BASELINE config 5; a 10 MB tensor: latency, not bandwidth)
    # and 320 channels at 128x128 (42 MB per tensor, the size class that holds most of the step's GroupNorm bytes)
    for name, hw, c in (("groupnorm_silu_gbs", 32 * 32, 1280), ("groupnorm_silu_320x128x128_gbs", 128 * 128, 320)):
        x = torch.randn(4, hw, c, device="cuda").to(torch.bfloat16)
        ga, be = torch.ones(c, device="cuda", dtype=torch.bfloat16), torch.zeros(c, device="cuda", dtype=torch.bfloat16)
        ms = timeit_graph(lambda: ops.groupnorm_fwd(x, ga, be, 1e-5, True))
        out[name] = round(4.0 * x.numel() / ms / 1e6, 1)
    x = torch.randn(4096, 1280, device="cuda").to(torch.bfloat16)
    ga, be = torch.ones(1280, device="cuda", dtype=torch.bfloat16), torch.zeros(1280, device="cuda", dtype=torch.bfloat16)
    y, mean, rstd = ops.layernorm_fwd(x, ga, be)
    out["layernorm_fwd_gbs"] = round(4.0 * x.numel() / timeit_graph(lambda: ops.layernorm_fwd(x, ga, be)) / 1e6, 1)
    out["layernorm_bwd_gbs"] = round(6.0 * x.numel() / timeit_graph(lambda: ops.layernorm_bwd(y, x, ga, mean, rstd)) / 1e6, 1)
    return out


def cpu_config1_step(steps, warmup):
    """BASELINE config 1 on the box's host cores, as BASELINE.md section 4 specifies: the reference's step semantics
    (train.py:2719-2784) through the CPU oracle -- random-init full SDXL UNet, 512x512 (latent 4x64x64), batch 1, epsilon, cached-shape
    conditioning, fp32 weights / fp32 Raven moments, autocast off -- timed with perf_counter and split into fwd+bwd / clip / Raven,
    best of ``steps`` (>= 3) after ``warmup`` (>= 1).  All host threads: torchrun exports OMP_NUM_THREADS=1, which is overridden."""
    import torch
    from oracle import host_ref
    from oracle.scheduler_ref import RefDDPMScheduler
    from oracle.train_step_ref import RefRaven, ref_forward_loss
    from oracle.unet_ref import RefUNet2DConditionModel, sdxl_config
    ncpu = os.cpu_count() or 1
    torch.set_num_threads(ncpu)
    res, batch, mode = 512, 1, "epsilon"
    torch.manual_seed(0)
    model = RefUNet2DConditionModel(sdxl_config())
    with torch.no_grad():
        for name, p in model.named_parameters():
            if p.dim() == 1 and name.endswith("weight"):
                p.fill_(1.0)
            elif p.dim() == 1:
                p.zero_()
            else:
                p.normal_(0.0, 0.02)
    params = list(model.parameters())
    # fp32 weights + gradients + fp32 moments = 41 GB (+ activations); a small host keeps the moments in bf16 (SURVEY.md 8d) and says so
    try:
        import psutil
        avail_gb = psutil.virtual_memory().available / 2 ** 30
    except Exception:
        avail_gb = 1e9
    mdt = torch.float32 if avail_gb >= 64 else torch.bfloat16
    opt = RefRaven(params, lr=8e-7, momentum_dtype=mdt, **Cfg.RAVEN)
    sch = RefDDPMScheduler(prediction_type=mode)
    sampler = host_ref.RefTimestepSampler(Cfg.MAX_TRAIN_STEPS, batch, Cfg.SEED, None, False)
    b = synth_batch(batch, res, 1)
    rb = dict(latents=b["latents"], embeds=b["embeds"].float(), pooled=b["pooled"].float(),
              time_ids_data=[[res, res, 0, 0, res, res]] * batch)
    rows = []
    for i in range(warmup + steps):
        ts, _ = sampler.sample(batch)
        t0 = time.perf_counter()
        loss, _, _, _ = ref_forward_loss(model, sch, rb, prediction_type=mode, timesteps=ts, micro_step=i + 1, seed=Cfg.SEED,
                                         compute_dtype=torch.float32, autocast=False)
        loss.backward()
        t1 = time.perf_counter()
        torch.nn.utils.clip_grad_norm_(params, Cfg.CLIP_GRAD_NORM)
        t2 = time.perf_counter()
        opt.step()
        opt.zero_grad(set_to_none=True)
        t3 = time.perf_counter()
        if i >= warmup:
            rows.append((t3 - t0, t1 - t0, t2 - t1, t3 - t2))
    best = min(rows)                                          # best whole step; its own split is reported
    return dict(sec=best[0], fwd_bwd_s=best[1], clip_s=best[2], raven_s=best[3], threads=torch.get_num_threads(), cpus=ncpu,
                steps_timed=len(rows), mean_sec=sum(r[0] for r in rows) / len(rows), loss=float(loss.detach()),
                moments="fp32" if mdt == torch.float32 else "bf16 (host has < 64 GB free)")


DUMP_PER_TENSOR = 2048              # sampled elements per trainable tensor: SDXL's 1680 tensors -> 31 MB in the three float32 arrays


def dump_outputs(out_dir, res, unet, opt, dp, rank):
    """What a caller of ``SDXLTrainStep.step`` holds after the last timed step, as float32 / float64 .npy files: the returned
    ``loss``, ``grad_norm`` (norm, clip coefficient, sum of squares) and ``timesteps``, and the state the step updated in place --
    ``params``, ``exp_avg`` and ``exp_avg_sq`` (Raven moments) -- as a fixed, seeded sample of ``DUMP_PER_TENSOR`` elements of
    every trainable tensor in ``named_parameters`` order (the full state is 15 GB).  Data parallel: every rank takes part in
    gathering the parameters and moments; rank 0 writes."""
    import numpy as np
    import torch
    params = [p for p in unet.parameters() if p.requires_grad]
    if dp is None:
        moments = [(opt.state[p]["exp_avg"].reshape(-1), opt.state[p]["exp_avg_sq"].reshape(-1)) for p in params]
    else:
        dp.gather_params()
        full_m, full_v = dp.gather_shards(opt.m_shard), dp.gather_shards(opt.v_shard)
        moments = [(full_m[o:o + p.numel()], full_v[o:o + p.numel()]) for o, p in zip(dp.layout.offsets, params)]
    if rank != 0:
        return
    g = torch.Generator().manual_seed(0)
    picks = [torch.arange(p.numel()) if p.numel() <= DUMP_PER_TENSOR else torch.randint(p.numel(), (DUMP_PER_TENSOR,), generator=g)
             for p in params]

    def sample(flats):
        return torch.cat([f[i.to(f.device)].float() for f, i in zip(flats, picks)]).cpu().numpy()

    arrays = dict(loss=res.loss.float().cpu().numpy(), grad_norm=res.grad_norm.float().cpu().numpy(),
                  timesteps=res.timesteps.cpu().numpy().astype(np.float64), params=sample([p.detach().reshape(-1) for p in params]),
                  exp_avg=sample([m for m, _ in moments]), exp_avg_sq=sample([v for _, v in moments]))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


CONFIG1 = ("BASELINE config 1: SDXL UNet random-init single train step, epsilon, 512x512 (64x64x4 latents), batch 1, cached 77x2048 "
           "text embeds + 1280 pooled, Raven step, fp32 weights and moments, torch-CPU")


def cpu_baseline_record(r):
    return dict(value=round(1.0 / r["sec"], 6), unit="imgs/s", cores=r["threads"], kind="port",
                sample=(f"{CONFIG1}; best of {r['steps_timed']} steps after warm-up, 1 image of 512x512 per step, no rescaling "
                        f"(the GPU arm's images are 1024x1024: 4x the pixels, so the two imgs/s are not the same unit of work)"),
                seconds_per_step=round(r["sec"], 3), fwd_bwd_s=round(r["fwd_bwd_s"], 3), clip_s=round(r["clip_s"], 3),
                raven_s=round(r["raven_s"], 3), mean_seconds_per_step=round(r["mean_sec"], 3), os_cpu_count=r["cpus"],
                torch_threads=r["threads"], same_config=False, raven_moments=r["moments"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="aozora")
    ap.add_argument("--workload", type=int, default=2, choices=(2, 3, 4),
                    help="BASELINE.json configs[1..3]: 2 = 1024x1024 batch 4 v_prediction (default, the metric's config); "
                         "3 = rectified_flow + logit-normal tickets, batch 8/GPU; 4 = layer exclusion (down_blocks.0, attn2) over "
                         "896x1152 / 1216x832 / 1024x1024 buckets")
    ap.add_argument("--batch", type=int, default=None, help="images per GPU (default: 4; workload 3: 8)")
    ap.add_argument("--res", type=int, default=1024)
    ap.add_argument("--mode", default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-table", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="issue every kernel from Python instead of replaying the captured step")
    ap.add_argument("--nccl-ctas", type=int, default=-1,
                    help="data parallel: cap NCCL at this many CTAs (NCCL_MAX_CTAS) and leave them their own SMs (persistent GEMMs are "
                         "sized to the rest); 0 = NCCL defaults, all SMs to the GEMMs; default: the measured best")
    ap.add_argument("--bucket-mb", type=int, default=512, help="data parallel: gradient reduce-scatter bucket size")
    ap.add_argument("--no-defer-all-gather", action="store_true",
                    help="data parallel: all-gather the updated parameters at the end of the step instead of behind the next forward pass")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32 / float64, < 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU step; the reference arm has none")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    metric = "SDXL 1024x1024 UNet train step throughput"
    if args.batch is None:
        args.batch = 8 if args.workload == 3 else 4
    if args.mode is None:
        args.mode = "rectified_flow" if args.workload == 3 else "v_prediction"
    # (width, height) of the image buckets the steps cycle through (SURVEY.md 8d: config 4 = 896x1152, 1216x832, 1024x1024)
    buckets = [(896, 1152), (1216, 832), (1024, 1024)] if args.workload == 4 else [(args.res, args.res)]
    exclude = ["down_blocks.0", "attn2"] if args.workload == 4 else []
    workload = (f"BASELINE config {args.workload}: SDXL UNet bf16 " + " / ".join(f"{w}x{h}" for w, h in buckets) +
                f" batch {args.batch}/GPU, {args.mode}, " +
                ("logit-normal(-0.5, 1) timestep tickets, " if args.workload == 3 else "uniform timestep tickets, ") +
                (f"exclude keywords {exclude} (frozen: no wgrad / reduce / Raven state), " if exclude else "") +
                "Raven (bf16 moments), cached 77x2048 text embeds + 1280 pooled, random-init weights")

    if args.impl == "reference":
        if rank != 0:
            return
        # Each "step" is one BASELINE config 1 micro-step (the reference's CPU-runnable case) on all host cores; the run is
        # bounded: 1 warm-up + at most 5 timed steps whatever --steps / --warmup ask for (a step takes ~10-20 s of CPU).
        k = max(3, min(args.steps, 5))
        r = cpu_config1_step(k, 1)
        rec = cpu_baseline_record(r)
        line = dict(impl="reference", metric=metric, value=rec["value"], unit="imgs/s", n_gpus=args.gpus, steps=args.steps,
                    warmup=args.warmup, ms_per_step=r["sec"] * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                    data="synthetic", config=dict(workload=CONFIG1, same_config=False, steps_timed=k, warmup_run=1,
                                                  own_arm_workload=workload), gpu_launches=0, cpu_baseline=rec,
                    e2e=dict(value=rec["value"], unit="imgs/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
        print(json.dumps(line))
        return

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: CUDA device required (aozora-b200 has no CPU path; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dp = None
    nccl_ctas = args.nccl_ctas if args.nccl_ctas >= 0 else NCCL_CTAS_DEFAULT
    if world > 1:
        import torch.distributed as dist
        if nccl_ctas > 0:                                  # read by NCCL when the communicator is created
            os.environ["NCCL_MAX_CTAS"] = str(nccl_ctas)
            os.environ["NCCL_MIN_CTAS"] = str(min(nccl_ctas, int(os.environ.get("NCCL_MIN_CTAS", nccl_ctas))))
        dist.init_process_group("nccl", device_id=dev)
    from aozora_sdxl_training_b200 import ops
    from aozora_sdxl_training_b200.optimizers import RavenAdamW
    from aozora_sdxl_training_b200.trainer import SDXLTrainStep
    from aozora_sdxl_training_b200.unet import UNet2DConditionModel, init_weights_fast_, sdxl_config
    peaks = load_peaks()
    if world > 1 and nccl_ctas > 0:
        from aozora_sdxl_training_b200 import _lib as _l
        _l.call("aoz_gemm_set_sm_budget", _l.query("aoz_sm_count") - nccl_ctas)

    from aozora_sdxl_training_b200 import host
    with torch.device(dev):
        unet = UNet2DConditionModel(sdxl_config()).to(torch.bfloat16)
    init_weights_fast_(unet, seed=Cfg.SEED)
    frozen = host.apply_exclusion(unet, exclude) if exclude else 0            # train.py:2664-2667
    # config 3: the GUI's logit-normal recipe (gui/gui.py:5594-5603) for TIMESTEP_ALLOCATION; otherwise uniform bins
    alloc = host.logit_normal_allocation(-0.5, 1.0, Cfg.MAX_TRAIN_STEPS) if args.workload == 3 else None
    cfg = type("BenchCfg", (Cfg,), dict(BATCH_SIZE=args.batch * world, PREDICTION_TYPE=args.mode, TIMESTEP_ALLOCATION=alloc))
    if world > 1:
        from aozora_sdxl_training_b200.parallel import DataParallel
        dp = DataParallel(unet, momentum_dtype=torch.bfloat16, defer_all_gather=not args.no_defer_all_gather, bucket_mb=args.bucket_mb)
        opt = dp.make_optimizer(lr=8e-7, **Cfg.RAVEN)
    else:
        opt = RavenAdamW([{"params": [p for p in unet.parameters() if p.requires_grad], "lr_scale": 1.0}], lr=8e-7,
                         momentum_dtype=torch.bfloat16, **Cfg.RAVEN)
    param_numels = [p.numel() for p in unet.parameters()]
    # the device side of the step (NCCL reduce-scatter / all-gather included) is captured once per batch shape and replayed
    use_graph = not args.no_graph
    step = SDXLTrainStep(unet, opt, cfg, device=dev, dp=dp, use_cuda_graph=use_graph)

    host_batches = [synth_batch(args.batch, wh, 100 + rank + 1000 * i, pin=True) for i, wh in enumerate(buckets)]
    dev_batches = [{k: v.to(dev) for k, v in hb.items()} for hb in host_batches]
    nb = len(buckets)
    h2d = sum(v.numel() * v.element_size() for hb in host_batches for v in hb.values()) // nb     # mean over the bucket cycle

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
        return ms.item()

    from aozora_sdxl_training_b200 import _lib
    per_shape_launches = []
    for db in dev_batches:
        r = step.step(db)                                      # first eager step of this shape: sizes workspaces, GEMM tile plans
        l0 = _lib.query("aoz_launch_count")                    # counted inside the library at every kernel launch site
        r = step.step(db)                                      # second eager step: its launches are what the graph replays
        per_shape_launches.append(_lib.query("aoz_launch_count") - l0)
    # untimed steps: the requested warm-up (>= 3) plus the capture call and a few replays per shape -- under data parallel the first
    # replays of the captured NCCL kernels still run slower than steady state (8 GPUs: 171 ms vs 157 ms per step)
    n_warm = (max(3, args.warmup) + (6 if use_graph else 1) + (12 if (use_graph and world >= 4) else 0)) * nb
    for i in range(n_warm):
        r = step.step(dev_batches[i % nb])
    loss0 = r.loss_value()
    clocks = ClockSampler(local_rank)
    clocks.start()
    ms_dev = timed(lambda i: step.step(dev_batches[i % nb]), args.steps)
    launches = sum(per_shape_launches[i % nb] for i in range(args.steps))      # replayed from the captured graphs
    clk = clocks.stop()

    last = {}

    def e2e_step(i):
        res = last["res"] = step.step(host_batches[i % nb])
        return res.loss_value()                                 # device -> host read of the step's loss

    def timed_wall(fn, n):
        """End-to-end: host wall clock around the user-facing calls (pinned-host inputs in, loss value out), max over ranks."""
        barrier()
        t0 = time.perf_counter()
        for i in range(n):
            fn(i)
        torch.cuda.synchronize()
        ms = torch.tensor([(time.perf_counter() - t0) * 1e3], device=dev)
        barrier()
        if world > 1:
            torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
        return ms.item()

    e2e_step(0)
    ms_e2e = timed_wall(e2e_step, args.steps)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last["res"], unet, opt, dp, rank)

    imgs = args.batch * world * args.steps
    value = imgs / (ms_dev * 1e-3)
    e2e_val = imgs / (ms_e2e * 1e-3)
    line = dict(metric=metric, value=round(value, 3), unit="imgs/s", n_gpus=world, steps=args.steps, warmup=max(3, args.warmup),
                ms_per_step=round(ms_dev / args.steps, 3), higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16",
                data="synthetic",
                config=dict(workload=workload, global_batch=args.batch * world,
                            parallelism=f"dp{world}" + ("" if world == 1 else (" (sharded Raven; parameter all-gather behind the next forward pass)"
                                                                               if not args.no_defer_all_gather else " (sharded Raven)")),
                            l2="per-step working set (5.1 GB weights + activations) far exceeds the 126 MB L2; no explicit flush",
                            recompute="none (all activations kept in HBM)",
                            launch="CUDA graph replay of the captured step" if use_graph else "eager",
                            untimed_steps=n_warm + 2, **({"nccl_ctas": nccl_ctas} if world > 1 else {})),
                e2e=dict(value=round(e2e_val, 3), unit="imgs/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=4,
                         ms_per_step=round(ms_e2e / args.steps, 3),
                         how="SDXLTrainStep.step(batch in pinned host memory) + loss_value() per step, host wall clock"),
                gpu_launches=int(launches), clocks=clk, loss=loss0)
    if args.workload != 4:      # 20.28 TFLOP per 1024x1024 image, every weight gradient included (workload 4 freezes 21 % of them)
        tf = value * TRAIN_TFLOP_PER_IMG * (args.res / 1024) ** 2 / world
        line.update(step_tflops=round(tf, 1), step_frac_of_sustained_bf16_peak=round(tf / peaks["tf_sust"], 4))
    else:
        line["config"].update(frozen_params=int(frozen), buckets=[f"{w}x{h}" for w, h in buckets])
    # teardown order matters under data parallel: the captured graphs hold NCCL kernels, so they go first, then the step
    # object and the optimizer shards, and only then the process group (see the end of main)
    step._graphs.clear()
    del step, opt, dp, unet, dev_batches
    import gc
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    if rank == 0:
        line["roofline"] = gemm_roofline(torch, peaks)
        if not args.no_kernel_table:
            try:
                line["kernels"] = kernel_table(torch, peaks, param_numels)
            except Exception as e:                              # side table must never take the headline down
                line["kernels"] = dict(error=str(e)[:200])
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_record(cpu_config1_step(3, 1))
        else:
            line["cpu_baseline"] = None
        print(json.dumps(line))
        sys.stdout.flush()
    if world > 1:
        # graphs are gone (above); a watchdog keeps a wedged communicator from turning a finished measurement into a hung job
        import threading
        dog = threading.Timer(60.0, lambda: os._exit(0))
        dog.daemon = True
        dog.start()
        torch.distributed.barrier()
        torch.cuda.synchronize()
        torch.distributed.destroy_process_group()
        dog.cancel()


if __name__ == "__main__":
    main()
