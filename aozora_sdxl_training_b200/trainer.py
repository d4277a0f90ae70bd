"""The SDXL micro-step of the reference (train.py:2719-2784) as one fused B200 pipeline.

``SDXLTrainStep.step(batch)`` does, with hand-written sm_100a kernels only and no host synchronisation:

  host->device copy of the cached batch (train.py:2719-2721) -> tickets (2733) -> seeded noise (2735-2742) ->
  noising + target in one kernel (2743-2758) -> UNet forward (2760) -> weighted MSE + dL/dpred in one kernel
  (2763, 2765) -> explicit reverse sweep (2765) -> [data-parallel: bucketed gradient reduce-scatter over NCCL,
  overlapped with the sweep] -> gradient norm + clip coefficient on device (2772-2781) -> Raven update with the
  coefficient applied in-kernel (2783) -> zero_grad (2784) -> LR curve (2769).

The reference synchronises three times per micro-step (``loss.item()``, the clip norm ``.item()``, the sigma print);
here the loss and the norm stay device tensors and are read back only when the caller asks (``result.loss_value()``).
"""
from __future__ import annotations

from dataclasses import dataclass

import torch

from . import _lib, host, ops
from .optimizers.raven import MultiTensorPlan, _Staging
from .scheduler import DDPMScheduler

BF16 = torch.bfloat16


@dataclass
class StepResult:
    loss: torch.Tensor                 # device fp32 [1]
    grad_norm: torch.Tensor | None     # device fp32 [3] (norm, clip coefficient, sum of squares) on optimizer steps
    timesteps: torch.Tensor
    did_optimizer_step: bool
    lr: float

    def loss_value(self) -> float:
        return float(self.loss.item())

    def grad_norm_value(self) -> float:
        return float(self.grad_norm[0].item()) if self.grad_norm is not None else float("nan")


class SDXLTrainStep:
    """One object per training run.  ``config`` carries the reference's flat keys (SURVEY.md section 5): SEED,
    BATCH_SIZE (global batch), MAX_TRAIN_STEPS, GRADIENT_ACCUMULATION_STEPS, CLIP_GRAD_NORM, PREDICTION_TYPE,
    TIMESTEP_ALLOCATION, TIMESTEP_STRATIFIED_SAMPLING, TIMESTEP_LOSS_WEIGHT_CURVE, LR_CUSTOM_CURVE."""

    def __init__(self, unet, optimizer, config, *, device="cuda", dp=None, use_cuda_graph=False, graph_warmup=2):
        self.unet = unet
        self.optimizer = optimizer
        self.config = config
        self.device = torch.device(device)
        self.dp = dp                                    # parallel.DataParallel or None
        self.world = 1 if dp is None else dp.world
        self.rank = 0 if dp is None else dp.rank
        self.prediction_type = getattr(config, "PREDICTION_TYPE", "epsilon")
        self.is_rf = self.prediction_type == "rectified_flow"
        self.seed = config.SEED if config.SEED else 42
        self.grad_accum = max(1, int(getattr(config, "GRADIENT_ACCUMULATION_STEPS", 1)))
        self.clip = float(getattr(config, "CLIP_GRAD_NORM", 1.0))
        self.global_batch = int(config.BATCH_SIZE)
        if self.global_batch % self.world:
            raise ValueError("BATCH_SIZE (global) must be divisible by the number of ranks")
        self.local_batch = self.global_batch // self.world
        if not hasattr(config, "is_rectified_flow"):
            config.is_rectified_flow = self.is_rf
        self.sampler = host.TimestepSampler(config, self.device)
        self.loss_table = host.timestep_loss_curve_from_config(config, 1000, device=self.device)
        self.scheduler = DDPMScheduler(prediction_type=self.prediction_type)
        self.alphas_cumprod = self.scheduler.alphas_cumprod.to(self.device)
        curve = getattr(config, "LR_CUSTOM_CURVE", None)
        total_micro = int(config.MAX_TRAIN_STEPS)
        self.lr_scheduler = host.CustomCurveLRScheduler(optimizer, [list(p) for p in curve], total_micro) if curve else None
        self.noise_gen = torch.Generator(device=self.device)
        self.micro_step = 0
        self.optimizer_steps = 0
        self._accum = None              # {param: grad} carried across micro-steps when GRADIENT_ACCUMULATION_STEPS > 1
        self._acc = None                # the captured step's accumulator: one flat bf16 buffer, one 16-byte-aligned view per parameter
        self._acc_views = None
        self._acc_plan = MultiTensorPlan()
        self._acc_stage = _Staging()
        self.trainable = [p for p in unet.parameters() if p.requires_grad]
        self.use_cuda_graph = use_cuda_graph          # capture the device side of the step once, replay it afterwards
        self.graph_warmup = graph_warmup
        self._graphs = {}
        self._pools = {}                # GRADIENT_ACCUMULATION_STEPS > 1: one graph memory pool per input shape, shared by its phases

    # ---- pieces ------------------------------------------------------------------------------------------
    def _to_device(self, t, dtype=None):
        if t.device != self.device:
            t = t.to(self.device, non_blocking=True)
        if dtype is not None and t.dtype != dtype:
            t = t.to(dtype)
        return t.contiguous()

    def _noise(self, shape_local, global_len, row_offset):
        """train.py:2735-2742: ``randn(latents.shape)`` after the per-step reseed.  The draw has the shape of the batch the
        single-process run would see -- (global_len, 4, h, w), which on one GPU is exactly ``latents.shape``, short leftover
        batches included (CUDA Philox output depends on the element count, so a larger draw would not reproduce it) -- and a
        data-parallel rank keeps its own rows: N ranks see the noise of one process with the same global batch (SURVEY.md 8e)."""
        b = shape_local[0]
        gshape = (global_len,) + tuple(shape_local[1:])
        noise = host.generate_noise(torch.empty(gshape, device="meta"), self.noise_gen, self.device, step=self.micro_step + 1,
                                    seed=self.seed)
        if global_len == b:
            return noise
        return noise[row_offset:row_offset + b].contiguous()

    def _jitter(self, b, global_len, row_offset):
        gen = host.seeded_torch_generator(self.device, self.seed, self.micro_step + 1, 0x5D1)
        j = torch.rand((global_len,), device=self.device, dtype=torch.float32, generator=gen)
        return j if global_len == b else j[row_offset:row_offset + b].contiguous()

    # ---- the step ------------------------------------------------------------------------------------------
    def _device_step(self, latents, embeds, pooled, time_ids, tickets, noise, jitter, global_len, taps=None):
        """Everything that runs on the GPU for one micro-step (graph-capturable: no host reads, static shapes).
        ``global_len``: rows of the GLOBAL batch of this micro-step -- the loss is the mean over them (train.py:2408-2416), so
        the sum of the ranks' gradients is the single-process gradient also when the ranks hold unequal row counts."""
        if self.dp is not None and self.dp.defer_all_gather:
            # the all-gather of the PREVIOUS update starts now and hides behind the down path: every UNet block waits only for the
            # buckets that hold its own weights
            self.dp.begin_forward()
            self.unet.param_gate = self.dp.gate
        xt8, target, cond = ops.noise_target(latents, noise, tickets, None if self.is_rf else self.alphas_cumprod, jitter,
                                             self.prediction_type, cpad=8)
        pred, bwd = self.unet.forward_nhwc(xt8, cond, embeds, pooled, time_ids, taps=taps)
        if self.dp is not None and self.dp.defer_all_gather:
            self.dp.gate(None)
        denom = float(global_len)
        loss, _, dpred8 = ops.mse_loss(pred, target, tickets, self.loss_table, denom=denom,
                                       grad_scale=1.0 / (denom * self.grad_accum), pred_nhwc=True, dpred_ld=8)
        if self.dp is None:
            grads = bwd(dpred8)
        else:       # gradients are written straight into the flat buffer; each bucket is reduced as soon as it is complete
            grads = bwd(dpred8, on_grad=self.dp.grad_ready, dest=self.dp.grad_view)
        return loss, grads

    def _host_inputs(self, batch, noise, jitter):
        latents = self._to_device(batch["latents"], BF16)
        embeds = self._to_device(batch["embeds"], BF16)
        pooled = self._to_device(batch["pooled"], BF16)
        tid = batch["time_ids"]
        if not torch.is_tensor(tid):
            tid = torch.tensor(tid, dtype=BF16)
        time_ids = self._to_device(tid, BF16)
        b = latents.shape[0]
        global_len, row_offset = self._global_rows(batch, b)
        if self.world == 1:
            tickets, _ = self.sampler.sample(b)
        else:
            tickets, _ = self.sampler.sample_rows(global_len, row_offset, b)
        # ``noise`` / ``jitter`` overrides exist for parity tests (the CPU oracle cannot reproduce CUDA Philox draws)
        if noise is None:
            noise = self._noise(latents.shape, global_len, row_offset)
        else:
            noise = self._to_device(noise, torch.float32)
            if tuple(noise.shape) != tuple(latents.shape):
                raise ValueError(f"noise override has shape {tuple(noise.shape)}, latents {tuple(latents.shape)}")
        if self.is_rf:
            jitter = self._jitter(b, global_len, row_offset) if jitter is None else self._to_device(jitter, torch.float32)
        else:
            jitter = None
        return latents, embeds, pooled, time_ids, tickets, noise, jitter, global_len

    def _global_rows(self, batch, b):
        """(rows of the global batch, offset of this rank's first row).  One process: the batch IS the global batch.  Data
        parallel: ``BatchFeeder`` attaches both numbers; a caller that does not is taken to feed every rank ``b`` rows."""
        if self.world == 1:
            return b, 0
        gl = batch.get("global_batch_len")
        if gl is None:
            return b * self.world, self.rank * b
        return int(gl), int(batch.get("global_row_offset", self.rank * b))

    def _rank_without_rows(self, batch):
        """Data parallel, short global batch: this rank has no sample in the micro-step (train.py:493-496 leftovers cut over N
        ranks).  It still advances every host-side stream exactly like the others (tickets, micro-step, LR curve) and joins the
        collectives with an all-zero gradient, so the reduce-scatter / all-gather sequence stays aligned across ranks."""
        global_len, row_offset = self._global_rows(batch, 0)
        tickets, _ = self.sampler.sample_rows(global_len, row_offset, 0)
        if self.dp.defer_all_gather:                   # the other ranks open their step with the all-gather of the previous update
            self.dp.begin_forward()
            self.dp.gate(None)
        self.micro_step += 1
        if self.lr_scheduler is not None:
            self.lr_scheduler.step(self.micro_step)
        self.dp.no_gradients_this_step()
        phase = self._phase()
        norm = None
        if phase == "last":
            norm = self._optimizer_phase(None)
            self.optimizer_steps += 1
        else:
            self.dp.reduce_accumulate(first=phase == "first")
        return StepResult(loss=torch.zeros(1, dtype=torch.float32, device=self.device), grad_norm=norm, timesteps=tickets,
                          did_optimizer_step=phase == "last", lr=self.optimizer.param_groups[0]["lr"])

    def _phase(self):
        """Where the micro-step just counted sits in its accumulation window: "first", "middle" or "last" (optimizer step).
        With GRADIENT_ACCUMULATION_STEPS = 1 every micro-step is "last"."""
        r = self.micro_step % self.grad_accum
        return "last" if r == 0 else "first" if r == 1 else "middle"

    @torch.no_grad()
    def step(self, batch, *, noise=None, jitter=None, taps=None) -> StepResult:
        """batch: dict with ``latents`` [b,4,h,w] (bf16, pinned host or device), ``embeds`` [b,L,2048], ``pooled`` [b,1280],
        ``time_ids`` [b,6] (list or tensor; converted to bf16 as train.py:2726-2731 does)."""
        if self.dp is not None and batch.get("latents") is None:
            return self._rank_without_rows(batch)
        inputs = self._host_inputs(batch, noise, jitter)
        if self.use_cuda_graph and taps is None:
            return self._graph_step(inputs)
        latents, embeds, pooled, time_ids, tickets, noise, jitter, global_len = inputs
        loss, grads = self._device_step(latents, embeds, pooled, time_ids, tickets, noise, jitter, global_len, taps=taps)
        self.micro_step += 1
        if self.grad_accum > 1 and self.dp is None:
            if self._accum is None:
                self._accum = grads
            else:
                ps = list(grads)
                acc = [self._accum[p] for p in ps]
                ops.grad_accum_mt(acc, acc, [grads[p] for p in ps], self._acc_plan, self._acc_stage)
            grads = self._accum
        if self.lr_scheduler is not None:
            self.lr_scheduler.step(self.micro_step)
        phase = self._phase()
        did = phase == "last"
        norm = None
        if did:
            norm = self._optimizer_phase(grads)
            self._accum = None
            self.optimizer_steps += 1
        elif self.dp is not None:
            self.dp.reduce_accumulate(first=phase == "first")
        return StepResult(loss=loss, grad_norm=norm, timesteps=tickets, did_optimizer_step=did,
                          lr=self.optimizer.param_groups[0]["lr"])

    def _optimizer_phase(self, grads):
        if self.dp is not None:
            return self.dp.reduce_clip_step(self.optimizer, self.clip, accumulated=self.grad_accum > 1)
        return self.optimizer.clip_and_step(self.clip, grads=grads)

    def _after_sweep(self, grads, phase):
        """The device work that follows the reverse sweep in the captured form of the step (also run eagerly by its warm-up).
        One GPU with GRADIENT_ACCUMULATION_STEPS > 1 accumulates into the persistent ``_acc``: the first micro-step of a window
        copies its gradient there, the middle ones add to it, and the last adds it into its own gradient tensors in place -- so
        the norm and Raven launches of the last phase are exactly the ones a window of one captures.  Data parallel accumulates
        the reduced shard instead (``DataParallel.reduce_accumulate``).  Returns the norm on the last phase, else None."""
        if phase != "last":
            if self.dp is not None:
                self.dp.reduce_accumulate(first=phase == "first")
                return None
            ps = [p for p in self.trainable if p in grads]
            acc, g = self._accumulator(ps), [grads[p] for p in ps]
            ops.grad_accum_mt(acc, acc, g, self._acc_plan, self._acc_stage, copy=phase == "first")
            return None
        if self.dp is None and self.grad_accum > 1:
            ps = [p for p in self.trainable if p in grads]
            g = [grads[p] for p in ps]
            ops.grad_accum_mt(g, self._accumulator(ps), g, self._acc_plan, self._acc_stage)
        return self._optimizer_phase(grads)

    def _accumulator(self, params):
        if self._acc is None:
            offs, off = [], 0
            for p in self.trainable:
                offs.append(off)
                off += (p.numel() + 7) // 8 * 8
            self._acc = torch.empty(off, dtype=BF16, device=self.device)
            self._acc_views = {p: self._acc[o:o + p.numel()].view(p.shape) for p, o in zip(self.trainable, offs)}
        return [self._acc_views[p] for p in params]

    # ---- CUDA-graph path: the whole device side of the step is captured once and replayed ---------------------
    def _graph_step(self, inputs):
        latents, embeds, pooled, time_ids, tickets, noise, jitter, global_len = inputs
        key = (tuple(latents.shape), tuple(embeds.shape), global_len)      # the loss normaliser is baked into the captured kernels
        self.micro_step += 1
        if self.lr_scheduler is not None:
            self.lr_scheduler.step(self.micro_step)
        phase = self._phase()
        pool = None
        if self.grad_accum > 1:
            # every phase of one shape shares one memory pool: a replay's intermediates are dead when it ends, and what outlives
            # it (static inputs, st["out"], the accumulators) is allocated outside the pool or never freed
            pool = self._pools.get(key)
            if pool is None:
                pool = self._pools[key] = torch.cuda.graph_pool_handle()
            key = key + (phase,)
        last = phase == "last"
        if self.grad_accum > 1 and self.dp is None:
            self._accumulator(())          # before the first warm-up's activations, whose cached segments it would otherwise split
        st = self._graphs.get(key)
        if st is None:
            st = self._graphs[key] = dict(calls=0, graph=None)
        st["calls"] += 1
        if st["graph"] is None and st["calls"] <= self.graph_warmup:
            # eager warm-up: sizes the workspaces, allocates optimizer state, loads every kernel
            loss, grads = self._device_step(latents, embeds, pooled, time_ids, tickets, noise, jitter, global_len)
            norm = self._after_sweep(grads, phase)
            self.optimizer_steps += int(last)
            return StepResult(loss=loss, grad_norm=norm, timesteps=tickets, did_optimizer_step=last,
                              lr=self.optimizer.param_groups[0]["lr"])
        if st["graph"] is None:
            st["static"] = [t.clone() if t is not None else None for t in (latents, embeds, pooled, time_ids, tickets, noise, jitter)]
            self.unet._packs.d.clear()             # packed conv weights must be (re)built inside the graph on every replay
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, pool=pool):
                sl, se, sp, sti, stk, sn, sj = st["static"]
                loss, grads = self._device_step(sl, se, sp, sti, stk, sn, sj, global_len)
                norm = self._after_sweep(grads, phase)
                st["out"] = (loss, norm)
                del grads
            st["graph"] = g
            self.unet._packs.d.clear()
        for dst, src in zip(st["static"], (latents, embeds, pooled, time_ids, tickets, noise, jitter)):
            if dst is not None:
                dst.copy_(src, non_blocking=True)
        if last:
            self.optimizer.advance_host_state()
        st["graph"].replay()
        self.optimizer_steps += int(last)
        loss, norm = st["out"]
        return StepResult(loss=loss.clone(), grad_norm=norm.clone() if last else None, timesteps=tickets, did_optimizer_step=last,
                          lr=self.optimizer.param_groups[0]["lr"])
