"""Data-parallel training step with optimizer state sharded across GPUs (one process per GPU, NCCL over NVLink).

The reference is single-GPU (SURVEY.md M4); semantics here are *global-batch equivalence* (SURVEY.md 8e): N ranks x b
samples reproduce one process with BATCH_SIZE = N*b -- same tickets, same noise rows, loss normalised by the global
count, so the SUM of per-rank gradients equals the single-process gradient.

Layout: every trainable parameter lives in one flat bf16 buffer (``flat_p``; parameters become views), gradients are
gathered into ``flat_g`` of the same layout.  The flat space is cut into buckets; as soon as the reverse sweep has
produced every gradient of a bucket, its **reduce-scatter** is issued asynchronously (NCCL stream) and overlaps with the
rest of the sweep.  Rank r owns slice r of every bucket: Raven moments exist only for those slices (state sharded N
ways, replacing the reference's CPU offload, raven.py:64-69/114-117).  After the sweep: local sum of squares over the
owned slices -> all-reduce of one fp32 scalar -> clip coefficient on device -> ONE multi-tensor Raven launch over the
owned segments -> per-bucket **all-gather** of the updated bf16 parameters.  No host synchronisation anywhere.

``defer_all_gather=True`` moves that all-gather off the tail of the step: it is issued at the START of the next step, bucket by
bucket in the order the forward pass first touches the parameters (embeddings, conv_in, down blocks, mid block, up blocks, output
convolution -- not the flat / registration order, in which ``mid_block`` comes last), asynchronously on NCCL's stream, and every
UNet block waits only for the buckets that hold its own weights (``gate``): the transfer hides behind the down path instead of
being 4.5 GB of serial tail at 8 GPUs.  Between steps the non-owned slices of ``flat_p`` are then stale: anything that reads the
parameters outside a step (checkpoint export, evaluation, comparing weights) calls ``gather_params()`` first.

Deviation stated: the data-parallel gradient norm is the fp32 norm of the summed gradient (torch's bf16 per-tensor
rounding, SURVEY.md a7, cannot be reproduced on slices); the single-GPU path emulates it exactly.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist

from . import _lib, ops
from .optimizers.raven import RavenAdamW, raven_host_scalars, _DT

ALIGN = 8                    # elements: keeps every parameter slot 16-byte aligned for the vector kernels


class _KernelBackend:
    """Device math through the C ABI (product path).  ``tables``: device pointer tables of the owned segments, uploaded
    once (the flat buffers never move), which also keeps the calls CUDA-graph capturable."""

    @staticmethod
    def sumsq(seg_g, numels, plan, out3, gdt, tables=None):
        _lib.call("aoz_gradnorm_mt", plan.n_tensors, plan.n_chunks, tables["g"].data_ptr(), plan.numel.data_ptr(),
                  plan.chunk_start.data_ptr(), plan.chunk_tensor.data_ptr(), plan.partial.data_ptr(), 3.0e38, 0, out3.data_ptr(),
                  _DT[gdt], torch.cuda.current_stream().cuda_stream)

    @staticmethod
    def clip_coef(sumsq, max_norm, out2):
        _lib.call("aoz_clip_coef_from_sumsq", sumsq.data_ptr(), float(max_norm), 0, out2.data_ptr(),
                  torch.cuda.current_stream().cuda_stream)

    @staticmethod
    def raven(seg_p, seg_g, seg_m, seg_v, plan, hyper, clip_coef, pdt, gdt, mdt, tables=None):
        _lib.call("aoz_raven_step_mt", plan.n_tensors, plan.n_chunks, tables["p"].data_ptr(), tables["g"].data_ptr(),
                  tables["m"].data_ptr(), tables["v"].data_ptr(), plan.numel.data_ptr(), plan.chunk_start.data_ptr(),
                  plan.chunk_tensor.data_ptr(), hyper.data_ptr(), 0 if clip_coef is None else clip_coef.data_ptr(), _DT[pdt],
                  _DT[gdt], _DT[mdt], torch.cuda.current_stream().cuda_stream)

    @staticmethod
    def add(a, b, out):
        ops.add(a, b, out=out)


def _ptr_table(tensors, device):
    arr = np.fromiter((t.data_ptr() for t in tensors), dtype=np.uint64, count=len(tensors))
    return torch.from_numpy(arr.view(np.int64)).to(device)


class FlatLayout:
    """Flat placement of the trainable parameters and its bucket / shard geometry (pure host logic, unit-tested on CPU)."""

    def __init__(self, numels, world, bucket_elems):
        self.world = world
        self.offsets = []
        off = 0
        for n in numels:
            self.offsets.append(off)
            off += (n + ALIGN - 1) // ALIGN * ALIGN
        self.used = off
        quantum = world * ALIGN
        bucket_elems = max(quantum, bucket_elems // quantum * quantum)
        self.buckets = []                      # (start, end), each a multiple of world*ALIGN long
        start = 0
        while start < off:
            end = min(start + bucket_elems, (off + quantum - 1) // quantum * quantum)
            self.buckets.append((start, end))
            start = end
        self.total = self.buckets[-1][1] if self.buckets else 0
        self.numels = list(numels)

    def bucket_of_param(self, i):
        """Buckets a parameter's slot overlaps (a large tensor can span several)."""
        a, b = self.offsets[i], self.offsets[i] + self.numels[i]
        return [k for k, (s, e) in enumerate(self.buckets) if s < b and a < e]

    def shard_range(self, bucket, rank):
        s, e = self.buckets[bucket]
        n = (e - s) // self.world
        return s + rank * n, s + (rank + 1) * n

    def shard_elems(self):
        return self.total // self.world

    def segments(self, rank):
        """[(param index, offset inside the param, flat offset, length, offset inside this rank's shard storage)]"""
        segs = []
        base = 0
        for k in range(len(self.buckets)):
            lo, hi = self.shard_range(k, rank)
            for i, (off, n) in enumerate(zip(self.offsets, self.numels)):
                a, b = max(lo, off), min(hi, off + n)
                if a < b:
                    segs.append((i, a - off, a, b - a, base + (a - lo)))
            base += hi - lo
        return segs


class ShardedRavenAdamW(RavenAdamW):
    """RavenAdamW whose moments cover only this rank's slices of the flat parameter space.  Same constructor, same
    ``param_groups`` keys, same ``save_cpu_state`` / ``load_cpu_state`` format (gathered / scattered across ranks)."""

    _name = "ShardedRavenAdamW"

    def attach(self, dp):
        self.dp = dp
        self.step_count = 0
        n = dp.layout.shard_elems()
        self.m_shard = torch.zeros(n, dtype=self._momentum_dtype, device=dp.device)
        self.v_shard = torch.zeros(n, dtype=self._momentum_dtype, device=dp.device)
        return self

    def step(self, closure=None, clip_coef=None):
        raise _lib.AozoraError("ShardedRavenAdamW is stepped by DataParallel.reduce_clip_step()")

    def advance_host_state(self):
        """Host side of one replayed step (CUDA graphs): bump the step counter and upload the hyper-parameter table."""
        self.step_count += 1
        self.dp.upload_hyper(self)

    def hyper_table(self, seg_params):
        group_of = {}
        for group in self.param_groups:
            for p in group["params"]:
                group_of[p] = group
        hy = np.empty((len(seg_params), 8), dtype=np.float32)
        cache = {}
        for i, p in enumerate(seg_params):
            g = group_of[p]
            key = id(g)
            if key not in cache:
                cache[key] = raven_host_scalars(g["lr"], g["betas"], g["eps"], g["weight_decay"], g["debias_strength"], self.step_count)
            hy[i] = cache[key]
        return hy

    def save_cpu_state(self):
        """Gather the sharded moments into the reference's per-parameter CPU format (raven.py:156-169)."""
        dp = self.dp
        full_m, full_v = dp.gather_shards(self.m_shard), dp.gather_shards(self.v_shard)
        cpu_state = {"_momentum_dtype": self._momentum_dtype}
        if self.step_count == 0:
            return cpu_state
        for i, p in enumerate(dp.params):
            off, n = dp.layout.offsets[i], dp.layout.numels[i]
            cpu_state[i] = {"step": self.step_count, "exp_avg_cpu": full_m[off:off + n].view(p.shape).cpu().clone(),
                            "exp_avg_sq_cpu": full_v[off:off + n].view(p.shape).cpu().clone()}
        return cpu_state

    def load_cpu_state(self, cpu_state):
        dp = self.dp
        full_m = torch.zeros(dp.layout.total, dtype=self._momentum_dtype, device=dp.device)
        full_v = torch.zeros_like(full_m)
        steps = set()
        for i, p in enumerate(dp.params):
            if i not in cpu_state:
                continue
            s = cpu_state[i]
            m = s.get("exp_avg", s.get("exp_avg_cpu"))
            v = s.get("exp_avg_sq", s.get("exp_avg_sq_cpu"))
            st = s.get("step", 0)
            steps.add(int(st.item()) if torch.is_tensor(st) else int(st))
            off, n = dp.layout.offsets[i], dp.layout.numels[i]
            if m is not None:
                full_m[off:off + n] = m.to(dp.device, self._momentum_dtype).reshape(-1)
                full_v[off:off + n] = v.to(dp.device, self._momentum_dtype).reshape(-1)
        if len(steps) > 1:
            raise _lib.AozoraError("ShardedRavenAdamW: per-parameter step counters differ; cannot shard this state")
        self.step_count = steps.pop() if steps else 0
        self.m_shard.copy_(dp.take_shard(full_m))
        self.v_shard.copy_(dp.take_shard(full_v))


class DataParallel:
    def __init__(self, unet, momentum_dtype=torch.bfloat16, bucket_mb=512, group=None, backend=None, flat_dtype=None,
                 bucket_elems=None, defer_all_gather=False):
        # bucket_mb: measured at 2 B200 (profiles/r02_bench_dp2_mb*.json, ms per step): 16 MB 148.0, 64 MB 139.8, 256 MB 138.5 on one
        # box; 256 / 512 / 1024 MB 136.6 / 136.6 / 136.1 on another -- every collective launch disturbs the persistent GEMM waves, so
        # fewer, larger buckets win until the last bucket's un-overlapped reduce-scatter starts to show; at 8 B200: 64 MB 145.9,
        # 256 MB 140.5, 512 MB 139.5 ms per step
        self.group = group
        self.defer_all_gather = bool(defer_all_gather)
        self._params_stale = False           # deferred mode: the last update's slices have not been gathered yet
        self._ag_works = None                # deferred mode, inside a step: (bucket, work) in issue order, not yet waited for
        self._gate_rank = {}                 # module -> how many all-gathers (in issue order) must have completed before it runs
        self._ag_order = None
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.backend = backend or _KernelBackend
        self.params = [p for p in unet.parameters() if p.requires_grad]
        if not self.params:
            raise ValueError("DataParallel: no trainable parameters")
        self.device = self.params[0].device
        self.dtype = flat_dtype or self.params[0].dtype
        esize = torch.empty((), dtype=self.dtype).element_size()
        self.layout = FlatLayout([p.numel() for p in self.params], self.world, bucket_elems or bucket_mb * (1 << 20) // esize)
        L = self.layout
        self.flat_p = torch.zeros(L.total, dtype=self.dtype, device=self.device)
        self.flat_g = torch.zeros(L.total, dtype=self.dtype, device=self.device)
        self.g_shard = torch.zeros(L.shard_elems(), dtype=self.dtype, device=self.device)
        self.acc_shard = None                # gradient accumulation across micro-steps (reduce_accumulate)
        self.index = {}
        with torch.no_grad():
            for i, p in enumerate(self.params):
                off, n = L.offsets[i], p.numel()
                self.flat_p[off:off + n].copy_(p.detach().reshape(-1))
                p.data = self.flat_p[off:off + n].view(p.shape)
                p._aoz_flat = True             # UNet.fuse_projection_storage must not move it (q/k/v are adjacent here already)
                self.index[p] = i
        self.param_buckets = [L.bucket_of_param(i) for i in range(len(self.params))]
        self.bucket_need = [0] * len(L.buckets)
        for bl in self.param_buckets:
            for k in bl:
                self.bucket_need[k] += 1
        self.momentum_dtype = momentum_dtype
        self._segs = L.segments(self.rank)
        # shard-storage offsets of each bucket slice
        self._slice_base = []
        base = 0
        for k in range(len(L.buckets)):
            lo, hi = L.shard_range(k, self.rank)
            self._slice_base.append(base)
            base += hi - lo
        self._plan = None
        self._seg_cache = None
        self._pending = None
        self._works = []
        self._issued = []                    # buckets reduced so far in this micro-step, in issue order
        self._reduce_order = list(range(len(L.buckets)))     # the last complete micro-step's issue order
        self._norm = torch.zeros(4, dtype=torch.float32, device=self.device)
        self._coef = torch.zeros(2, dtype=torch.float32, device=self.device)
        self.optimizer = None
        self._reset_pending()
        if self.defer_all_gather:
            self._plan_gather_order(unet)

    # ---- deferred all-gather -------------------------------------------------------------------------------
    def _plan_gather_order(self, unet):
        """Order the buckets by first use in the forward pass and note, per gated module, how many of them it needs.  Gated modules
        are the units ``UNet2DConditionModel.forward_nhwc`` announces (``_forward_units``); a model without that method gets one
        gate over everything."""
        units = list(unet._forward_units()) if hasattr(unet, "_forward_units") else [unet]
        order, seen = [], set()
        self._gate_rank = {}
        for mod in units:
            need = 0
            for p in mod.parameters(recurse=True):
                i = self.index.get(p)
                if i is None:
                    continue
                for k in self.param_buckets[i]:
                    if k not in seen:
                        seen.add(k)
                        order.append(k)
                    need = max(need, order.index(k) + 1)
            self._gate_rank[mod] = need
        for k in range(len(self.layout.buckets)):               # buckets no announced module touches (padding only): last
            if k not in seen:
                order.append(k)
        self._ag_order = order

    def _all_gather_bucket(self, k, async_op):
        s, e = self.layout.buckets[k]
        n = (e - s) // self.world
        mine = self.flat_p[s + self.rank * n:s + (self.rank + 1) * n]
        if dist.get_backend(self.group) == "nccl":
            return dist.all_gather_into_tensor(self.flat_p[s:e], mine, group=self.group, async_op=async_op)
        outs = [torch.empty_like(mine) for _ in range(self.world)]
        dist.all_gather(outs, mine.clone(), group=self.group)
        self.flat_p[s:e].copy_(torch.cat(outs))
        return None

    def begin_forward(self):
        """Deferred mode, first thing in a step: issue the all-gather of the previous update, every bucket asynchronously, in
        forward-use order.  Always issued (the first step gathers identical data): a captured step must not depend on host state."""
        if not self.defer_all_gather:
            return
        self._ag_works = [(k, self._all_gather_bucket(k, async_op=True)) for k in self._ag_order]
        self._ag_done = 0
        # NCCL writes flat_p behind autograd's back: caches keyed on the version counters (the UNet's packed conv weights) must be
        # rebuilt by this forward pass -- each after its module's gate, i.e. from gathered data
        torch.autograd.graph.increment_version(self.params)

    def gate(self, mod=None):
        """Make the current stream wait for the buckets ``mod`` reads (``None``: all of them)."""
        if self._ag_works is None:
            return
        need = len(self._ag_works) if mod is None else self._gate_rank.get(mod, len(self._ag_works))
        while self._ag_done < need:
            w = self._ag_works[self._ag_done][1]
            if w is not None:
                w.wait()
            self._ag_done += 1
        if self._ag_done == len(self._ag_works):
            self._ag_works = None
            self._params_stale = False

    def gather_params(self):
        """Deferred mode, outside a step: bring every rank's ``flat_p`` up to date (no-op when it already is)."""
        if self.defer_all_gather and self._params_stale:
            self.begin_forward()
            self.gate(None)

    def make_optimizer(self, **raven_kwargs):
        opt = ShardedRavenAdamW([{"params": self.params, "lr_scale": 1.0}], momentum_dtype=self.momentum_dtype, **raven_kwargs)
        self.optimizer = opt.attach(self)
        return self.optimizer

    # ---- shard helpers ---------------------------------------------------------------------------------
    def take_shard(self, full):
        """This rank's slices of a full flat tensor, concatenated in bucket order."""
        parts = []
        for k in range(len(self.layout.buckets)):
            lo, hi = self.layout.shard_range(k, self.rank)
            parts.append(full[lo:hi])
        return torch.cat(parts)

    def gather_shards(self, shard):
        """Inverse of take_shard across ranks: every rank gets the full flat tensor."""
        full = torch.zeros(self.layout.total, dtype=shard.dtype, device=shard.device)
        for k, (s, e) in enumerate(self.layout.buckets):
            n = (e - s) // self.world
            piece = shard[self._slice_base[k]:self._slice_base[k] + n].contiguous()
            outs = [torch.empty_like(piece) for _ in range(self.world)]
            dist.all_gather(outs, piece, group=self.group)
            full[s:e] = torch.cat(outs)
        return full

    # ---- gradient path -----------------------------------------------------------------------------------
    def _reset_pending(self):
        if len(self._issued) == len(self.layout.buckets):
            self._reduce_order = self._issued
        self._issued = []
        self._pending = list(self.bucket_need)
        self._arrived = bytearray(len(self.params))
        self._works = []

    def no_gradients_this_step(self):
        """This rank holds no sample of the micro-step (short global batch): its contribution to every bucket is zero."""
        self._reset_pending()
        self.flat_g.zero_()
        self._arrived = bytearray(b"\x01" * len(self.params))
        for k in self._reduce_order:              # collectives pair up by issue order: the order the other ranks' sweeps use
            self._pending[k] = 0
            self._reduce_bucket(k)

    def _reduce_bucket(self, k):
        self._issued.append(k)
        s, e = self.layout.buckets[k]
        n = (e - s) // self.world
        out = self.g_shard[self._slice_base[k]:self._slice_base[k] + n]
        if dist.get_backend(self.group) == "nccl":
            self._works.append(dist.reduce_scatter_tensor(out, self.flat_g[s:e], op=dist.ReduceOp.SUM, group=self.group, async_op=True))
        else:       # gloo (CPU tests): all-reduce then keep the owned slice
            buf = self.flat_g[s:e].clone()
            dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=self.group)
            out.copy_(buf[self.rank * n:(self.rank + 1) * n])

    def grad_view(self, p):
        """Where the reverse sweep should write ``p``'s gradient: its slot of the flat gradient buffer (None if unmanaged).
        Kernels that write there directly (GEMM / conv weight gradients, column sums, norm parameter gradients) save the
        staging copy -- 1680 small copy launches and 10 GB of traffic per step otherwise."""
        i = self.index.get(p)
        if i is None:
            return None
        off = self.layout.offsets[i]
        return self.flat_g[off:off + p.numel()].view(p.shape)

    def grad_ready(self, p, g):
        """Called by the reverse sweep the moment a parameter's gradient is final: stage it into the flat gradient
        buffer (unless it was produced there) and launch the reduce-scatter of every bucket that just became complete
        (overlaps the sweep)."""
        i = self.index.get(p)
        if i is None:
            return
        if self._arrived[i]:
            raise _lib.AozoraError("DataParallel: a parameter's gradient arrived twice in one sweep (its bucket may already be reduced)")
        self._arrived[i] = 1
        off = self.layout.offsets[i]
        if g.data_ptr() != self.flat_g.data_ptr() + off * self.flat_g.element_size() or not g.is_contiguous():
            self.flat_g[off:off + p.numel()].copy_(g.reshape(-1))
        for k in self.param_buckets[i]:
            self._pending[k] -= 1
            if self._pending[k] == 0:
                self._reduce_bucket(k)

    def _segment_views(self, opt):
        if self._seg_cache is None:
            seg_p, seg_g, seg_m, seg_v, seg_params = [], [], [], [], []
            for (i, _, flat_off, n, shard_off) in self._segs:
                seg_p.append(self.flat_p[flat_off:flat_off + n])
                seg_g.append(self.g_shard[shard_off:shard_off + n])
                seg_m.append(opt.m_shard[shard_off:shard_off + n])
                seg_v.append(opt.v_shard[shard_off:shard_off + n])
                seg_params.append(self.params[i])
            from .optimizers.raven import MultiTensorPlan
            self._plan = MultiTensorPlan()
            self._plan.ensure([s[3] for s in self._segs], self.device)
            tables = None
            if self.backend is _KernelBackend:
                tables = dict(p=_ptr_table(seg_p, self.device), g=_ptr_table(seg_g, self.device),
                              m=_ptr_table(seg_m, self.device), v=_ptr_table(seg_v, self.device))
            self._seg_cache = (seg_p, seg_g, seg_m, seg_v, seg_params, tables)
        return self._seg_cache

    def upload_hyper(self, opt):
        seg_params = self._segment_views(opt)[4]
        hy = opt.hyper_table(seg_params)
        if self.device.type == "cuda":
            return opt._stage.put("dp_hyper", hy, self.device)
        return torch.from_numpy(hy)

    def _finish_reduce(self):
        """Reduce every bucket the sweep left incomplete and wait for all reduce-scatters of this micro-step: ``g_shard`` then
        holds this rank's slices of the summed gradient."""
        if any(c != 0 for c in self._pending):
            # parameters that produced no gradient in this sweep: their slots still hold an earlier step's values -- this
            # rank's contribution is zero, so clear them before the buckets they sit in are reduced
            for i, seen in enumerate(self._arrived):
                if not seen:
                    off = self.layout.offsets[i]
                    self.flat_g[off:off + self.layout.numels[i]].zero_()
            for k, c in enumerate(self._pending):
                if c != 0:
                    self._reduce_bucket(k)
        for w in self._works:
            w.wait()
        self._reset_pending()

    def reduce_accumulate(self, first):
        """GRADIENT_ACCUMULATION_STEPS > 1, every micro-step of a window but the last: finish this micro-step's reduce-scatter
        and accumulate the reduced shard (``first``: start the window with it), in bf16 with one rounding per add as torch's
        ``p.grad`` accumulation does.  The accumulator is 1/N of the flat gradient, allocated on the first call."""
        self._finish_reduce()
        if self.acc_shard is None:
            self.acc_shard = torch.empty_like(self.g_shard)
        if first:
            self.acc_shard.copy_(self.g_shard)
        else:
            self.backend.add(self.acc_shard, self.g_shard, self.acc_shard)

    def reduce_clip_step(self, optimizer, max_norm, accumulated=False):
        """Finish the reduce-scatter, clip by the GLOBAL norm, update this rank's slices, all-gather the parameters.
        ``accumulated``: last micro-step of an accumulation window -- the shard accumulated by ``reduce_accumulate`` is added to
        this micro-step's before the norm.  CUDA-graph capturable: under capture the step counter / hyper table are left to
        ``advance_host_state``."""
        capturing = self.device.type == "cuda" and torch.cuda.is_current_stream_capturing()
        self._finish_reduce()
        if accumulated:
            self.backend.add(self.acc_shard, self.g_shard, self.g_shard)
        opt = optimizer
        seg_p, seg_g, seg_m, seg_v, seg_params, tables = self._segment_views(opt)
        if capturing:
            hyper = opt._stage.device_buffer("dp_hyper")
        else:
            opt.step_count += 1
            hyper = self.upload_hyper(opt)
        be = self.backend
        kw = dict(tables=tables) if tables is not None else {}
        be.sumsq(seg_g, None, self._plan, self._norm, self.dtype, **kw)
        sumsq = self._norm[2:3]
        dist.all_reduce(sumsq, op=dist.ReduceOp.SUM, group=self.group)
        clip = max_norm is not None and max_norm > 0
        be.clip_coef(sumsq, max_norm if clip else 3.0e38, self._coef)
        be.raven(seg_p, seg_g, seg_m, seg_v, self._plan, hyper, self._coef[1:2] if clip else None, self.dtype, self.dtype,
                 opt._momentum_dtype, **kw)
        # all-gather the updated parameter slices (in place inside flat_p) -- or leave it to the start of the next step
        if self.defer_all_gather:
            self._params_stale = True
        else:
            for k in range(len(self.layout.buckets)):
                self._all_gather_bucket(k, async_op=False)
        # the parameters changed behind autograd's back (kernels / NCCL wrote flat_p): bump their version counters so caches
        # keyed on them -- the packed conv weights of the UNet -- are rebuilt (RavenAdamW.step does the same)
        torch.autograd.graph.increment_version(self.params)
        return torch.stack([self._coef[0], self._coef[1], sumsq[0]])
