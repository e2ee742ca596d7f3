"""The training step around the hot path -- SURVEY.md 8(f) rank 4: the B200 counterpart of the loop body of the reference's
`ddp_train.py:160-166` (zero_grad, forward, CrossEntropy, backward, `optimizer.step()`) and of its DistributedDataParallel
wrapping (`ddp_train.py:132-134`: one process per GPU, per-rank BatchNorm -- no SyncBN -- and DDP's default per-iteration
buffer broadcast).

    step = TrainStep(net, lr=1e-4, autocast=torch.bfloat16, ddp=world > 1, local_rank=local_rank)
    step.warmup(x, y)            # eager iterations on a side stream (cuDNN autotune, DDP bucket build)
    step.capture(x, y)           # forward + loss + backward (+ the NCCL all-reduces) + fused Adam in ONE CUDA graph
    loss = step(x, y)            # copies the batch into the graph's static inputs and replays

What is B200-specific here:
  * the whole step is one CUDA graph: ~2 900 kernel launches per MedMamba-T step, most of them microsecond-scale at
    stages 2-3, cost nothing on the host (the reference launches them one by one);
  * fused (multi-tensor, capturable) Adam;
  * DDP buckets sized for launch latency and overlap, not for link count (NVSwitch gives every pair full bandwidth): small
    buckets (`bucket_cap_mb`, default 8 MB instead of PyTorch's 25) so that the LAST bucket -- stage-0 / patch-embed
    gradients, ready only when backward ends -- leaves a short exposed all-reduce tail, `gradient_as_bucket_view=True`
    (no gradient copy into the buckets), `static_graph=True`;
  * `broadcast_buffers=False`: DDP's default re-broadcasts rank 0's BatchNorm running statistics before every forward
    (`ddp_train.py:134` keeps that default).  In training mode BatchNorm normalises with batch statistics, so the broadcast never
    changes a gradient or a weight, and rank 0 is never
    overwritten: the validation accuracy it logs and the checkpoint it saves (`ddp_train.py:181-193`, main process only) are bit-identical either way.  Skipping it removes ~90 small broadcasts (one coalesced launch plus
    its dependencies) from every step: 24.64 -> 24.43 ms at N = 2 (`profiles/bench_r02_n2*.json`).  Pass True to get DDP's default
    back (ranks > 0 then evaluate with rank 0's statistics);
  * optional bf16 gradient compression of the all-reduce payload (`grad_bf16=True`: PyTorch's bf16_compress_hook);
    off by default because the reference reduces fp32 gradients;
  * `ddp_impl="flat"` (default): `FlatGradSync` below replaces DistributedDataParallel's reducer.  All gradients live in ONE fp32
    buffer laid out in the order backward produces them (last layer first); the buffer is split into a few contiguous chunks whose
    sizes shrink geometrically (75 % / 19 % / 6 % of the bytes), and each chunk is all-reduced (average) with one NCCL call on a side
    stream the moment its last gradient has been accumulated.  On NVSwitch a 58 MB all-reduce costs a fraction of a millisecond
    whatever the rank count, so what matters is the number of collectives, what they wait for and the exposed tail: the big
    chunks hold the wide late stages (ready early in backward), the small last chunk holds stage 0 / the patch embedding (ready
    when backward ends).  Same arithmetic as DDP (`ddp_train.py:134`): mean of the per-rank fp32 gradients; parameters are
    broadcast from rank 0 once at construction.  `ddp_impl="torch"` keeps DistributedDataParallel.
"""
from __future__ import annotations

import torch
import torch.distributed as dist

from ._lib import is_dense as _dense


class FlatGradSync:
    """Gradient all-reduce of a data-parallel replica without DistributedDataParallel (reference: `ddp_train.py:132-134,160-166`).

    One flat fp32 buffer holds every gradient, ordered as backward produces them and cut into a few contiguous chunks.  During
    backward autograd hands each parameter its gradient as usual (no per-parameter copy or add kernel: with `p.grad is None` the
    engine just keeps the tensor the backward kernel wrote).  A post-accumulate hook per parameter counts arrivals; when a chunk is
    complete its gradients are gathered into the buffer with ONE multi-tensor copy and the chunk is all-reduced (average) with ONE
    NCCL call, both on `self.stream` after every compute stream that produced one of them (the model runs its two branches on two
    streams), and `p.grad` is re-pointed at the parameter's view of the buffer, which is what the optimizer
    reads.  `finish()` sends what is left (parameters that received no gradient count as zero) and joins the side stream.
    Everything is stream-ordered, so the whole exchange is captured in the step's CUDA graph.  (DistributedDataParallel, and a first
    version of this class that let autograd accumulate into the views, pay one small kernel per parameter per step -- ~230 for
    MedMamba-T, 0.5-0.9 ms inside a 23.7 ms step.)"""

    def __init__(self, net, fractions=(0.75, 0.94, 1.0), process_group=None, broadcast=True):
        self.group = process_group
        self.world = dist.get_world_size(process_group)
        params = [p for p in net.parameters() if p.requires_grad]
        if not params:
            raise ValueError("FlatGradSync: the module has no trainable parameter")
        self.dev = params[0].device
        self.params = list(reversed(params))                 # ~ the order in which backward produces the gradients
        offs, total = [], 0
        for p in self.params:
            if p.dtype != torch.float32 or not _dense(p):
                raise ValueError("FlatGradSync: parameters must be dense fp32 tensors")
            offs.append(total)
            total += (p.numel() + 3) // 4 * 4                # 16-byte aligned slices (vectorised optimizer / reduction kernels)
        self.flat = torch.zeros(total, dtype=torch.float32, device=self.dev)
        self.views = [self.flat.as_strided(p.shape, p.stride(), o) for p, o in zip(self.params, offs)]
        # chunk boundaries at the given fractions of the bytes, on parameter boundaries
        self.bounds, k = [], 0
        for f in fractions:
            lim = f * total
            while k < len(self.params) and (offs[k] + self.params[k].numel() <= lim or f >= 1.0):
                k += 1
            if k > (self.bounds[-1] if self.bounds else 0):
                self.bounds.append(k)
        if self.bounds[-1] != len(self.params):
            self.bounds.append(len(self.params))
        self.ranges = [((self.bounds[c - 1] if c else 0), hi) for c, hi in enumerate(self.bounds)]
        ends = [offs[hi] if hi < len(self.params) else total for hi in self.bounds]
        self.slices = [self.flat[a:b] for a, b in zip([0] + ends[:-1], ends)]
        self.need = [hi - lo for lo, hi in self.ranges]
        self.got = [0] * len(self.ranges)
        self.sent = [False] * len(self.ranges)
        self.seen = [set() for _ in self.ranges]
        self.active = False
        self.stream = torch.cuda.Stream(device=self.dev) if self.dev.type == "cuda" else None
        self.avg = dist.get_backend(process_group) == "nccl"
        if broadcast:                                        # DDP's construction-time sync: every rank starts from rank 0's values
            for t in list(net.parameters()) + list(net.buffers()):
                dist.broadcast(t.data, 0, group=process_group)
        for c, (lo, hi) in enumerate(self.ranges):
            for p in self.params[lo:hi]:
                p.grad = None
                p.register_post_accumulate_grad_hook(self._make_hook(c))

    def chunk_bytes(self):
        return [int(s.numel()) * 4 for s in self.slices]

    def _make_hook(self, c):
        def hook(_p):
            if self.active:
                if self.stream is not None:                  # gradients of one chunk may come from several streams (models.branch_stream)
                    self.seen[c].add(torch.cuda.current_stream(self.dev))
                self.got[c] += 1
                if self.got[c] == self.need[c]:
                    self._send(c)
        return hook

    def _send(self, c):
        if self.sent[c]:
            return
        self.sent[c] = True
        lo, hi = self.ranges[c]
        src = [p.grad for p in self.params[lo:hi]]
        if self.stream is None and any(g is None for g in src):   # parameters outside this step's graph: their gradient is zero
            self.slices[c].zero_()
        dst = [v for v, g in zip(self.views[lo:hi], src) if g is not None]
        src = [g for g in src if g is not None]
        buf = self.slices[c]
        if self.stream is not None:
            # gather and reduce on the side stream, after every stream that produced one of the chunk's gradients: an event recorded
            # now on such a stream covers all of them (their kernels were enqueued before this hook ran)
            self.seen[c].add(torch.cuda.current_stream(self.dev))
            for st in self.seen[c]:
                self.stream.wait_stream(st)
            with torch.cuda.stream(self.stream):
                if any(g is None for g in (p.grad for p in self.params[lo:hi])):
                    buf.zero_()
                if src:
                    torch._foreach_copy_(dst, src)           # one multi-tensor kernel (per ~100 tensors), not one copy per parameter
                    for g in src:
                        g.record_stream(self.stream)         # allocated on a compute stream, last read here
                self._reduce(buf)
        else:
            if src:
                torch._foreach_copy_(dst, src)
            self._reduce(buf)
        for p, v in zip(self.params[lo:hi], self.views[lo:hi]):
            p.grad = v

    def _reduce(self, buf):
        if self.avg:
            dist.all_reduce(buf, op=dist.ReduceOp.AVG, group=self.group)
        else:
            dist.all_reduce(buf, group=self.group)
            buf.mul_(1.0 / self.world)

    def begin(self):
        """Before forward: drop last step's gradient views (autograd then keeps the tensors its kernels write) and arm the hooks."""
        for p in self.params:
            p.grad = None
        self.got = [0] * len(self.ranges)
        self.sent = [False] * len(self.ranges)
        self.seen = [set() for _ in self.ranges]
        self.active = True

    def finish(self):
        """After backward, before the optimizer: reduce whatever is still pending and wait for the side stream."""
        for c in range(len(self.ranges)):
            self._send(c)
        self.active = False
        if self.stream is not None:
            torch.cuda.current_stream(self.dev).wait_stream(self.stream)


class TrainStep:
    def __init__(self, net, lr=1e-4, autocast=torch.bfloat16, ddp=False, local_rank=0, graph=True, bucket_cap_mb=8,
                 grad_bf16=False, broadcast_buffers=False, loss_fn=None, ddp_impl="flat"):
        self.net = net
        self.dev = next(net.parameters()).device
        if self.dev.type != "cuda":
            raise RuntimeError("TrainStep runs on CUDA modules only: the B200 path has no CPU fallback")
        self.autocast = autocast
        # the models issue their two branches on two streams on purpose (models.SS_Conv_SSM): the engine's advisory about
        # AccumulateGrad nodes created on another stream than the gradient's producer does not apply (it synchronises them itself)
        _quiet = getattr(torch.autograd.graph, "set_warn_on_accumulate_grad_stream_mismatch", None)
        if _quiet is not None:
            _quiet(False)
        self.use_graph = bool(graph)
        self.ddp = bool(ddp)
        self.loss_fn = loss_fn or torch.nn.functional.cross_entropy
        self.side = torch.cuda.Stream(device=self.dev)
        self.sync = None
        if ddp_impl not in ("flat", "torch"):
            raise ValueError("ddp_impl must be 'flat' or 'torch'")
        self.ddp_impl = ddp_impl if self.ddp else None
        if self.ddp and ddp_impl == "flat":
            if grad_bf16 or broadcast_buffers:
                raise ValueError("grad_bf16 / broadcast_buffers are DistributedDataParallel options: use ddp_impl='torch'")
            self.model = net
            self.sync = FlatGradSync(net)
        elif self.ddp:
            self.side.wait_stream(torch.cuda.current_stream(self.dev))
            with torch.cuda.stream(self.side):   # DDP built on the capture-warm-up stream (PyTorch CUDA-graph + DDP recipe)
                self.model = torch.nn.parallel.DistributedDataParallel(
                    net, device_ids=[local_rank], gradient_as_bucket_view=True, bucket_cap_mb=bucket_cap_mb, static_graph=True,
                    broadcast_buffers=broadcast_buffers)
                if grad_bf16:
                    from torch.distributed.algorithms.ddp_comm_hooks import default_hooks
                    self.model.register_comm_hook(None, default_hooks.bf16_compress_hook)
            torch.cuda.current_stream(self.dev).wait_stream(self.side)
        else:
            self.model = net
        self.local_rank = local_rank
        self.opt = torch.optim.Adam(self.model.parameters(), lr=lr, fused=True, capturable=self.use_graph)
        self.graph = None
        self.static_x = self.static_y = self.static_loss = None
        self.note = "eager"

    # ---- one step, eagerly -----------------------------------------------------------------------------------------
    def _fwd_bwd_opt(self, x, y):
        if self.sync is not None:
            self.sync.begin()
        if self.autocast is not None:
            with torch.autocast("cuda", dtype=self.autocast):
                loss = self.loss_fn(self.model(x).float(), y)
        else:
            loss = self.loss_fn(self.model(x), y)
        loss.backward()
        if self.sync is not None:
            self.sync.finish()
        self.opt.step()
        return loss

    def eager(self, x, y):
        if self.sync is None:
            self.opt.zero_grad(set_to_none=True)
        return self._fwd_bwd_opt(x, y)

    def barrier(self):
        if self.ddp:
            dist.barrier(device_ids=[self.local_rank])
        torch.cuda.synchronize(self.dev)

    def warmup(self, x, y, n=3):
        """n eager steps on a side stream (>= 11 under DDP: its buckets are rebuilt during the first iterations and must be
        final before a capture)."""
        n = max(n, 11 if (self.ddp and self.use_graph) else 1)
        self.side.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(self.side):
            for _ in range(n):
                self.eager(x, y)
        torch.cuda.current_stream(self.dev).wait_stream(self.side)
        self.barrier()

    def capture(self, x, y):
        """Capture forward, loss, backward (with DDP's bucketed all-reduces) and the fused Adam update in one CUDA graph.
        Falls back to eager launches (and says so in .note) if the capture fails."""
        if not self.use_graph:
            return False
        try:
            self.static_x, self.static_y = x.clone(), y.clone()
            if self.sync is None:
                self.opt.zero_grad(set_to_none=True)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self.static_loss = self._fwd_bwd_opt(self.static_x, self.static_y)
            self.note = "whole step captured in one CUDA graph"
            return True
        except Exception as exc:
            self.graph = None
            self.note = f"eager (graph capture failed: {type(exc).__name__}: {str(exc)[:120]})"
            torch.cuda.synchronize(self.dev)
            if self.sync is None:
                self.opt.zero_grad(set_to_none=True)
            return False

    def __call__(self, x, y):
        if self.graph is None:
            return self.eager(x, y)
        if x is not self.static_x:
            self.static_x.copy_(x, non_blocking=True)
            self.static_y.copy_(y, non_blocking=True)
        self.graph.replay()
        return self.static_loss
