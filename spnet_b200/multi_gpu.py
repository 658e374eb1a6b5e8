"""Data parallelism for the SPNet training step — the B200 replacement of the reference's
spnet/multi_gpu.py (make_parallel: single-process TF towers, per-GPU tf.slice of the batch,
outputs concatenated on the CPU, gradients summed implicitly through shared variables; disabled
in the reference at train_spnet.py:55).

Here: one process per GPU (torchrun), every rank holds a full replica and takes rows
[r*B/n, (r+1)*B/n) of the global batch (the reference's get_slice: shape[0]//parts, remainder
dropped, spnet/multi_gpu.py:49-54), BatchNorm statistics stay per replica exactly as in the tower
scheme (:61-79 calls the shared-weight model once per slice), and the gradients are averaged with
one NCCL all-reduce per step over NVLink 5 / NVSwitch, issued as buckets in the order backward
completes them: the Dense-head bucket (73 % of the bytes, offset 0 of the flat gradient buffer) and
the exit + middle-flow bucket are reduced on a side stream while backward is still running.
"""
import torch


def get_available_gpus():
    """Names in the reference's format ('/gpu:0', ...), spnet/multi_gpu.py:26-32."""
    if not torch.cuda.is_available():
        return []
    return ["/device:GPU:%d" % i for i in range(torch.cuda.device_count())]


def world():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def batch_slice(n_rows, rank, parts):
    """Row range of this replica: the reference's get_slice (size = shape[0] // parts)."""
    size = n_rows // parts
    return rank * size, (rank + 1) * size


class GradAllReduce:
    """engine.grad_hook: average the gradients over the ranks and apply Adam, bucket by bucket, in the order backward
    completes them:
      head  the Dense head (offset 0 of the flat buffer, 73 % of the bytes): final right after the head's backward;
      tail  exit + middle flow (the end of the buffer): final after part A of the backbone backward;
      rest  stem, block 1, entry flow, residual convolutions: final when backward is done.
    head and tail are reduced on a side stream while backward continues, and the Adam update of a bucket is
    launched on that stream as soon as its all-reduce is done (the weights of a bucket are no longer read by the
    rest of that step's backward), so only the small `rest` bucket and its update trail the backward pass.

    comm_dtype 'bf16' (default for the bf16 engine): gradients cross NVLink as bf16 - the Dense-head weight gradient
    is written in bf16 by its GEMM, the other buckets are cast - half the bytes of fp32; Adam reads the averaged bf16
    gradient. 'fp32' keeps everything in fp32 (default for the fp32 engine, used by the N-GPU == 1-GPU gradient test)."""

    def __init__(self, engine, group=None, comm_dtype=None, trace=None):
        import os
        import torch.distributed as dist
        self.dist, self.group = dist, group
        self.world = dist.get_world_size(group)
        comm_dtype = comm_dtype or os.environ.get("SPNET_B200_DP_COMM") or ("bf16" if engine.lowp else "fp32")
        assert comm_dtype in ("bf16", "fp32")
        self.lowp_comm = comm_dtype == "bf16"
        off, n, _ = engine.offsets["FinalOutput/kernel"]
        assert off == 0
        n_head = (n + 7) // 8 * 8
        N = engine.grads.numel()
        t0 = engine.offsets[engine.tail_param_key][0] if engine.tail_param_key else N
        self.ranges = {"head": (0, n_head), "tail": (t0, N), "rest": (n_head, t0)}
        self.on_cuda = torch.device(engine.device).type == "cuda"
        if self.lowp_comm:
            self.glp = torch.zeros(N, device=engine.device, dtype=torch.bfloat16)
            engine.head_grad_lp = self.glp[:n_head].view(engine.g["FinalOutput/kernel"].shape) if n == n_head else None
        else:
            self.glp = None
        if self.on_cuda:
            self.side = torch.cuda.Stream(device=engine.device)
            self.ready = {k: torch.cuda.Event() for k in ("head", "tail")}
            self.done = {k: torch.cuda.Event() for k in ("head", "tail")}
        self.in_flight = set()
        self.trace = bool(int(os.environ.get("SPNET_B200_DP_TRACE", "0"))) if trace is None else trace
        self.trace_log, self._ev = [], None

    # ---- optional per-stream timeline (SPNET_B200_DP_TRACE=1): CUDA events at the bucket boundaries of every step
    def _mark(self, name, stream=None):
        if self._ev is not None:
            e = torch.cuda.Event(enable_timing=True)
            e.record(stream if stream is not None else torch.cuda.current_stream())
            self._ev.append((name, e))

    def step_begin(self, engine):
        if self.trace and self.on_cuda:
            self._ev = []
            self._mark("step_begin")

    def timeline(self):
        """Median offset (ms) of every mark from step_begin over the traced steps (call after a synchronize); the median
        ignores the first steps (NCCL set-up, eager warm-up before the graph capture)."""
        acc = {}
        for ev in self.trace_log:
            t0 = ev[0][1]
            for name, e in ev[1:]:
                acc.setdefault(name, []).append(t0.elapsed_time(e))
        return {k: sorted(v)[len(v) // 2] for k, v in acc.items()}

    def _reduce_and_step(self, engine, which, stream=None):
        """all-reduce bucket `which` and apply Adam to it, on the current stream."""
        lo, hi = self.ranges[which]
        if hi <= lo:
            return
        self._mark(which + "_ar_begin", stream)
        if self.lowp_comm:
            from . import ops
            if not (which == "head" and engine.head_grad_lp is not None):
                ops.cast_f32_to_bf16(engine.grads[lo:hi], self.glp[lo:hi])
            self.dist.all_reduce(self.glp[lo:hi], group=self.group)
        else:
            self.dist.all_reduce(engine.grads[lo:hi], group=self.group)
        self._mark(which + "_ar_end", stream)
        engine.optimizer_step(grad_scale=1.0 / self.world, lo=lo, hi=hi, g_bf16=self.glp)
        self._mark(which + "_adam_end", stream)

    def bucket_ready(self, engine, which):
        """Called by the engine right after the gradients of bucket `which` are complete."""
        lo, hi = self.ranges[which]
        if not self.on_cuda or hi <= lo:
            return
        self._mark(which + "_ready")
        self.ready[which].record()
        with torch.cuda.stream(self.side):
            self.side.wait_event(self.ready[which])
            self._reduce_and_step(engine, which, self.side)
            self.done[which].record(self.side)
        self.in_flight.add(which)

    def __call__(self, engine):
        self._mark("backward_end")
        for which in ("head", "tail"):
            if which not in self.in_flight:
                self._reduce_and_step(engine, which)
        self._reduce_and_step(engine, "rest")
        for which in self.in_flight:
            torch.cuda.current_stream().wait_event(self.done[which])
        self.in_flight.clear()
        self._mark("step_end")
        if self._ev is not None:
            self.trace_log.append(self._ev)
            self._ev = None
        engine.skip_default_optimizer = True


def attach_data_parallel(engine, group=None, comm_dtype=None, trace=None):
    hook = GradAllReduce(engine, group, comm_dtype=comm_dtype, trace=trace)
    engine.grad_hook = hook
    return hook


def make_parallel(model):
    """Keras-surface entry point (spnet/multi_gpu.py:35-88): returns the model wrapped for data
    parallelism when the process group has more than one rank, the model itself otherwise."""
    rank, n = world()
    if n < 2:
        return model
    model.parallel = True
    return model


def get_serial_part(model, parallel=True):
    """spnet/multi_gpu.py:15-23 — the replica itself (there is no wrapper layer to peel off)."""
    return getattr(model, "serial_model", model)
