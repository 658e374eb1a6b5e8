#!/usr/bin/env python
"""Benchmark of the SPNet hot path on B200: Xception-SPNet full training step
(forward + YOLO-ellipse loss + backward + Keras Adam), bf16, batch 64 per GPU, 384x512x1
gen_fake_espi-style synthetic frames (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Prints ONE JSON line (rank 0). N > 1 is launched by torchrun (one rank per GPU, NCCL).
`value`   : images/s with the batch already resident in HBM (CUDA-graph replay, device timed).
`e2e`     : images/s through the engine's public input path with HOST buffers: every step's inputs are
            copied from pinned host memory inside the timed region (prefetched one step ahead on a copy
            stream, exactly as SPNetModel.fit does) and the loss is read back to the host every step.
`roofline`: the dominant kernel family of the step (its launches of one step replayed as a CUDA graph
            and timed with CUDA events); `roofline_other` holds the other families.
`--dump-outputs DIR`: what the last step of the HBM-timed leg computed, as .npy files (dump_outputs).
`--impl reference`: the reference network's CPU path. TensorFlow 1.14 / Keras 2.1.3 cannot run in
this image (BASELINE.md §3), so this arm times the oracle restatement (kind "port") of the same
training step on the box's host cores.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W, N_OUT = 384, 512, 576
BATCH_PER_GPU = 64
METRIC = "train images/sec (Xception-SPNet, 512x384)"
LR = 4e-5


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """SM clock / throttle reasons while the timed region runs, sampled by a SEPARATE nvidia-smi process every 100 ms
    (the profiling recipe's clocks line). An in-process NVML poll takes driver locks that kernel launches from this
    process need: the end-to-end leg, whose host thread must keep the GPU's queue fed step by step, lost up to 40 % in
    some runs to exactly that; the in-process poll is only the fallback when nvidia-smi cannot be started."""
    FIELDS = ["clocks.sm", "clocks.max.sm", "clocks_event_reasons.hw_slowdown", "clocks_event_reasons.hw_thermal_slowdown",
              "clocks_event_reasons.sw_thermal_slowdown", "clocks_event_reasons.sw_power_cap"]

    def __init__(self, index):
        vis = [t.strip() for t in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if t.strip()]
        self.smi_id = vis[index] if index < len(vis) else str(index)   # nvidia-smi counts physical devices
        self.index, self.proc, self.thread = index, None, None

    def start(self):
        import subprocess
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", self.smi_id, "--query-gpu=" + ",".join(self.FIELDS),
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            self.thread = _NvmlPoll(self.index)
            self.thread.start()

    def stop(self):
        if self.proc is None:
            return self.thread.stop() if self.thread is not None else {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        import signal
        self.proc.send_signal(signal.SIGINT)
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out, _ = self.proc.communicate()
        mhz, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in (out or "").splitlines():
            f = [t.strip() for t in line.split(",")]
            if len(f) < 6 or not f[0].isdigit():
                continue
            mhz.append(int(f[0]))
            mx = int(f[1]) if f[1].isdigit() else mx
            for k, v in zip(names, f[2:6]):
                if v == "Active":
                    reasons.add(k)
        if not mhz:  # nvidia-smi produced nothing in time: one in-process reading now rather than no clocks at all
            poll = _NvmlPoll(self.index)
            if poll.nv is not None:
                try:
                    return {"sm_mhz": float(poll.nv.nvmlDeviceGetClockInfo(poll.h, poll.nv.NVML_CLOCK_SM)), "sm_max_mhz": poll.max_mhz,
                            "reasons": [], "sampler": "single NVML reading after the timed region (nvidia-smi gave no samples)"}
                except Exception:
                    pass
        return {"sm_mhz": float(np.median(mhz)) if mhz else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "sampler": "nvidia-smi -lms 100 (separate process), %d samples" % len(mhz)}


class _NvmlPoll(threading.Thread):
    """Fallback: in-process NVML poll, twice a second."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self._stop_evt = index, [], set(), None, threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.5)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "sampler": "in-process NVML poll"}


def make_pool(n, seed0):
    from spnet_b200 import fake_espi
    X, Y, _ = fake_espi.make_dataset(n, base_seed=seed0)
    return X, Y


def make_pool_u8(n, seed0, workers=1):
    """uint8 gen_fake_espi-style frames (n,384,512,1) + normalised targets; parallel worker processes (fork: call before
    CUDA is initialised in this process)."""
    from spnet_b200 import fake_espi
    X, Y, _ = fake_espi.make_frames_u8(n, base_seed=seed0, workers=workers)
    return X, Y


def normalise_host(Xu):
    X = Xu.astype(np.float32)
    X = X / 255.0   # spnet/utils.py:340-342
    X -= 0.5
    X *= 2.0
    return X


# -------------------------------------------------------------------------------------------------
# batch 32 (BASELINE.md section 3). cpu_baseline: median of 5 timed steps after 2 warm-ups, as section 3 states;
# --impl reference: median of exactly --steps timed steps (fewer than 5 if asked), no time budget
CPU_BATCH = 32


def cpu_train_steps(n_timed, n_warm):
    """The oracle restatement's training step (fwd + loss + bwd + Keras Adam, fp32, batch 32, 384x512 gen_fake_espi frames)
    on all host cores. Returns (median seconds per step, timed steps run, cores)."""
    import torch
    from oracle import xception_torch as xt
    ncores = os.cpu_count() or 1
    torch.set_num_threads(ncores)
    X, Y = make_pool(CPU_BATCH, 10_000)
    model = xt.OracleSPNet(xt.init_weights(xt.xception_spnet_spec(H, W, N_OUT), seed=1), H, W)
    ts = []
    for i in range(n_warm + n_timed):
        t0 = time.perf_counter()
        _, _, _, grads = model.loss_and_grads(X, Y)
        model.adam_step(grads, LR)
        dt = time.perf_counter() - t0
        if i >= n_warm:
            ts.append(dt)
    return float(np.median(ts)), len(ts), ncores


def cpu_cfg1(n_timed=5, n_warm=2):
    """BASELINE.json configs[0] on the host cores: forward + YOLO-ellipse loss, batch 32, inference-mode BatchNorm."""
    import torch
    from oracle import xception_torch as xt
    X, Y = make_pool(CPU_BATCH, 10_000)
    model = xt.OracleSPNet(xt.init_weights(xt.xception_spnet_spec(H, W, N_OUT), seed=1), H, W)
    yt = torch.as_tensor(Y)
    ts = []
    for i in range(n_warm + n_timed):
        t0 = time.perf_counter()
        with torch.no_grad():
            float(model.custom_loss(yt, model.forward(X, training=False)))
        if i >= n_warm:
            ts.append(time.perf_counter() - t0)
    return CPU_BATCH / float(np.median(ts))


def run_reference(args, rank):
    """CPU arm: oracle restatement of the same training step on the host cores (kind 'port': TensorFlow 1.14 / Keras 2.1.3
    cannot run in this image). Batch 32 per step (BASELINE.md section 3), --steps timed steps, --warmup untimed steps
    (1..5), median."""
    if rank != 0:
        return
    import torch
    nwarm = min(5, max(1, args.warmup))
    dt, nsteps, ncores = cpu_train_steps(args.steps, nwarm)
    ms = 1e3 * dt
    val = CPU_BATCH / dt
    out = {"impl": "reference", "metric": METRIC, "value": val, "unit": "images/s", "n_gpus": args.gpus,
           "steps": nsteps, "warmup": nwarm, "ms_per_step": ms, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": "Xception-SPNet train step fwd+bwd+YOLO-ellipse loss+Keras Adam, 384x512x1, batch 64/GPU",
                      "sample": "batch %d per step (bounded sample of the batch-64 workload, BASELINE.md section 3)" % CPU_BATCH,
                      "note": "reference CPU path = oracle restatement (TF1.14/Keras2.1.3 not runnable here)"},
           "cpu_baseline": {"value": val, "unit": "images/s", "cores": ncores, "kind": "port",
                            "sample": "median of %d timed steps (%d warm-ups) of %d images, oracle torch %s CPU fp32, all host cores" % (
                                nsteps, nwarm, CPU_BATCH, torch.__version__)},
           "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


# -------------------------------------------------------------------------------------------------
DUMP_PARAMS = 1 << 20   # sampled trainable parameters (4 MB); all of them are ~77 million at 384x512


def dump_outputs(eng, out_dir):
    """Writes what the last timed step handed its caller, float32, as out_dir/<name>.npy:
    loss (the [total, center, size, angle, noobj, class] data loss train_step returns), l2_loss, y_pred (the step's
    predictions), bn_moving_stats (every BatchNorm moving mean / variance after the step) and params_sample: the updated
    trainable parameters, concatenated in get_weights() order, at DUMP_PARAMS positions drawn with seed 0 (sorted).
    The bench inputs are seeded and the step starts from the engine's initial state (run_ours), so two runs, or two
    builds, with the same arguments can be compared file for file."""
    import torch
    torch.cuda.synchronize()
    flat = torch.cat([eng.w[k].reshape(-1) for k, _, trainable, _ in eng.spec if trainable])
    idx = np.sort(np.random.default_rng(0).choice(flat.numel(), size=min(flat.numel(), DUMP_PARAMS), replace=False))
    arrays = {"loss": eng.loss6, "l2_loss": eng.l2_out, "y_pred": eng.y_pred, "bn_moving_stats": eng.nontrainable,
              "params_sample": flat[torch.from_numpy(idx).to(flat.device)]}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def engine_state(eng):
    """Copy of what a training step reads and updates: weights, Adam moments, BatchNorm moving statistics, step count."""
    return [t.clone() for t in (eng.params, eng.adam_m, eng.adam_v, eng.nontrainable)], eng.step_count


def restore_engine_state(eng, state):
    tensors, eng.step_count = state
    for dst, src in zip((eng.params, eng.adam_m, eng.adam_v, eng.nontrainable), tensors):
        dst.copy_(src)
    eng.refresh_lowp()   # the bf16 working copy of the weights


def kernel_breakdown(eng, lib, steps=2):
    """Eager steps with a CUDA-event pair around every kernel launch -> per-family device time."""
    import torch
    lib.profile = []
    for _ in range(steps):
        eng.train_step(LR)
    torch.cuda.synchronize()
    prof, lib.profile = lib.profile, None
    fam = {}
    for name, args, e0, e1 in prof:
        d = fam.setdefault(name, {"ms": 0.0, "launches": 0, "items": []})
        ms = e0.elapsed_time(e1)
        d["ms"] += ms
        d["launches"] += 1
        d["items"].append((args, ms))
    return fam, steps


def algorithmic_work(name, a):
    """(bytes, flops) one launch must move / compute, from its C-ABI arguments."""
    def es(dtype):
        return 2 if dtype == 1 else 4
    a = tuple(a)
    if name == "spnet_dwconv3x3_fwd":      # in,k,a,b,relu,out,dtype,B,H,W,C,stream
        n = a[7] * a[8] * a[9] * a[10]
        return 2 * n * es(a[6]), 18 * n
    if name == "spnet_dwconv3x3_bwd_fused":  # gout,in,k,a,b,relu,mean,rstd,stats,add,adds,gin,dk,dk_acc,dtype,B,H,W,C
        n = a[15] * a[16] * a[17] * a[18]
        t = 3 + (1 if a[9] else 0)
        return t * n * es(a[14]), 36 * n
    if name == "spnet_gemm_bf16":          # A,lda,amn,B,ldb,bmn,D,ldd,slab_stride,mode,M,N,K,splits,...
        M, N, K = a[10], a[11], a[12]
        nout = (a[13] if a[9] == 3 else 1) * M * N   # slab mode: one [M, N] product per split
        return 2 * (M * K + N * K) + (2 if a[9] == 0 else 4) * nout, 2 * M * N * K
    return 0, 0


def run_ours(args, rank, world):
    import torch
    import torch.distributed as dist
    from spnet_b200._lib import lib as get_lib
    from spnet_b200 import engine as engine_mod
    from spnet_b200 import multi_gpu
    # the headline workload is Xception (BASELINE configs[1]); --backbone runs the same step on the other
    # backbones of BASELINE configs[2] / [3] for the record (profiles/README.md), not as the bench line
    Engine = {"Xception": engine_mod.XceptionSPNetEngine, "MobileNet": engine_mod.MobileNetSPNetEngine,
              "InceptionResNetV2": engine_mod.InceptionResNetV2SPNetEngine}[args.backbone]
    global METRIC
    METRIC = METRIC.replace("Xception", args.backbone)

    local = int(os.environ.get("LOCAL_RANK", 0))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    lib = get_lib()
    B = BATCH_PER_GPU
    npool = 2 * B
    Xu, Y, Xu_inf = args.pools           # uint8 frames, generated before CUDA was initialised (main)
    Xp = torch.from_numpy(Xu[:npool]).pin_memory()            # HOST buffers of the end-to-end legs: uint8 pixel values
    Yp = torch.from_numpy(Y[:npool]).pin_memory()
    Xd, Yd = torch.from_numpy(normalise_host(Xu[:npool])).to(dev), Yp.to(dev)   # resident inputs of the HBM-timed leg

    eng = Engine(H, W, B, dtype="bf16", device=str(dev), seed=1)
    initial = engine_state(eng)
    if world > 1:
        multi_gpu.attach_data_parallel(eng)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # eager warm-up (also counts kernel launches per step), then capture the step into a CUDA graph
    eng.x0.copy_(Xd[:B]); eng.y_true.copy_(Yd[:B])
    l0 = lib.launches
    eng.train_step(LR)
    torch.cuda.synchronize()
    launches_per_step = lib.launches - l0
    eng.capture()
    sampler = ClockSampler(local)   # started before the warm-up: nvidia-smi needs ~0.2 s before its first sample
    sampler.start()
    for i in range(args.warmup):
        o = (i % 2) * B
        eng.x0.copy_(Xd[o:o + B]); eng.y_true.copy_(Yd[o:o + B])
        eng.train_step(LR)
    barrier()

    # ---- timed region 1: inputs resident in HBM. The step adds weight gradients with fp32 reduce-adds whose order
    #      varies, so the weights drift apart in their last bits from run to run and every further step amplifies that.
    #      The last timed step therefore starts from the engine's initial state, restored between two timed windows:
    #      its batch, weights and optimiser state are the same in every run. What it computes still differs in the last
    #      bits (its own gradient reduce-adds), so compare dump_outputs files with a tolerance, not bit for bit.
    def step(i):
        o = (i % 2) * B
        eng.x0.copy_(Xd[o:o + B]); eng.y_true.copy_(Yd[o:o + B])
        eng.train_step(LR)
    ev0, ev1, ev_last0, ev_last1 = (torch.cuda.Event(enable_timing=True) for _ in range(4))
    barrier()
    ev0.record()
    for i in range(args.steps - 1):
        step(i)
    ev1.record()
    barrier()
    restore_engine_state(eng, initial)
    del initial   # ~0.9 GB of device memory the later legs can use
    barrier()
    ev_last0.record()
    step(args.steps - 1)
    ev_last1.record()
    barrier()
    ms_dev = ev0.elapsed_time(ev1) + ev_last0.elapsed_time(ev_last1)
    if args.dump_outputs and rank == 0:
        dump_outputs(eng, args.dump_outputs)

    # the box's pinned host->device rate for one batch of frames, measured alone (not part of any timed region):
    # the end-to-end figure below cannot exceed batch / (this copy's time) and single-GPU boxes differ a lot here
    hb0, hb1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    scratch_dev = torch.empty(Xp[:B].shape, device=dev, dtype=torch.uint8)
    scratch_dev.copy_(Xp[:B], non_blocking=True)
    torch.cuda.synchronize()
    hb0.record()
    for _ in range(5):
        scratch_dev.copy_(Xp[:B], non_blocking=True)
    hb1.record()
    torch.cuda.synchronize()
    h2d_gbps = 5 * scratch_dev.numel() / (hb0.elapsed_time(hb1) * 1e-3) / 1e9
    del scratch_dev

    # ---- timed region 2: end to end from host buffers (pinned H2D of every batch + D2H of every step's loss).
    #      The loss of step i is copied to pinned host memory asynchronously and read on the host while steps i+1 and
    #      i+2 are queued (a training loop that logs every step two steps late): every step's result still reaches the
    #      host inside the timed region, the last ones before the closing event.
    DEPTH = 3   # losses in flight: the host reads step i-2's loss while steps i-1 and i are queued, so one host hiccup
    #             (the clock sampler forks nvidia-smi from this process) does not drain the GPU's queue
    loss_host = [torch.zeros(6).pin_memory() for _ in range(DEPTH)]
    loss_ev = [torch.cuda.Event() for _ in range(DEPTH)]
    barrier()
    ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev2.record()
    last = None
    eng.prefetch_batch(Xp[:B], Yp[:B])  # the first batch's H2D copy is inside the timed region too
    for i in range(args.steps):
        eng.take_prefetched()
        if i + 1 < args.steps:
            o = ((i + 1) % 2) * B
            eng.prefetch_batch(Xp[o:o + B], Yp[o:o + B])  # next batch travels while this step computes (as Model.fit does)
        loss6 = eng.train_step(LR)
        loss_host[i % DEPTH].copy_(loss6, non_blocking=True)
        loss_ev[i % DEPTH].record()
        if i >= DEPTH - 1:
            j = i - (DEPTH - 1)
            loss_ev[j % DEPTH].synchronize()
            last = float(loss_host[j % DEPTH][0])
    for j in range(max(0, args.steps - (DEPTH - 1)), args.steps):   # the remaining losses, before the closing event
        loss_ev[j % DEPTH].synchronize()
        last = float(loss_host[j % DEPTH][0])
    ev3.record()
    barrier()
    ms_e2e = ev2.elapsed_time(ev3)
    clocks = sampler.stop()

    # ---- timed region 3: inference through the public API (SPNetModel.predict, reference call site
    #      predict_spnet.py:85) with HOST buffers: a pinned pool of uint8 frames cycled to ~50,000 frames per job
    #      (BASELINE.json configs[4]), every batch copied host -> device inside the timed region, results copied back,
    #      then decode + hawley_spnet.csv. Each rank predicts its contiguous share of the job (no collective).
    hook_obj = eng.grad_hook
    dp_timeline = None
    if hook_obj is not None and getattr(hook_obj, "trace", False):
        torch.cuda.synchronize()
        dp_timeline = hook_obj.timeline()
    infer = run_inference(args, rank, world, dev, Xu_inf, barrier)

    t = torch.tensor([ms_dev, ms_e2e, infer["ms_predict"], infer["ms_total"]], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e = float(t[0]), float(t[1])
    infer["ms_predict"], infer["ms_total"] = float(t[2]), float(t[3])
    if rank != 0:
        return
    frames_job = infer.pop("frames_per_rank") * world
    infer.update({"value": frames_job / (infer["ms_predict"] / 1e3), "unit": "images/s",
                  "value_with_decode_and_csv": frames_job / (infer["ms_total"] / 1e3), "frames": frames_job, "n_gpus": world})

    total_imgs = B * world * args.steps
    value = total_imgs / (ms_dev / 1e3)
    e2e = total_imgs / (ms_e2e / 1e3)
    peaks = load_peaks()

    # ---- per-family view of the step: eager steps with a CUDA-event pair around every launch give the
    #      share of each kernel family; the roofline numbers come from replaying each family's launches
    #      (same arguments, same buffers, step order) as one CUDA graph timed with CUDA events, so that
    #      the ~4 us per-launch cost of eager event pairs does not deflate kernels that run 10-30 us
    eng.graph = None
    hook, eng.grad_hook = eng.grad_hook, None  # time this rank's kernels only
    fam, psteps = kernel_breakdown(eng, lib)
    eng.grad_hook = hook
    total_ms = sum(d["ms"] for d in fam.values())
    share = sorted(((d["ms"] / total_ms, n, d["launches"] // psteps) for n, d in fam.items()), reverse=True)
    breakdown = [{"kernel": n, "share": round(s, 4), "launches_per_step": l} for s, n, l in share[:14]]

    def graph_us(calls, reps=4):
        """Average device time per launch of `calls` [(name, args)] replayed as one CUDA graph."""
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            st = torch.cuda.current_stream().cuda_stream
            for name, a in calls:
                rc = getattr(lib._dll, name)(*(tuple(a[:-1]) + (st,)))
                if rc != 0:
                    raise RuntimeError("%s failed in the family replay: %s" % (name, lib.last_error()))
        g.replay()
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(reps):
            g.replay()
        t1.record()
        torch.cuda.synchronize()
        return t0.elapsed_time(t1) * 1e3 / (reps * len(calls))

    RIDGE = peaks["tf_burst"] * 1e12 / (peaks["hbm"] * 1e9)  # FLOP/B above which a GEMM is tensor-bound
    one_step = {n: d["items"][:len(d["items"]) // psteps] for n, d in fam.items()}
    fams = {"gemm_tensor": ("tensor", "gemm_tc_kernel (tcgen05), shapes above the ridge (%.0f FLOP/B)" % RIDGE, []),
            "gemm_hbm": ("hbm", "gemm_tc_kernel (tcgen05), shapes below the ridge", []),
            "dwconv_fwd": ("hbm", "dw3x3_fwd_packed_kernel (+BN/ReLU on load)", []),
            "dwconv_bwd": ("hbm", "dw3x3_bwd_packed_kernel (dgrad+wgrad+mask+BN sums)", [])}
    for a, _ in one_step.get("spnet_gemm_bf16", []):
        b_, f_ = algorithmic_work("spnet_gemm_bf16", a)
        fams["gemm_tensor" if f_ / b_ >= RIDGE else "gemm_hbm"][2].append(("spnet_gemm_bf16", a))
    for a, _ in one_step.get("spnet_dwconv3x3_fwd", []):
        fams["dwconv_fwd"][2].append(("spnet_dwconv3x3_fwd", a))
    for a, _ in one_step.get("spnet_dwconv3x3_bwd_fused", []):
        fams["dwconv_bwd"][2].append(("spnet_dwconv3x3_bwd_fused", a))
    traffic = {}
    for rnd in ("r2", "r1"):   # per-launch DRAM traffic of one representative launch per family, from ncu --set full
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", rnd, "traffic.json")))
            break
        except Exception:
            pass
    roofs = {}
    for key, (bound, label, calls) in fams.items():
        if not calls:
            continue
        us = graph_us(calls)
        nb = sum(algorithmic_work(n, a)[0] for n, a in calls)
        nf = sum(algorithmic_work(n, a)[1] for n, a in calls)
        r = {"bound": bound, "kernel": label, "launches": len(calls), "avg_launch_ms": us * 1e-3,
             "traffic": traffic.get(key, {}).get("bytes_per_launch"), "traffic_source": traffic.get(key, {}).get("source"),
             "timing": "CUDA-graph replay of the family's launches of one step, CUDA events"}
        t_s = us * 1e-6 * len(calls)
        if bound == "hbm":
            ach = nb / t_s / 1e9
            r.update({"achieved": ach, "peak": peaks["hbm"], "unit": "GB/s", "frac": ach / peaks["hbm"],
                      "algorithmic_bytes_per_step": nb})
        else:
            ach = nf / t_s / 1e12
            # the family is replayed alone for a few milliseconds at full clock: the BURST peak is the denominator
            r.update({"achieved": ach, "peak": peaks["tf_burst"], "unit": "TFLOP/s", "frac": ach / peaks["tf_burst"],
                      "frac_of_sustained_peak": ach / peaks["tf_sust"], "algorithmic_flops_per_step": nf})
        r["share_of_step"] = t_s * 1e3 / (ms_dev / args.steps)
        roofs[key] = r
    # per-shape view of the GEMMs (M,N,K,a_mn,b_mn): eager-event time, TFLOP/s
    shapes = {}
    for a, ms in fam.get("spnet_gemm_bf16", {"items": []})["items"]:
        key = (a[10], a[11], a[12], a[2], a[5])
        d = shapes.setdefault(key, [0, 0.0])
        d[0] += 1
        d[1] += ms
    gemm_shapes = [{"M": k[0], "N": k[1], "K": k[2], "a_mn": k[3], "b_mn": k[4], "launches_per_step": v[0] // psteps,
                    "us_each_eager": round(1e3 * v[1] / v[0], 1), "tflops": round(2.0 * k[0] * k[1] * k[2] / (v[1] / v[0] * 1e-3) / 1e12, 1)}
                   for k, v in sorted(shapes.items(), key=lambda kv: -kv[1][1])[:args.gemm_shapes]]
    dominant = max(roofs.values(), key=lambda r: r["share_of_step"])
    other = [r for r in roofs.values() if r is not dominant]

    # ---- CPU baseline on this box's host cores: bounded sample of the same workload
    cpu = cpu_baseline() if (not args.quick and world == 1) else None   # N = 1 only (bench contract)
    fit_leg = None
    if world == 1 and not args.quick:
        del eng
        torch.cuda.empty_cache()
        nfit = min(512, Xu_inf.shape[0]) // BATCH_PER_GPU * BATCH_PER_GPU
        if nfit:
            fit_leg = run_fit(args, dev, Xu_inf[:nfit], args.fit_Y[:nfit])

    out = {"metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
           "config": {"workload": "%s-SPNet train step fwd+bwd+YOLO-ellipse loss+Keras Adam, 384x512x1, batch %d/GPU" % (args.backbone, B),
                      "global_batch": B * world, "parallelism": "dp%d" % world, "dropout": 0.1, "l2": 1e-4,
                      "input_pool": "%d distinct gen_fake_espi-style frames per rank" % npool,
                      "l2_cache": "per-step working set (activations, several GB) >> 126 MB L2; no explicit flush",
                      "cuda_graph": True, "loss_last": last},
           "clocks": clocks,
           "e2e": {"value": e2e, "unit": "images/s", "ms_per_step": ms_e2e / args.steps,
                   "h2d_bytes_per_step": int(B * (H * W * 1 + N_OUT * 4)), "d2h_bytes_per_step": 24,
                   "input": "uint8 frames from pinned host memory, normalised on the device ((v/255-0.5)*2, bit-exact)",
                   "h2d_gb_per_s_of_this_box": round(h2d_gbps, 2),
                   "h2d_bound_images_per_s": round(B * world / (B * H * W / (h2d_gbps * 1e9)), 1)},
           "gpu_launches": int(launches_per_step * args.steps * 2),
           "roofline": dominant, "roofline_other": other, "kernel_breakdown": breakdown, "eager_step_ms": total_ms / psteps, "gemm_shapes": gemm_shapes,
           "peaks": peaks, "inference": infer, "fit": fit_leg, "cpu_baseline": cpu, "dp_timeline_ms": dp_timeline}
    print(json.dumps(out), flush=True)


def run_inference(args, rank, world, dev, Xu_inf, barrier):
    """predict_spnet's hot loop through the public API: SPNetModel.predict over ~50k frames of host memory."""
    import torch
    import spnet.config as cf
    from spnet import models, utils
    import predict_spnet
    cf.compute_dtype, cf.basemodel, cf.model_type = "bf16", args.backbone, "big"
    B = args.infer_batch
    pool = torch.from_numpy(Xu_inf).pin_memory()
    npool = pool.shape[0]
    per_rank = (args.infer_frames // world + npool - 1) // npool * npool   # whole passes over the pool
    reps = per_rank // npool
    model = models.SPNetModel((H, W, 1), Y0size=N_OUT, quick_setup=True, backbone=args.backbone)
    model.predict(pool[:2 * B], batch_size=B)   # engine set-up + graph capture: not part of the timed region
    utils.setup_means_and_ranges([6, 6, 2, 8])
    import tempfile
    log_dir = tempfile.mkdtemp(prefix="bench_predict_rank%d_" % rank) + "/"   # ~72 rows per frame on random weights: >100 MB
    barrier()
    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    e0.record()
    parts = [model.predict(pool, batch_size=B) for _ in range(reps)]
    e1.record()
    Y_pred = np.concatenate(parts, axis=0)
    Yp, decoded = predict_spnet.decode_on_device(Y_pred)
    names = ["frame_%07d.png" % (rank * per_rank + i) for i in range(per_rank)]
    utils.show_pred_ellipses(Yp, Yp, names, num_draw=per_rank, log_dir=log_dir, out_csv=log_dir + "hawley_spnet.csv",
                             show_true=False, draw_images=False, decoded=decoded)
    e2.record()
    barrier()
    rows = sum(1 for _ in open(log_dir + "hawley_spnet.csv"))
    csv_bytes = os.path.getsize(log_dir + "hawley_spnet.csv")
    import shutil
    shutil.rmtree(log_dir, ignore_errors=True)
    return {"ms_predict": e0.elapsed_time(e1), "ms_total": e0.elapsed_time(e2), "frames_per_rank": per_rank, "batch": B,
            "api": "SPNetModel.predict(pinned uint8 host pool of %d frames, cycled %dx per rank), CUDA-graph forward, "
                   "H2D of every batch and D2H of every result inside the timed region" % (npool, reps),
            "h2d_bytes_per_batch": int(B * H * W), "csv_rows_rank0": rows, "csv_bytes_rank0": csv_bytes,
            "note": "random-initialised weights: ~72 'detections' per frame, so the CSV leg formats millions of rows; a trained "
                    "model writes a few rows per frame"}


def run_fit(args, dev, Xu, Y):
    """The training loop a user runs: SPNetModel.fit (reference call site train_spnet.py:118-128) on HOST arrays -
    shuffled batches gathered on the host, pinned staging, H2D on the copy stream one batch ahead, CUDA-graph step,
    epoch loss read back. Two passes over a pool of host frames; the second epoch (graph already captured) is timed
    with the host clock around fit()."""
    import torch
    import spnet.config as cf
    from spnet import models
    cf.compute_dtype, cf.basemodel, cf.model_type = "bf16", args.backbone, "big"
    B = BATCH_PER_GPU
    model = models.SPNetModel((H, W, 1), Y0size=N_OUT, quick_setup=True, backbone=args.backbone)
    model.compile(optimizer=models.Adam(lr=LR))
    out = {}
    # the pool is repeated to 2,048 frames (32 steps per epoch) so that the once-per-epoch work of fit() - loss
    # read-back, history, callbacks - weighs as little as in a real epoch of hundreds of steps
    rep = max(1, 2048 // Xu.shape[0])
    Xu, Y = np.concatenate([Xu] * rep), np.concatenate([Y] * rep)
    for label, X in (("uint8_frames", Xu), ("float32_frames", normalise_host(Xu))):
        steps = X.shape[0] // B
        model.fit(X, Y, batch_size=B, epochs=1, verbose=0)           # engine set-up, warm-up, graph capture
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        model.fit(X, Y, batch_size=B, epochs=2, verbose=0)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        out[label] = {"images_per_s": 2 * steps * B / dt, "ms_per_step": 1e3 * dt / (2 * steps), "steps_timed": 2 * steps}
    out["api"] = "SPNetModel.fit(X, Y, batch_size=%d) on host numpy arrays of %d frames, shuffled, host wall clock" % (B, Xu.shape[0])
    return out


def cpu_baseline():
    """Bounded CPU sample inside the default run: 5 timed training steps (2 warm-ups) of batch 32 + configs[0]."""
    dt, nsteps, ncores = cpu_train_steps(5, 2)
    return {"value": CPU_BATCH / dt, "unit": "images/s", "cores": ncores, "kind": "port",
            "sample": "median of %d timed steps (2 warm-ups) of %d images of the batch-64 workload, oracle torch-CPU fp32" % (nsteps, CPU_BATCH),
            "cfg1_forward_loss_batch32_images_per_s": cpu_cfg1()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--backbone", default="Xception", choices=["Xception", "MobileNet", "InceptionResNetV2"])
    ap.add_argument("--infer-frames", type=int, default=50_000, help="frames of the predict_spnet leg (whole job)")
    ap.add_argument("--infer-pool", type=int, default=512, help="distinct frames in the inference pool (cycled)")
    ap.add_argument("--infer-batch", type=int, default=BATCH_PER_GPU, dest="infer_batch", help="batch_size passed to SPNetModel.predict")
    ap.add_argument("--quick", action="store_true", help="diagnostic runs: skip the CPU baseline and the per-family roofline legs")
    ap.add_argument("--gemm-shapes", type=int, default=10, dest="gemm_shapes", help="how many GEMM shapes the per-shape table lists")
    ap.add_argument("--dump-outputs", metavar="DIR", dest="dump_outputs",
                    help="write what the last timed training step computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    args.steps_ref = max(1, min(args.steps, 3))
    args.warmup_ref = 1
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    # synthetic frames first: the generator forks worker processes, which must happen before CUDA / NCCL exist here
    nw = max(1, min(16, (os.cpu_count() or 1) // max(1, world)))
    Xu, Y = make_pool_u8(2 * BATCH_PER_GPU, 1_000_000 * rank, workers=nw)
    Xu_inf, Y_inf = make_pool_u8(args.infer_pool, 2_000_000 + 1_000_000 * rank, workers=nw)
    args.pools = (Xu, Y, Xu_inf)
    args.fit_Y = Y_inf
    # keep stdout clean for the single JSON line (NCCL prints its version banner to stdout)
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w")
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
        dist.init_process_group("nccl")
    run_ours(args, rank, world)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
