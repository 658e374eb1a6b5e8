"""LANCZOS resize on the device: the kernel alone, and predict_spnet's frame path with the resize on the host or the GPU.

    python tests/micro/resize_bench.py [--out resize_bench.json] [--frames 2048] [--dir DIR]

(a) spnet_resize_lanczos_u8, 384x512 -> 331x331, at 64 and 512 frames: CUDA events around >= 200 launches after a
    warm-up, each launch on the next of several input/output sets whose total exceeds the 126 MB L2, so every launch
    reads its frames from HBM. Algorithmic bytes per launch: n * (H*W + 4*OH*OW) (uint8 in, fp32 out).
(b) Frames/s of the monolithic default over `--frames` fake_espi PNGs (written before any timing), bf16, batch 64:
    host route   = utils.build_X(force_dim=331, raw_u8=True) + model.predict(X)
    device route = utils.build_X(..., defer_resize=True) + model.predict(X, resize=True)
    and both through utils.stream_X in chunks of 512. The routes alternate three times in one process; the decode
    (build_X) and predict times are reported apart, and the device route's build_X is the decode-only time.
The card's name and power limit are read in the same run and printed with the numbers."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def kernel_alone(n, launches=200, H=384, W=512, OH=331, OW=331):
    import torch
    from spnet_b200 import ops
    per = n * (H * W + 4 * OH * OW)
    sets = max(2, -(-300 * 2 ** 20 // per))  # > 2x the 126 MB L2 in rotation
    g = torch.Generator(device="cuda").manual_seed(n)
    xs = [torch.randint(0, 256, (n, H, W), dtype=torch.uint8, device="cuda", generator=g) for _ in range(sets)]
    outs = [torch.empty((n, OH, OW), device="cuda") for _ in range(sets)]
    for i in range(2 * sets):
        ops.resize_lanczos_u8(xs[i % sets], OH, OW, out=outs[i % sets])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(launches):
        ops.resize_lanczos_u8(xs[i % sets], OH, OW, out=outs[i % sets])
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / launches
    return {"n": n, "sets_rotated": sets, "working_set_MB": round(sets * per / 2 ** 20, 1), "launches": launches,
            "us_per_launch": round(us, 2), "algorithmic_GBps": round(per / (us * 1e-6) / 1e9, 1)}


def write_pngs(d, n):
    from PIL import Image
    from spnet_b200 import fake_espi
    files = []
    for i in range(n):
        p = os.path.join(d, "steelpan_%07d.png" % i)
        if not os.path.exists(p):
            img, _ = fake_espi.make_frame(10000 + i)
            Image.fromarray(img.reshape(img.shape[0], img.shape[1])).save(p)
        files.append(p)
    return files


def end_to_end(files, rounds=3, bs=64, chunk=512):
    import torch
    import spnet.config as cf
    from spnet import models, utils
    cf.model_type, cf.compute_dtype = "monolithic", "bf16"
    model, _ = models.setup_model(np.zeros((1, 331, 331, 1), np.float32), 576, try_checkpoint=False, freeze_fac=0.0,
                                  quick_setup=True)
    n = len(files)
    model.predict(np.zeros((bs, 331, 331, 1), np.uint8), batch_size=bs)  # engine, graph capture, resize tables warm
    model.predict(np.zeros((bs, 384, 512, 1), np.uint8), batch_size=bs, resize=True)
    torch.cuda.synchronize()

    def whole(defer):
        t0 = time.perf_counter()
        X, _ = utils.build_X(n, files, force_dim=331, grayscale=True, raw_u8=True, defer_resize=defer)
        t1 = time.perf_counter()
        Y = model.predict(X, batch_size=bs, resize=defer)
        t2 = time.perf_counter()
        return {"build_X_s": t1 - t0, "predict_s": t2 - t1, "frames_per_s": n / (t2 - t0)}, Y

    def streamed(defer):
        t0 = time.perf_counter()
        parts = [model.predict(X, batch_size=bs, resize=defer)
                 for _, X in utils.stream_X(files, chunk, force_dim=331, grayscale=True, raw_u8=True, defer_resize=defer)]
        t1 = time.perf_counter()
        return {"total_s": t1 - t0, "frames_per_s": n / (t1 - t0)}, np.concatenate(parts)

    rows = []
    for r in range(rounds):
        for route, defer in (("host", False), ("device", True)):
            w, yw = whole(defer)
            s, ys = streamed(defer)
            if route == "host":
                ref = yw
            assert np.array_equal(yw, ref) and np.array_equal(ys, ref), "routes disagree"
            rows.append({"round": r, "route": route, "whole": {k: round(v, 4) for k, v in w.items()},
                         "stream": {k: round(v, 4) for k, v in s.items()}})
            print(json.dumps(rows[-1]), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--frames", type=int, default=2048)
    ap.add_argument("--dir", default=None, help="directory for the PNGs (default: a temporary one)")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("resize_bench: no CUDA device")
    import __graft_entry__
    __graft_entry__.build()
    res = {"card": card(), "cpus": os.cpu_count(), "kernel": [kernel_alone(64), kernel_alone(512)]}
    print(json.dumps(res), flush=True)
    with tempfile.TemporaryDirectory() as tmp:
        d = args.dir or tmp
        os.makedirs(d, exist_ok=True)
        files = write_pngs(d, args.frames)
        res["frames"] = len(files)
        res["end_to_end"] = end_to_end(files)
    res["card_after"] = card()
    print(json.dumps({"card": res["card"], "card_after": res["card_after"]}))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
