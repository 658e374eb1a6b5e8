"""PNG decoding on the device: the kernel alone, and predict_spnet's frame path with the decode on the host or the GPU.

    python tests/micro/png_bench.py [--out png_bench.json] [--frames 2048] [--dir DIR]

(a) spnet_png_decode_u8 on 384x512 fake_espi frames written by Pillow (filter 0, two IDAT chunks) and by cv2 (filter 1
    on every row, many IDAT chunks), at 64, 512 and 2048 frames per launch: CUDA events around >= 50 launches after a
    warm-up, each launch on the next of several stream/scratch/output sets whose total exceeds the 126 MB L2. Reported:
    us per launch, frames/s, and compressed (stream bytes in) and inflated (scanline bytes) GB/s.
(b) Frames/s of the monolithic default over `--frames` fake_espi PNGs (written before any timing), bf16, batch 64:
    host/host     = utils.build_X(force_dim=331, raw_u8=True) + model.predict(X)
    host/device   = utils.build_X(..., defer_resize=True) + model.predict(X, resize=True)      (the parent's default)
    device/device = utils.build_X(..., defer_resize=True, device=True) + model.predict(X, resize=True)
    each whole-set and through utils.stream_X in chunks of 512. The routes alternate three times in one process and
    their outputs must be equal.
The card's name and power limit are read in the same run and printed with the numbers."""
import argparse
import io
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


def frame(seed):
    from spnet_b200 import fake_espi
    img, _ = fake_espi.make_frame(seed)
    return img.reshape(img.shape[0], img.shape[1])


def encode(img, writer):
    if writer == "pillow":
        from PIL import Image
        f = io.BytesIO()
        Image.fromarray(img).save(f, format="PNG")
        return f.getvalue()
    import cv2
    return cv2.imencode(".png", img)[1].tobytes()


def kernel_alone(writer, n, distinct=256, launches=50):
    import torch
    from spnet_b200 import ops, png
    streams = [png.parse(encode(frame(20000 + i), writer))[3] for i in range(distinct)]
    H, W = 384, 512
    per_set = None
    sets = []
    rng = np.random.default_rng(n)
    while True:
        order = rng.permutation(np.arange(n) % distinct)
        chosen = [streams[i] for i in order]
        offs = np.zeros(n + 1, np.int64)
        np.cumsum([len(s) for s in chosen], out=offs[1:])
        buf = torch.from_numpy(np.frombuffer(b"".join(chosen), np.uint8).copy()).cuda()
        scratch = torch.empty(n * H * (1 + W), dtype=torch.uint8, device="cuda")
        out = torch.empty((n, H, W), dtype=torch.uint8, device="cuda")
        sets.append((buf, torch.from_numpy(offs).cuda(), scratch, out))
        per_set = int(offs[-1]) + scratch.numel() + out.numel()
        if len(sets) >= 2 and len(sets) * per_set > 300 * 2 ** 20:
            break
    for i in range(len(sets)):
        st = ops.png_decode_u8(sets[i][0], sets[i][1], H, W, 1, sets[i][3], scratch=sets[i][2])
        assert not st.any().item()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(launches):
        b, o, s, out = sets[i % len(sets)]
        ops.png_decode_u8(b, o, H, W, 1, out, scratch=s)
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / launches
    comp = np.mean([sets[k][0].numel() for k in range(len(sets))])
    inflated = n * H * (1 + W)
    return {"writer": writer, "n": n, "sets_rotated": len(sets), "working_set_MB": round(len(sets) * per_set / 2 ** 20, 1),
            "launches": launches, "us_per_launch": round(us, 1), "frames_per_s": round(n / (us * 1e-6)),
            "compressed_GBps": round(comp / (us * 1e-6) / 1e9, 2), "inflated_GBps": round(inflated / (us * 1e-6) / 1e9, 2)}


def write_pngs(d, n):
    from PIL import Image
    files = []
    for i in range(n):
        p = os.path.join(d, "steelpan_%07d.png" % i)
        if not os.path.exists(p):
            Image.fromarray(frame(10000 + i)).save(p)
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
    utils.build_X(min(n, 64), files, force_dim=331, grayscale=True, raw_u8=True, defer_resize=True, device=True)
    torch.cuda.synchronize()
    routes = {"host/host": dict(), "host/device": dict(defer_resize=True), "device/device": dict(defer_resize=True, device=True)}

    def whole(kw):
        t0 = time.perf_counter()
        X, _ = utils.build_X(n, files, force_dim=331, grayscale=True, raw_u8=True, **kw)
        if torch.is_tensor(X):
            torch.cuda.synchronize()
        t1 = time.perf_counter()
        Y = model.predict(X, batch_size=bs, resize=bool(kw))
        t2 = time.perf_counter()
        return {"build_X_s": t1 - t0, "predict_s": t2 - t1, "frames_per_s": n / (t2 - t0)}, Y

    def streamed(kw):
        t0 = time.perf_counter()
        parts = [model.predict(X, batch_size=bs, resize=bool(kw))
                 for _, X in utils.stream_X(files, chunk, force_dim=331, grayscale=True, raw_u8=True, **kw)]
        t1 = time.perf_counter()
        return {"total_s": t1 - t0, "frames_per_s": n / (t1 - t0)}, np.concatenate(parts)

    rows, ref = [], None
    for r in range(rounds):
        for route, kw in routes.items():
            w, yw = whole(kw)
            s, ys = streamed(kw)
            ref = yw if ref is None else ref
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
        sys.exit("png_bench: no CUDA device")
    import __graft_entry__
    __graft_entry__.build()
    res = {"card": card(), "cpus": os.cpu_count(), "kernel": []}
    for writer in ("pillow", "cv2"):
        for n in (64, 512, 2048):
            res["kernel"].append(kernel_alone(writer, n))
            print(json.dumps(res["kernel"][-1]), flush=True)
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
