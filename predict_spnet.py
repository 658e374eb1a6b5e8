#! /usr/bin/env python3
"""Batch inference + hawley_spnet.csv — same CLI and behaviour as the reference's predict_spnet.py
(predict_network, :40-97; flags :100-115), running on the B200 engine. Extra flags (not in the
reference): --no-png skips the per-image PNG drawing, which at B200 inference rates is where all the
wall time goes; --dtype picks bf16 / fp32 compute."""
import glob
import os
import time

import numpy as np

from spnet.models import *   # noqa: F401,F403  (reference: `from spnet.models import *`)
from spnet.utils import *    # noqa: F401,F403
import spnet.config as cf
from spnet import models, utils

default_image_dir = "/home/shawley/datasets/zooniverse_steelpan/"


def _ranks():
    """(rank, world) of a torchrun launch (one process per GPU); (0, 1) otherwise."""
    return int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def predict_network(weights_file="spnet.model", datapath=default_image_dir, fraction=1.0, log_dir="logs/Predicting/",
                    batch_size=16, model=None, X_pred="", draw_images=True, stream_chunk=None, raw_u8=True, ranks=None):
    """stream_chunk (B200 build only): decode / predict the directory in chunks of that many frames, decoding chunk
    k+1 on the host threads while chunk k is on the GPU, instead of loading every frame into memory first.
    raw_u8: frames read from `datapath` travel to the GPU as uint8 and are normalised there (same values bit for bit);
    grayscale PNG frames used at their decoded size are also decoded there (utils.build_X(..., device=True)).

    Under `torchrun --nproc-per-node N` the sorted file list is cut into N contiguous shards, rank r predicts shard r on
    GPU r (no collective on the data path) and writes hawley_spnet.csv.part<r>; rank 0 then concatenates the parts in
    rank order, so the rows of hawley_spnet.csv are in sorted-file order exactly as in a single-process run."""
    img_file_list = None
    # ranks = (rank, world) overrides the torchrun environment: train_spnet.py's post-training pass runs on rank 0
    # ALONE (the other ranks have left), so it must not wait for their CSV parts
    rank, world = ranks if ranks is not None else _ranks()
    shard_lo = 0
    from_dir = isinstance(X_pred, str) and "" == X_pred
    streaming = stream_chunk is not None and from_dir
    if from_dir:
        print(f"Getting data from {datapath}, fraction = {fraction}.")
        if cf.model_type == "simple":
            grayscale, force_dim = False, 224
        elif cf.model_type == "big":
            grayscale, force_dim = True, None
        else:
            grayscale, force_dim = True, 331
        img_file_list = sorted(glob.glob(datapath + "/*.png"))
        if len(img_file_list) == 0:
            img_file_list += sorted(glob.glob(datapath + "/*.bmp"))
        total_files = len(img_file_list)
        total_load = int(total_files * fraction)
        if batch_size is not None:
            total_load = utils.nearest_multiple(total_load, batch_size)
        print("      Total files = ", total_files, ", going to load total_load = ", total_load)
        img_file_list = img_file_list[:total_load]
        if world > 1:
            # contiguous shards of the sorted list (the last ranks take one frame less when it does not divide)
            per, extra = divmod(total_load, world)
            shard_lo = rank * per + min(rank, extra)
            img_file_list = img_file_list[shard_lo:shard_lo + per + (1 if rank < extra else 0)]
            total_load = len(img_file_list)
            print("      rank %d / %d: frames [%d, %d)" % (rank, world, shard_lo, shard_lo + total_load))
    if model is None:
        print("Loading model from", weights_file)
        if ".hdf5" in weights_file:
            print("   Defining model, then loading weights")
            if from_dir:  # setup_model reads only X[0].shape: the frame shape the loaders will deliver
                if force_dim is None:
                    from PIL import Image
                    w, h = Image.open(img_file_list[0]).size
                    X_pred = np.zeros((1, h, w, 1 if grayscale else 3), np.float32)
                else:
                    X_pred = np.zeros((1, force_dim, force_dim, 1 if grayscale else 3), np.float32)
            model, serial_model = models.setup_model(X_pred, try_checkpoint=True, no_cp_fatal=True,
                                                     weights_file=weights_file, parallel=False, freeze_fac=0.0,
                                                     quick_setup=True)
        else:
            print("   Loading whole model")
            model = models.load_model(weights_file)
    # frames whose model input is the force_dim square travel at their decoded size and are resized on the GPU, the
    # same bytes as PIL's LANCZOS (a directory of mixed frame sizes is resized on the host, as the loaders fall back)
    defer = (from_dir and raw_u8 and grayscale and force_dim is not None
             and (getattr(model, "H", None), getattr(model, "W", None)) == (force_dim, force_dim))
    # frames used at their decoded size are decoded on this process's GPU (spnet_b200.png: the bytes PIL decodes; files
    # outside the PNG subset it takes, and frames it rejects, are decoded by PIL)
    device = from_dir and raw_u8 and grayscale and (defer or force_dim is None)

    def predict(X):
        if defer:
            return model.predict(X, batch_size=batch_size, resize=tuple(X.shape[1:3]) != (force_dim, force_dim))
        return model.predict(X, batch_size=batch_size)

    if from_dir:
        if streaming:
            chunks = utils.stream_X(img_file_list, int(stream_chunk), force_dim=force_dim, grayscale=grayscale, raw_u8=raw_u8,
                                    defer_resize=defer, device=device)
            first_lo, X_pred = next(chunks)
        else:
            X_pred, img_dims = utils.build_X(total_load, img_file_list, force_dim=force_dim, grayscale=grayscale,
                                             raw_u8=raw_u8, defer_resize=defer, device=device)
        print("")
    m = len(img_file_list) if streaming else X_pred.shape[0]
    print("    Predicting... (m = ", m, " frames in dataset)", sep="")
    start_time = time.time()
    if streaming:
        parts = [predict(X_pred)]
        for _, Xc in chunks:
            parts.append(predict(Xc))
        Y_pred = np.concatenate(parts, axis=0)
    else:
        Y_pred = predict(X_pred)
    elapsed = time.time() - start_time
    print("    ...elapsed time to predict = ", elapsed, "s.   FPS = ", m * 1.0 / elapsed)

    print("    Drawing ellipse images...")
    utils.make_sure_path_exists(log_dir)
    pred_shape = [6, 6, 2, cf.vars_per_pred]
    utils.setup_means_and_ranges(pred_shape)
    if img_file_list is None:
        img_file_list = ["frame_%07d.png" % i for i in range(m)]
        draw_images = False
    Yp, decoded = decode_on_device(Y_pred)
    out_csv = log_dir + "hawley_spnet.csv"
    if world > 1:
        utils.show_pred_ellipses(Yp, Yp, img_file_list, num_draw=m, log_dir=log_dir, out_csv=out_csv + ".part%d" % rank,
                                 show_true=False, draw_images=False, decoded=decoded)
        merge_csv_parts(out_csv, rank, world)
    else:
        utils.show_pred_ellipses(Yp, Yp, img_file_list, num_draw=m, log_dir=log_dir, out_csv=out_csv,
                                 show_true=False, draw_images=draw_images, decoded=decoded)
    return model


def merge_csv_parts(out_csv, rank, world, timeout_s=600.0):
    """Rank-ordered concatenation of the per-rank CSV parts (row order = sorted file order). Each rank publishes
    `<part>.done` after closing its part; rank 0 waits for all of them (the file system is the only thing the ranks
    share on this path - no process group, no collective), concatenates and removes the parts."""
    # the marker carries a token shared by the ranks of THIS launch (same torchrun parent, same rendezvous port), so a
    # marker left behind by an earlier run in the same directory is never mistaken for this run's
    token = "%s_%d" % (os.environ.get("MASTER_PORT", "0"), os.getppid())
    done = lambda r: out_csv + ".part%d.done_%s" % (r, token)  # noqa: E731
    open(done(rank), "w").close()
    if rank != 0:
        return
    t0 = time.time()
    for r in range(world):
        while not os.path.exists(done(r)):
            if time.time() - t0 > timeout_s:
                raise RuntimeError("predict_network: rank %d never delivered %s.part%d" % (r, out_csv, r))
            time.sleep(0.01)
    with open(out_csv, "w") as f:
        for r in range(world):
            with open(out_csv + ".part%d" % r) as g:
                f.write(g.read())
    for r in range(world):
        os.remove(out_csv + ".part%d" % r)
        os.remove(done(r))


def decode_on_device(Y_pred):
    """denorm_Y + integer rounding + existence flags in one CUDA kernel (ops.decode_detections)."""
    import torch
    from spnet_b200 import ops
    y = torch.from_numpy(np.ascontiguousarray(Y_pred, np.float32)).cuda()
    means = torch.from_numpy(np.asarray(utils.means, np.float32)).cuda()
    ranges = torch.from_numpy(np.asarray(utils.ranges, np.float32)).cuda()
    denorm, ints, exists = ops.decode_detections(y, means, ranges)
    return denorm.cpu().numpy(), (ints.cpu().numpy().astype(np.int64), exists.cpu().numpy().astype(bool))


if __name__ == "__main__":
    np.random.seed(1)
    import argparse
    parser = argparse.ArgumentParser(description="tests network on test dataset",
                                     formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    parser.add_argument("-w", "--weights", help="weights file in hdf5 format", default="spnet.model")
    parser.add_argument("-d", "--datapath", help="Dataset directory with list of images", default=default_image_dir)
    parser.add_argument("-f", "--fraction", type=float, help="Fraction of dataset to use", default=1.0)
    parser.add_argument("-l", "--logdir", help="Directory of log/output files", default="logs/Predicting/")
    parser.add_argument("-b", "--batch_size", type=int, help="Batch size to use", default=16)
    parser.add_argument("--no-png", action="store_true", help="write only hawley_spnet.csv, skip the per-image PNGs")
    parser.add_argument("--stream", type=int, default=None, metavar="N",
                        help="decode and predict N frames at a time (next chunk decoded while this one is on the GPU)")
    parser.add_argument("--dtype", choices=["bf16", "fp32"], default=cf.compute_dtype)
    parser.add_argument("--model_type", default=cf.model_type, help="'big' keeps 384x512 input, default resizes to 331x331")
    args = parser.parse_args()
    cf.compute_dtype = args.dtype
    cf.model_type = args.model_type
    if _ranks()[1] > 1:
        import torch
        # one process per GPU, no process group needed (more ranks than GPUs share them round-robin)
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)) % max(1, torch.cuda.device_count()))
    model = predict_network(weights_file=args.weights, datapath=args.datapath, fraction=args.fraction,
                            log_dir=args.logdir, batch_size=args.batch_size, draw_images=not args.no_png,
                            stream_chunk=args.stream)
