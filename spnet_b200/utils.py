"""Host side of the data <-> tensor codec, same names / arguments / error behaviour as the
reference's spnet/utils.py for the functions on the hot path's boundary (SURVEY.md §8a rows
A1-A3, D1, X1): grid assignment and normalisation of targets, image loading, detection
decoding and the hawley_spnet.csv writer.

Detection decoding for prediction runs on the device (ops.decode_detections: denormalise,
round-half-even integers, existence flags); the host only formats the rows.
"""
import csv
import errno
import glob
import os
import random
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from . import config as cf

orig_img_dims = [512, 384]
means = []
ranges = []


def make_sure_path_exists(path):
    try:
        os.makedirs(path)
    except OSError as exception:
        if exception.errno != errno.EEXIST:
            raise


def nearest_multiple(a, b):
    return int(a / b) * b


def add_to_stack(a, b):
    if a is None:
        return [b]
    return a + [b]


# ------------------------------------------------------------------ targets
def setup_means_and_ranges(pred_shape):
    """Per-cell defaults / means / ranges (spnet/utils.py:144-176). Sets the module globals
    `means`, `ranges`; returns (cx_min, cy_min, cx_max, cy_max, xbinsize, ybinsize, gridYi)."""
    global means, ranges
    cx_min, cy_min, cx_max, cy_max = 40, 40, 470, 350
    nx, ny = int(pred_shape[0]), int(pred_shape[1])
    xbin = int((cx_max - cx_min) / nx)
    ybin = int((cy_max - cy_min) / ny)
    shape = tuple(int(s) for s in pred_shape)
    gcx = (np.arange(nx) * xbin + cx_min + xbin / 2)[:, None, None]
    gcy = (np.arange(ny) * ybin + cy_min + ybin / 2)[None, :, None]
    defaults = np.zeros(shape, dtype=cf.dtype)
    gmeans = np.zeros(shape, dtype=cf.dtype)
    granges = np.zeros(shape, dtype=cf.dtype)
    defaults[..., 0], defaults[..., 1] = gcx, gcy
    defaults[..., 2:] = [xbin / 2, ybin / 2, -1, 0, 1, 0]
    gmeans[..., 0], gmeans[..., 1] = gcx, gcy
    gmeans[..., 2:] = [xbin / 2, ybin / 2, 0, 0, 0, 5]
    granges[...] = [xbin, ybin, xbin, ybin, 2, 2, 1, 10]
    means = gmeans.flatten()
    ranges = granges.flatten()
    return cx_min, cy_min, cx_max, cy_max, xbin, ybin, defaults


def norm_Y(Y, set_means_ranges=False):
    return (Y - means) / ranges


def denorm_Y(normY):
    return normY * ranges + means


def true_to_pred_grid(true_arr, pred_shape, num_classes=11, img_filename=None):
    """YOLO-style assignment (spnet/utils.py:191-244): cell = trunc((c - 40)/bin) clamped to the
    grid, slot = arrival order in the cell; AssertionError when a cell gets more antinodes than
    it has predictors."""
    cx_min, cy_min, _, _, xbin, ybin, grid = setup_means_and_ranges(pred_shape)
    true_arr = np.asarray(true_arr, dtype=np.float64)
    if true_arr.size == 0:
        return grid
    true_arr = true_arr.reshape(-1, cf.vars_per_pred)
    # float64 divide then truncation toward zero, exactly as int(x / bin) does
    ix = np.clip(np.trunc((true_arr[:, 0] - cx_min) / xbin).astype(np.int64), 0, int(pred_shape[0]) - 1)
    iy = np.clip(np.trunc((true_arr[:, 1] - cy_min) / ybin).astype(np.int64), 0, int(pred_shape[1]) - 1)
    counts = np.zeros(grid.shape[0:2], dtype=np.int64)
    for an in range(true_arr.shape[0]):
        slot = counts[ix[an], iy[an]]
        assert slot < pred_shape[2]
        grid[ix[an], iy[an], slot] = true_arr[an]
        counts[ix[an], iy[an]] = slot + 1
    return grid


def parse_meta_rows(rows):
    """rows of [cx, cy, a, b, angle, rings] -> sorted list of 8-variable antinode rows
    (spnet/utils.py:260-286: drop duplicate rows, a >= b with angle += 90 on swap, rings > 0 only)."""
    seen, arrs = set(), []
    for r in rows:
        key = tuple(float(v) for v in r[:6])
        if key in seen:
            continue
        seen.add(key)
        cx, cy, a, b, angle, rings = key
        if b > a:
            a, b = b, a
            angle = angle + 90
        if rings > 0.0:
            t = 2 * np.deg2rad(angle)
            arrs.append([cx, cy, a, b, np.cos(t), np.sin(t), 0, rings])
    return sorted(arrs, key=lambda r: (r[0], r[1]))


def parse_meta_file(meta_filename):
    rows = []
    with open(meta_filename, newline="") as f:
        for rec in csv.reader(f):
            if rec:
                rows.append([float(v) for v in rec[:6]])
    return parse_meta_rows(rows)


def build_Y_from_rows(list_of_rows, pred_grid=[6, 6, 2]):
    pred_shape = np.array([pred_grid[0], pred_grid[1], pred_grid[2], cf.vars_per_pred], dtype=int)
    Y = np.zeros([len(list_of_rows), int(np.prod(pred_shape))], dtype=cf.dtype)
    for i, rows in enumerate(list_of_rows):
        Y[i, :] = true_to_pred_grid(np.array(parse_meta_rows(rows)), pred_shape).flatten()
    setup_means_and_ranges(pred_shape)
    return norm_Y(Y).astype(cf.dtype), pred_shape


def pack_annotations(list_of_arrs):
    """[[8-variable antinode rows] per image] (parse_meta_file / parse_meta_rows output) -> (ann [n, max_obj, 8] float64,
    counts [n] int32): the device-side input of ops.assign_grid / ops.yolo_ellipse_loss_ann."""
    n = len(list_of_arrs)
    max_obj = max([len(a) for a in list_of_arrs] + [1])
    ann = np.zeros((n, max_obj, cf.vars_per_pred), np.float64)
    counts = np.zeros(n, np.int32)
    for i, a in enumerate(list_of_arrs):
        counts[i] = len(a)
        if len(a):
            ann[i, :len(a)] = np.asarray(a, np.float64).reshape(-1, cf.vars_per_pred)
    return ann, counts


def grid_tables(pred_shape, device):
    """(defaults, means, ranges) of setup_means_and_ranges as flat fp32 device tensors."""
    import torch
    _, _, _, _, _, _, defaults = setup_means_and_ranges(pred_shape)
    mk = lambda a: torch.from_numpy(np.ascontiguousarray(a, np.float32).ravel()).to(device)  # noqa: E731
    return mk(defaults), mk(means), mk(ranges)


def build_Y_device(list_of_arrs, pred_grid=[6, 6, 2], device="cuda"):
    """true_to_pred_grid + norm_Y for a whole dataset in ONE kernel launch (csrc/loss.cu assign_grid_kernel; the
    reference loops over images and antinodes in Python, spnet/utils.py:191-244,312-318). Returns the normalised
    targets as a CUDA tensor [n, prod(pred_shape)] (what SPNetModel.fit takes for a device-resident run) and
    pred_shape. Raises AssertionError exactly where the reference's `assert slot < preds_per_cell` (:240) would."""
    import torch
    from . import ops
    pred_shape = np.array([pred_grid[0], pred_grid[1], pred_grid[2], cf.vars_per_pred], dtype=int)
    ann, counts = pack_annotations(list_of_arrs)
    defaults, mean_t, range_t = grid_tables(pred_shape, device)
    Y, err = ops.assign_grid(torch.from_numpy(ann).to(device), torch.from_numpy(counts).to(device), defaults, mean_t, range_t,
                             int(pred_grid[0]), int(pred_grid[1]), int(pred_grid[2]))
    bad = torch.nonzero(err).flatten()
    assert bad.numel() == 0, "true_to_pred_grid: image %d offers more than %d antinodes to one grid cell (antinode %d)" % (
        int(bad[0]), int(pred_grid[2]), int(err[bad[0]]) - 1)
    return Y, pred_shape


def build_Y(total_load, meta_file_list, img_file_list, pred_grid=[6, 6, 2], set_means_ranges=False):
    pred_shape = np.array([pred_grid[0], pred_grid[1], pred_grid[2], cf.vars_per_pred], dtype=int)
    Y = np.zeros([total_load, int(np.prod(pred_shape))], dtype=cf.dtype)
    for i in range(total_load):
        if 0 == i % 5000:
            print("      Reading metadata file i =", i, "/", total_load, ":", meta_file_list[i])
        arrs = parse_meta_file(meta_file_list[i])
        Y[i, :] = true_to_pred_grid(np.array(arrs), pred_shape, img_filename=img_file_list[i]).flatten()
    setup_means_and_ranges(pred_shape)
    return norm_Y(Y, set_means_ranges=set_means_ranges).astype(cf.dtype), pred_shape


# ------------------------------------------------------------------ images
def _load_one(args):
    filename, force_dim, grayscale = args[:3]
    raw_u8 = len(args) > 3 and args[3]
    from PIL import Image
    img = Image.open(filename).convert("RGB")
    if force_dim is not None:
        img = img.resize((force_dim, force_dim), Image.LANCZOS)
    if raw_u8:  # pixel values as decoded (and resized) by PIL: the normalisation below then runs on the device
        arr = np.asarray(img, dtype=np.uint8)
        return arr[:, :, 0:1] if grayscale else arr
    arr = np.asarray(img, dtype=np.float32)
    arr = arr / 255.0
    arr -= 0.5
    arr *= 2.0
    return arr[:, :, 0:1] if grayscale else arr


def build_X(total_load, img_file_list, force_dim=224, grayscale=False, raw_u8=False, defer_resize=False, device=False):
    """Images -> X float32 NHWC in [-1,1] (spnet/utils.py:325-421): PIL decode, optional LANCZOS
    resize to a force_dim square, (v/255 - 0.5)*2, channel 0 only when grayscale.
    raw_u8 (B200 build only): return the uint8 pixel values instead; SPNetModel.predict / the engine apply the
    same normalisation on the device, bit for bit, and a quarter of the bytes cross PCIe.
    defer_resize (B200 build only; with raw_u8, grayscale and a force_dim): leave the LANCZOS resize to the device
    (SPNetModel.predict(X, resize=True), the same bytes as PIL's) and return the frames at their decoded size - unless
    one frame's size differs from the first's, in which case the whole call returns the host-resized frames.
    device (B200 build only; with raw_u8, grayscale, and force_dim None or defer_resize): decode the PNGs on the
    current CUDA device (spnet_b200.png, the bytes PIL decodes) and return X as a CUDA uint8 tensor; frames of
    different sizes, or a file PIL fails on, make the call return (or raise) what it does without `device`."""
    print("      Reading images and assigning as input X...")
    if device and raw_u8 and grayscale and (force_dim is None or defer_resize):
        X = _device_frames(img_file_list[:total_load])
        if X is not None:
            return X, (X.shape[1], X.shape[2], 3)
    defer = defer_resize and raw_u8 and grayscale and force_dim is not None
    dim = None if defer else force_dim
    first = _load_one((img_file_list[0], dim, grayscale, raw_u8))
    img_dims = first.shape if not grayscale else (first.shape[0], first.shape[1], 3)
    X = np.zeros((total_load,) + first.shape, dtype=np.uint8 if raw_u8 else cf.dtype)
    nproc = os.cpu_count() or 1
    ragged = False
    with ThreadPoolExecutor(nproc) as ex:
        for i, arr in enumerate(ex.map(_load_one, [(f, dim, grayscale, raw_u8) for f in img_file_list[:total_load]])):
            if defer and arr.shape != first.shape:
                ragged = True
                break
            X[i] = arr
    if ragged:
        return build_X(total_load, img_file_list, force_dim=force_dim, grayscale=grayscale, raw_u8=raw_u8)
    return X, img_dims


def _device_frames(files, items=None, decoder=None):
    """uint8 frames [n, H, W, 1] decoded on the current CUDA device (spnet_b200.png), or None when the host route
    must run instead (frames of different sizes, or a file PIL fails on). items: png.read of each file, when the caller
    has read them already; decoder: the png.Decoder to reuse (stream_X keeps one per generator)."""
    import torch
    from . import png
    if items is None:
        with ThreadPoolExecutor(os.cpu_count() or 1) as ex:
            items = list(ex.map(png.read, files))
    dev = torch.device("cuda", torch.cuda.current_device())
    return (decoder or png.Decoder()).frames(files, items, dev)


def stream_X(img_file_list, chunk, force_dim=224, grayscale=False, raw_u8=False, defer_resize=False, device=False):
    """Generator over (start, X_chunk): the frames of build_X in chunks of `chunk` files, the NEXT chunk being
    decoded by the worker threads while the caller consumes the current one (SURVEY.md section 8(f) rank 1: at
    B200 inference rates PIL decode, not the network, bounds predict_spnet over tens of thousands of frames, and
    the whole set no longer has to fit in host memory). Values are identical to build_X's, chunk by chunk
    (defer_resize: native-size frames, or the host-resized ones for a chunk whose frames differ in size; device: CUDA
    uint8 frames decoded on the device, the worker threads reading and parsing the next chunk's files while the
    caller consumes this one, or the host route's values for a chunk whose frames differ in size)."""
    nproc = os.cpu_count() or 1
    n = len(img_file_list)
    defer = defer_resize and raw_u8 and grayscale and force_dim is not None
    on_device = device and raw_u8 and grayscale and (force_dim is None or defer_resize)

    def host(files):
        with ThreadPoolExecutor(nproc) as ex:
            frames = list(ex.map(_load_one, [(f, None if defer else force_dim, grayscale, raw_u8) for f in files]))
            if defer and any(a.shape != frames[0].shape for a in frames):
                frames = list(ex.map(_load_one, [(f, force_dim, grayscale, raw_u8) for f in files]))
        return np.stack(frames).astype(np.uint8 if raw_u8 else cf.dtype)

    def decode(lo):
        files = img_file_list[lo:lo + chunk]
        if not on_device:
            return host(files)
        with ThreadPoolExecutor(nproc) as ex:
            return list(ex.map(png.read, files))

    from . import png
    decoder = png.Decoder() if on_device else None
    with ThreadPoolExecutor(1) as bg:
        fut = bg.submit(decode, 0) if n else None
        lo = 0
        while lo < n:
            X = fut.result()
            nxt = lo + chunk
            fut = bg.submit(decode, nxt) if nxt < n else None
            if on_device:  # the copy and the launch are issued here, on the caller's thread and current stream
                files = img_file_list[lo:lo + chunk]
                Xd = _device_frames(files, X, decoder)
                X = Xd if Xd is not None else host(files)
            yield lo, X
            lo = nxt


def build_dataset(path="Train/", load_frac=1.0, set_means_ranges=False, pred_grid=[6, 6, 2], batch_size=None,
                  shuffle=True):
    """spnet/utils.py:425-482."""
    if cf.model_type == "simple":
        grayscale, force_dim = False, 224
    elif cf.model_type == "big":
        grayscale, force_dim = True, None
    else:
        grayscale, force_dim = True, 331
    print("Loading data from", path, ", fraction =", load_frac)
    img_file_list = sorted(glob.glob(path + "*.png"))
    meta_file_list = sorted(glob.glob(path + "*" + cf.meta_extension))
    assert len(img_file_list) == len(meta_file_list), "Error: len(img_file_list) = " + str(len(img_file_list)) + \
        " but len(meta_file_list) = " + str(len(meta_file_list))
    if shuffle:
        c = list(zip(img_file_list, meta_file_list))
        random.shuffle(c)
        img_file_list, meta_file_list = zip(*c)
    total_files = len(img_file_list)
    total_load = int(total_files * load_frac)
    if batch_size is not None:
        total_load = nearest_multiple(total_load, batch_size)
    print("      Total files = ", total_files, ", going to load total_load = ", total_load)
    Y, pred_shape = build_Y(total_load, meta_file_list, img_file_list, pred_grid=pred_grid,
                            set_means_ranges=set_means_ranges)
    X, img_dims = build_X(total_load, img_file_list, force_dim=force_dim, grayscale=grayscale)
    return X, Y, img_file_list, pred_shape


# ------------------------------------------------------------------ decode + CSV
def cleanup_antinode_vars(Y_subarr):
    """spnet/utils.py:56-64."""
    [cx, cy, a, b, cos2t, sin2t, noobj, rings] = Y_subarr
    [cx, cy, a, b, noobj] = [int(round(x)) for x in [cx, cy, a, b, noobj]]
    angle = np.rad2deg(np.arctan2(sin2t, cos2t) / 2.0)
    angle = angle if angle > 0 else angle + 180
    return cx, cy, a, b, angle, noobj, rings


def _angles(Yp):
    """float32 angle column for every predictor, same op sequence as cleanup_antinode_vars."""
    v = cf.vars_per_pred
    ang = np.rad2deg(np.arctan2(Yp[:, cf.ind_angle2::v], Yp[:, cf.ind_angle1::v]) / np.float32(2.0))
    return np.where(ang > 0, ang, ang + np.float32(180)).astype(Yp.dtype)


def decode_host(Yp):
    """(ints [n,npred,5], exists [n,npred]) from denormalised Yp — numpy statement of what
    ops.decode_detections computes on the device."""
    v = cf.vars_per_pred
    cols = [Yp[:, i::v] for i in (cf.ind_cx, cf.ind_cy, cf.ind_semi_a, cf.ind_semi_b, cf.ind_noobj)]
    ints = np.stack([np.rint(c).astype(np.int64) for c in cols], axis=-1)
    exists = (ints[..., 4] == 0) & (Yp[:, cf.ind_rings::v] > 0) & (ints[..., 2] >= 0) & (ints[..., 3] >= 0)
    return ints, exists


def csv_rows(Yp, ints, exists, file_list):
    """One text block per image, rows in predictor order: cx,cy,filename,rings,a,b,angle
    (spnet/utils.py:122-126). The reference formats numpy float32 scalars with "{}".format, which prints the value as a
    Python float (shortest repr of the double): the columns are converted to Python lists once and formatted with %r /
    %d - the same text, without a numpy scalar per field."""
    v = cf.vars_per_pred
    ang = _angles(Yp)
    rings = Yp[:, cf.ind_rings::v]
    n = Yp.shape[0]
    jj, aa = np.nonzero(np.asarray(exists)[:n])
    sel = np.asarray(ints)[jj, aa]
    c0, c1, c4, c5 = (sel[:, i].tolist() for i in range(4))
    r = np.asarray(rings[jj, aa], dtype=np.float64).tolist()
    g = np.asarray(ang[jj, aa], dtype=np.float64).tolist()
    counts = np.bincount(jj, minlength=n).tolist()
    out, k = [], 0
    for j in range(n):
        base = os.path.basename(file_list[j])
        m = counts[j]
        if m == 0:
            out.append("0,0," + base + ",0,0,0,0\n")
            continue
        out.append("".join(["%d,%d,%s,%r,%d,%d,%r\n" % (c0[i], c1[i], base, r[i], c4[i], c5[i], g[i]) for i in range(k, k + m)]))
        k += m
    return out


def draw_ellipse(img, center, axes, angle, startAngle=0, endAngle=360, color=(0), thickness=2, lineType=None, shift=10):
    import cv2
    lineType = cv2.LINE_AA if lineType is None else lineType
    center = (int(round(center[0] * 2 ** shift)), int(round(center[1] * 2 ** shift)))
    axes = (int(round(axes[0] * 2 ** shift)), int(round(axes[1] * 2 ** shift)))
    return cv2.ellipse(img, center, axes, -angle, startAngle, endAngle, color, thickness, lineType, shift)


def show_pred_ellipses(Yt, Yp, file_list, num_draw=40, log_dir="./logs/", ind_extra=None, out_csv=None, show_true=True,
                       verbosity=0, draw_images=True, decoded=None):
    """Same contract as spnet/utils.py:67-137: Yt, Yp are DE-normalised; writes one PNG per
    image into log_dir (skipped with draw_images=False — a B200-side option: at 10^4 img/s the
    PNG drawing, not the network, dominates predict_spnet) and the zooniverse-style CSV.
    `decoded` = (ints, exists) from the device decode kernel; computed on the host if absent."""
    m = Yt.shape[0]
    num_draw = min(num_draw, m, len(file_list))
    Yp = np.asarray(Yp)
    ints, exists = decoded if decoded is not None else decode_host(Yp[:num_draw])
    blocks = csv_rows(Yp[:num_draw], ints[:num_draw], exists[:num_draw], file_list)
    if out_csv is not None:
        with open(out_csv, "w") as f:
            f.write("".join(blocks))
    if not draw_images:
        return
    import cv2
    from PIL import Image
    ang = _angles(Yp[:num_draw])
    if show_true:
        Yt = np.asarray(Yt)
        t_ints, t_exists = decode_host(Yt[:num_draw])
        t_ang = _angles(Yt[:num_draw])
    for j in range(num_draw):
        img = cv2.cvtColor(np.array(Image.open(file_list[j]).convert("RGB")), cv2.COLOR_RGB2BGR)
        layers = ([(Yt, t_ints, t_exists, t_ang, cf.truecolor, cf.black, 0)] if show_true else []) + \
                 [(Yp, ints, exists, ang, cf.predcolor, cf.lightgrey, 27)]
        for Y, ii, ee, aa, color, bg, yo in layers:
            for an in np.nonzero(ee[j])[0]:
                cx, cy, a, b = (int(v) for v in ii[j, an, :4])
                draw_ellipse(img, [cx, cy], [a, b], float(aa[j, an]), color=color, thickness=3)
                txt = "{: >3.1f}".format(float(Y[j, an * cf.vars_per_pred + cf.ind_rings]))
                cv2.putText(img, txt, (cx - 12, cy + yo), cv2.FONT_HERSHEY_TRIPLEX, 0.95, color=bg, thickness=2, lineType=cv2.LINE_AA)
                cv2.putText(img, txt, (cx - 10, cy + yo), cv2.FONT_HERSHEY_TRIPLEX, fontScale=0.9, color=color, thickness=1, lineType=cv2.LINE_AA)
        name = os.path.basename(file_list[j])
        cv2.putText(img, name, (7, orig_img_dims[1] - 3), cv2.FONT_HERSHEY_SIMPLEX, 0.55, cf.black, lineType=cv2.LINE_AA)
        cv2.putText(img, name, (5, orig_img_dims[1] - 5), cv2.FONT_HERSHEY_SIMPLEX, 0.55, cf.white, lineType=cv2.LINE_AA)
        cv2.imwrite(log_dir + "/steelpan_pred_" + str(j).zfill(5) + ".png", img)
