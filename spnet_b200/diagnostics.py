"""Evaluation metrics with the reference's names (spnet/diagnostics.py): calc_errors, compute_iou, precision,
calc_map - computed on the GPU (csrc/diagnostics.cu through the C ABI; there is no CPU path).

The reference's calc_map rasterises 2 x 72 x N anti-aliased 512 x 384 ellipse masks with cv2 for EACH of its ten
thresholds; here every (image, slot) pair's IoU comes out of one kernel launch and the ten precisions are
counted from that matrix. The rasteriser is an integer port of cv2's own (polygon of the ellipse, anti-aliased
edges with their pixel values, convex fill): intersection and union are the reference's pixel counts, so IoU,
precision and mAP are the reference's numbers bit for bit (tests/test_diagnostics.py against
tests/golden/ref_diagnostics.npz). calc_errors is exact."""
import numpy as np

from . import config as cf


def _dev(a):
    import torch
    if torch.is_tensor(a):
        return a.to("cuda", torch.float32).contiguous()
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


def calc_errors(Yp, Yt):
    """Ring-count and existence errors of denormalised predictions (diagnostics.py:13-60). Returns
    (ring_miscounts, ring_truecounts, total_obj, false_obj_pos, false_obj_neg, true_obj_pos, true_obj_neg,
    pix_err, ipem)."""
    import torch
    from . import ops
    yp, yt = _dev(Yp), _dev(Yt)
    counters, pix_err = ops.calc_errors(yp, yt)
    c = [int(v) for v in counters.cpu().numpy()]
    pe = pix_err.cpu().numpy()
    return c[0], c[1], c[2], c[3], c[4], c[5], c[6], pe, int(np.argmax(pe))


def iou_matrix(Yp, Yt):
    """IoU of every (image, predictor slot) pair: intersection / union of the reference's pixel counts in float64, and
    -1 where the reference's compute_iou returns -1 (union = 0)."""
    from . import ops
    counts = ops.ellipse_iou(_dev(Yp), _dev(Yt)).cpu().numpy().astype(np.float64)
    inter, union = counts[..., 0], counts[..., 1]
    iou = np.full(union.shape, -1.0)
    live = union > 0
    iou[live] = inter[live] / union[live]   # num_i / num_u in double, as the reference divides
    return iou


def compute_iou(args_p, args_t, display=False):
    """One pair of 8-tuples (cx, cy, a, b, cos2t, sin2t, noobj, rings), diagnostics.py:85-120."""
    v = iou_matrix(np.asarray(args_p, np.float32).reshape(1, -1), np.asarray(args_t, np.float32).reshape(1, -1))[0, 0]
    return -1 if v < 0 else float(v)


def precision(Yp, Yt, thresh=0.5, iou=None):
    """diagnostics.py:125-150 (prints the same two lines)."""
    Yp, Yt = np.asarray(Yp), np.asarray(Yt)
    iou = iou_matrix(Yp, Yt) if iou is None else iou
    v = cf.vars_per_pred
    p_no, t_no = Yp[:, cf.ind_noobj::v], Yt[:, cf.ind_noobj::v]
    live = iou >= 0
    hit = live & (iou > thresh)
    fp = live & ~hit & (p_no < 0.5) & (t_no >= 0.5)
    fn = live & ~hit & ~fp & (p_no >= 0.5) & (t_no < 0.5)
    tp_count, fp_count, fn_count = int(hit.sum()), int(fp.sum()), int(fn.sum())
    print("precision: thresh = ", thresh, ",tp_count, fp_count, fn_count = ", tp_count, fp_count, fn_count)
    prec = tp_count / (tp_count + fp_count + fn_count)
    print("precision: thresh, prec = ", thresh, prec)
    return prec, tp_count, fp_count, fn_count


def calc_map(Yp, Yt):
    """Mean average precision over the IoU thresholds 0.5 ... 0.95 (diagnostics.py:153-162); one IoU pass."""
    print("\ncalc_map: Calculating mean average precision. Yp.shape[0] =", np.asarray(Yp).shape[0])
    iou = iou_matrix(Yp, Yt)
    threshes = [0.5, 0.55, 0.6, 0.65, 0.7, 0.75, 0.8, 0.85, 0.9, 0.95]
    return sum(precision(Yp, Yt, thresh=t, iou=iou)[0] for t in threshes) / len(threshes)
