"""ORACLE — test infrastructure only (never imported by the product path).

CPU restatement of the reference's evaluation metrics (spnet/diagnostics.py) for the device kernels in
spnet_b200/csrc/diagnostics.cu:

* calc_errors (:13-60): exact restatement (integer counters, first-predictor pixel error). Pinned bit for bit
  against the reference's own output in tests/golden/ref_diagnostics.npz.
* compute_iou (:85-120): the reference rasterises both ellipses with cv2.ellipse(..., thickness=-1, LINE_AA,
  shift=10) on a 512 x 384 canvas and counts non-zero pixels, i.e. every pixel the ANTI-ALIASED filled polygon
  touches. That rasteriser (third-party: OpenCV drawing.cpp) is restated in integers in oracle/cv2_raster.py and
  pinned pixel for pixel against cv2 itself; the IoUs here are therefore the reference's own, bit for bit
  (tests/test_diagnostics.py compares with tests/golden/ref_diagnostics.npz).
* precision (:125-150) and calc_map (:153-162): exact restatements on top of the IoU matrix.
"""
import numpy as np

VARS = 8  # spnet/config.py:30
THRESHES = (0.5, 0.55, 0.6, 0.65, 0.7, 0.75, 0.8, 0.85, 0.9, 0.95)  # diagnostics.py:156


def _round_half_even_int(x):
    return int(round(float(x)))  # Python round(): half to even, as the reference's int(round(.))


def calc_errors(Yp, Yt):
    """diagnostics.py:13-60. Returns (ring_miscounts, ring_truecounts, total_obj, false_obj_pos, false_obj_neg,
    true_obj_pos, true_obj_neg, pix_err, ipem)."""
    slots = Yt.shape[1] // VARS
    diff = Yp - Yt
    pix_err = np.sqrt(diff[:, 0] ** 2 + diff[:, 1] ** 2)
    ipem = np.argmax(pix_err)
    miss = true = total = fpos = fneg = tpos = tneg = 0
    for j in range(Yt.shape[0]):
        for an in range(slots):
            ind, i_noobj = 7 + an * VARS, 6 + an * VARS
            if _round_half_even_int(Yt[j, i_noobj]) == 0:
                total += 1
                if _round_half_even_int(Yp[j, i_noobj]) == 0:
                    tpos += 1
                    if np.abs(Yt[j, ind] - Yp[j, ind]) > 0.5:
                        miss += 1
                    else:
                        true += 1
                else:
                    fneg += 1
            elif _round_half_even_int(Yp[j, i_noobj]) == 0:
                fpos += 1
            else:
                tneg += 1
    return miss, true, total, fpos, fneg, tpos, tneg, pix_err, ipem


def ellipse_mask(args, nx=512, ny=384):
    """EXACT: the pixels the reference's create_ellipse_image (:68-80) leaves non-zero, through the integer restatement
    of cv2's anti-aliased filled-polygon rasteriser (oracle/cv2_raster.py, pinned pixel for pixel against cv2)."""
    from . import cv2_raster
    cx, cy, a, b, c2, s2, noobj = [np.float32(v) for v in args[:7]]
    if not noobj < 0.5:
        return np.zeros((ny, nx), bool)
    angle = np.rad2deg(np.arctan2(s2, c2) / 2.0)   # float32 arithmetic, as the reference's numpy scalars
    return cv2_raster.ellipse_mask(cx, cy, a, b, angle, nx, ny)


def ellipse_image(args, nx=512, ny=384):
    """uint8 canvas with the reference's pixel VALUES (create_ellipse_image :68-80): arguments keep their dtype, exactly as
    the reference's numpy scalars do (float32 rows of Yp / Yt, or Python floats)."""
    from . import cv2_raster
    cx, cy, a, b, c2, s2, noobj = args[:7]
    if not noobj < 0.5:
        return np.zeros((ny, nx), np.uint8)
    angle = np.rad2deg(np.arctan2(s2, c2) / 2.0)
    return cv2_raster.ellipse_image(cx, cy, a, b, angle, nx, ny)


def compute_iou(args_p, args_t):
    """diagnostics.py:85-120: -1 when the true slot is empty (noobj > 0.99) or neither ellipse is drawn. Intersection /
    union are counted on cv2.bitwise_and / bitwise_or of the pixel VALUES (two partially covered edge pixels can AND to
    zero), as the reference does."""
    if args_t[6] > 0.99:
        return -1.0
    vp, vt = ellipse_image(args_p), ellipse_image(args_t)
    ni, nu = int(((vp & vt) != 0).sum()), int(((vp | vt) != 0).sum())
    if ni == 0 and nu == 0:
        return -1.0
    return ni / nu


def iou_matrix(Yp, Yt):
    n, slots = Yp.shape[0], Yp.shape[1] // VARS
    out = np.zeros((n, slots))
    for i in range(n):
        for s in range(slots):
            out[i, s] = compute_iou(Yp[i, s * VARS:(s + 1) * VARS], Yt[i, s * VARS:(s + 1) * VARS])
    return out


def precision_from_iou(iou, Yp, Yt, thresh=0.5):
    """diagnostics.py:125-150 given the IoU of every (image, slot)."""
    tp = fp = fn = 0
    for i in range(iou.shape[0]):
        for s in range(iou.shape[1]):
            v = iou[i, s]
            if v < 0:
                continue
            p_no, t_no = Yp[i, s * VARS + 6], Yt[i, s * VARS + 6]
            if v > thresh:
                tp += 1
            elif p_no < 0.5 and t_no >= 0.5:
                fp += 1
            elif p_no >= 0.5 and t_no < 0.5:
                fn += 1
    return tp / (tp + fp + fn), tp, fp, fn


def calc_map_from_iou(iou, Yp, Yt):
    """diagnostics.py:153-162."""
    return sum(precision_from_iou(iou, Yp, Yt, t)[0] for t in THRESHES) / len(THRESHES)
