"""Tensor-level wrappers over the C ABI (include/spnet_b200.h).

PyTorch is used only as the owner of device memory and streams: every function here
forwards raw device pointers and shapes to libspnet_b200.so on the current CUDA stream.
Nothing in this module computes with torch ops, and nothing falls back to them.
"""
import math

import torch

from ._lib import lib

F32, BF16 = 0, 1


def _p(t):
    return None if t is None else t.data_ptr()


def _s():
    return torch.cuda.current_stream().cuda_stream


def dtype_code(t):
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise TypeError("activation tensors must be float32 or bfloat16, got %s" % t.dtype)


def _chk(*ts):
    for t in ts:
        if t is not None:
            assert t.is_cuda and t.is_contiguous(), "spnet_b200 ops need contiguous CUDA tensors"


# ----------------------------------------------------------------------------- loss / head
def yolo_ellipse_loss(y_true, y_pred, hybrid=False, sel_sigmoid=False, out6=None, grad=None):
    _chk(y_true, y_pred, out6, grad)
    B, n = y_pred.shape
    if out6 is None:
        out6 = torch.empty(6, device=y_pred.device, dtype=torch.float32)
    lib().yolo_ellipse_loss(_p(y_true), _p(y_pred), B, n, int(hybrid), int(sel_sigmoid), _p(out6), _p(grad), _s())
    return out6


def selective_sigmoid_fwd(x, start, end, skip, out=None):
    _chk(x, out)
    rows, n = x.shape
    end = n if end is None else (end if end >= 0 else n + end)
    if out is None:
        out = torch.empty_like(x)
    lib().selective_sigmoid_fwd(_p(x), _p(out), rows, n, start, end, skip, _s())
    return out


def selective_sigmoid_bwd(y, dy, start, end, skip, out=None):
    _chk(y, dy, out)
    rows, n = y.shape
    end = n if end is None else (end if end >= 0 else n + end)
    if out is None:
        out = torch.empty_like(dy)
    lib().selective_sigmoid_bwd(_p(y), _p(dy), _p(out), rows, n, start, end, skip, _s())
    return out


def decode_detections(y, means, ranges):
    _chk(y, means, ranges)
    n, ncols = y.shape
    denorm = torch.empty_like(y)
    ints = torch.empty(n, ncols // 8, 5, device=y.device, dtype=torch.int32)
    exists = torch.empty(n, ncols // 8, device=y.device, dtype=torch.uint8)
    lib().decode_detections(_p(y), _p(means), _p(ranges), n, ncols, _p(denorm), _p(ints), _p(exists), _s())
    return denorm, ints, exists


# ----------------------------------------------------------------------------- depthwise
def dwconv3x3_fwd(x, k, in_a=None, in_b=None, relu=False, out=None):
    _chk(x, k, in_a, in_b, out)
    B, H, W, C = x.shape
    if out is None:
        out = torch.empty_like(x)
    lib().dwconv3x3_fwd(_p(x), _p(k), _p(in_a), _p(in_b), int(relu), _p(out), dtype_code(x), B, H, W, C, _s())
    return out


def dwconv3x3_bwd_fused(gout, x, k, dk, in_a=None, in_b=None, relu=False, bn_mean=None, bn_rstd=None, stats=None,
                        add_src=None, add_strided=None, out=None, acc=None, zo=None, zo_mean=None, zo_rstd=None,
                        zo_stats=None, mask_a=None, mask_b=None):
    """gin, dk (+=) and optional BatchNorm-backward sums in one pass (see dwconv_packed.cu).
    zo: raw input of the BatchNorm whose output gradient gin is; its sums go to zo_stats, taken on the final gin,
    which is first masked by (mask_a*zo + mask_b > 0) when mask_a/mask_b are given."""
    _chk(gout, x, k, dk, in_a, in_b, stats, add_src, add_strided, out, zo, zo_mean, zo_rstd, zo_stats, mask_a, mask_b)
    B, H, W, C = gout.shape
    if out is None:
        out = torch.empty_like(gout)
    lib().dwconv3x3_bwd_fused(_p(gout), _p(x), _p(k), _p(in_a), _p(in_b), int(relu), _p(bn_mean), _p(bn_rstd),
                              _p(stats), _p(add_src), _p(add_strided), _p(out), _p(dk), _p(acc), dtype_code(gout), B, H, W, C,
                              _p(zo), _p(zo_mean), _p(zo_rstd), _p(zo_stats), _p(mask_a), _p(mask_b), _s())
    if acc is not None:  # order-independent kernel gradient: accumulators -> dk (+=), accumulators cleared
        lib().acc_to_f32(_p(acc), _p(dk), dk.numel(), 1, 1, _s())
    return out


# ----------------------------------------------------------------------------- GEMM
OUT_T, OUT_F32, OUT_ATOMIC, OUT_SLAB = 0, 1, 2, 3


def slab_reduce(slabs, nslabs, M, N, out, bias=None, accumulate=False, ldo=None, slab_stride=None):
    """out[M,N] = [out +] bias + slab_0 + slab_1 + ... in that order (slabs: zero-initialised [nslabs, M, N] fp32 buffer
    written by gemm(..., out_mode=OUT_SLAB, splits=nslabs); slabs the GEMM did not need stay zero)."""
    _chk(slabs, out, bias)
    lib().slab_reduce(_p(slabs), nslabs, slab_stride if slab_stride is not None else M * N, N, _p(bias), _p(out),
                      ldo if ldo is not None else N, M, N, int(accumulate), _s())
    return out


def gemm(A, a_mn, B, b_mn, D, M, N, K, out_mode=OUT_T, splits=1, colstats=None, lda=None, ldb=None, ldd=None,
         slab_stride=None):
    """D[M,N] (op)= A[M,K] @ B[K,N].

    a_mn / b_mn False: operand stored [rows, K] (K contiguous); True: stored [K, rows].
    bf16 operands run on tcgen05 (gemm_tc.cu), fp32 operands on the exact FFMA kernel.
    out_mode OUT_SLAB: split s of the K range stores its partial product at D + s * slab_stride elements (default
    M * N: a dense [splits, M, N] buffer) - fixed-order split-K (slab_reduce) or a batch of GEMMs stacked along K.
    """
    _chk(A, B, D, colstats)
    lda = lda if lda is not None else (M if a_mn else K)
    ldb = ldb if ldb is not None else (N if b_mn else K)
    ldd = ldd if ldd is not None else N
    ss = (slab_stride if slab_stride is not None else M * ldd) if out_mode == OUT_SLAB else 0
    if A.dtype == torch.bfloat16:
        assert B.dtype == torch.bfloat16
        lib().gemm_bf16(_p(A), lda, int(a_mn), _p(B), ldb, int(b_mn), _p(D), ldd, ss, out_mode, M, N, K, splits,
                        _p(colstats), _s())
    else:
        assert A.dtype == torch.float32 and B.dtype == torch.float32
        sa = (1, lda) if a_mn else (lda, 1)
        sb = (1, ldb) if b_mn else (ldb, 1)
        lib().gemm_simt(_p(A), sa[0], sa[1], _p(B), sb[0], sb[1], _p(D), ldd, ss, out_mode, M, N, K, splits, _p(colstats),
                        _s())
    return D


def conv_tc_fwd(x, wt, y, pt, pl, colstats=None, ldx=None, ldy=None):
    """y[B,OH,OW,Cout] = conv(x[B,H,W,Cin], wt[KH,KW,Cin,Cout]), stride 1, bf16, implicit GEMM on tcgen05.
    x / y may be channel slices of wider NHWC buffers (ldx / ldy = pixel stride in elements)."""
    _chk(wt, colstats)
    assert x.is_cuda and y.is_cuda and (ldx is not None or x.is_contiguous()) and (ldy is not None or y.is_contiguous())
    B, H, W, Cin = x.shape
    KH, KW, _, Cout = wt.shape
    lib().conv_tc_fwd(_p(x), ldx or Cin, B, H, W, Cin, _p(wt), _p(y), ldy or Cout, y.shape[1], y.shape[2], Cout, KH, KW,
                      pt, pl, _p(colstats), _s())
    return y


def conv_tc_fwd_kwfold(x, wt, y, colstats=None):
    """'valid' convolution of a dense NHWC tensor, the KW taps of a filter row folded into the channel axis
    (csrc/gemm_tc.cu spnet_conv_tc_fwd_kwfold): y[B,H-KH+1,W-KW+1,Cout]."""
    _chk(x, wt, y, colstats)
    assert x.is_contiguous() and y.is_contiguous()
    B, H, W, Cin = x.shape
    KH, KW, _, Cout = wt.shape
    assert tuple(y.shape) == (B, H - KH + 1, W - KW + 1, Cout)
    lib().conv_tc_fwd_kwfold(_p(x), B, H, W, Cin, _p(wt), _p(y), Cout, Cout, KH, KW, _p(colstats), _s())
    return y


def conv_tc_wgrad_kwfold(x, gy, gw):
    """gw[KH,KW,Cin,Cout] (fp32) += weight gradient of conv_tc_fwd_kwfold."""
    _chk(x, gy, gw)
    assert x.is_contiguous() and gy.is_contiguous() and gw.is_contiguous()
    B, H, W, Cin = x.shape
    KH, KW, _, Cout = gw.shape
    assert tuple(gy.shape) == (B, H - KH + 1, W - KW + 1, Cout)
    lib().conv_tc_wgrad_kwfold(_p(x), B, H, W, Cin, _p(gy), Cout, Cout, _p(gw), KH, KW, _s())
    return gw


def conv_tc_dgrad(gy, wt, gx, pt, pl, ldy=None, ldx=None):
    """gx[B,H,W,Cin] = data gradient of conv_tc_fwd from gy[B,OH,OW,Cout] (overwrites gx)."""
    _chk(gy, wt, gx)
    B, OH, OW, Cout = gy.shape
    KH, KW, Cin, _ = wt.shape
    lib().conv_tc_dgrad(_p(gy), ldy or Cout, B, OH, OW, Cout, _p(wt), _p(gx), ldx or Cin, gx.shape[1], gx.shape[2], Cin,
                        KH, KW, pt, pl, _s())
    return gx


def conv_tc_wgrad(x, gy, gw, pt, pl, ldx=None, ldy=None):
    """gw[KH,KW,Cin,Cout] (fp32) += x (*) gy."""
    _chk(x, gy, gw)
    B, H, W, Cin = x.shape
    _, OH, OW, Cout = gy.shape
    KH, KW = gw.shape[0], gw.shape[1]
    lib().conv_tc_wgrad(_p(x), ldx or Cin, B, H, W, Cin, _p(gy), ldy or Cout, OH, OW, Cout, _p(gw), KH, KW, pt, pl, _s())
    return gw


# ----------------------------------------------------------------------------- batch norm
def bn_finalize(stats, count, gamma, beta, a, b, save_mean, save_rstd, moving_mean=None, moving_var=None,
                eps=1e-3, momentum=0.99, unbiased=True):
    C = a.numel()
    lib().bn_finalize(_p(stats), count, _p(gamma), _p(beta), eps, momentum, int(unbiased), _p(a), _p(b),
                      _p(save_mean), _p(save_rstd), _p(moving_mean), _p(moving_var), C, _s())


def bn_inference_affine(gamma, beta, moving_mean, moving_var, a, b, eps=1e-3, save_mean=None, save_rstd=None):
    lib().bn_inference_affine(_p(gamma), _p(beta), _p(moving_mean), _p(moving_var), eps, _p(a), _p(b), _p(save_mean),
                              _p(save_rstd), a.numel(), _s())


def bn_apply(z, a, b, act=0, x=None, out=None):
    _chk(z, a, b, x, out)
    C = z.shape[-1]
    rows = z.numel() // C
    if out is None:
        out = torch.empty_like(z)
    lib().bn_apply(_p(z), _p(a), _p(b), act, _p(x), _p(out), dtype_code(z), rows, C, _s())
    return out


def bn_bwd_reduce(g, z, save_mean, save_rstd, stats, relu_a=None, relu_b=None, act=1):
    _chk(g, z, stats)
    C = z.shape[-1]
    rows = z.numel() // C
    lib().bn_bwd_reduce(_p(g), _p(z), _p(save_mean), _p(save_rstd), _p(relu_a), _p(relu_b), act, _p(stats),
                        dtype_code(z), rows, C, _s())


def bn_bwd_finalize(stats, count, dgamma, dbeta, c1, c2):
    lib().bn_bwd_finalize(_p(stats), count, _p(dgamma), _p(dbeta), _p(c1), _p(c2), c1.numel(), _s())


def bn_bwd_dz(g, z, a, save_mean, save_rstd, c1, c2, out=None):
    _chk(g, z, out)
    C = z.shape[-1]
    rows = z.numel() // C
    if out is None:
        out = torch.empty_like(g)
    lib().bn_bwd_dz(_p(g), _p(z), _p(a), _p(save_mean), _p(save_rstd), _p(c1), _p(c2), _p(out), dtype_code(z), rows,
                    C, _s())
    return out


def pw_bwd_bn_slabs(M, device=None):
    """Slabs spnet_pw_bwd_bn writes in deterministic mode: one per CTA of its persistent grid."""
    n_sms = torch.cuda.get_device_properties(device if device is not None else torch.cuda.current_device()).multi_processor_count
    return min(-(-M // 128), n_sms)


def pw_bwd_bn(g, z, t, W, a, save_mean, save_rstd, c1, c2, gA, gW, M, cin, cout, slabs=None):
    """Backward of a pointwise conv z = t W followed by a BatchNorm, in one kernel: dz = bn_bwd_dz(g, z, ...) stays on
    chip, gA [M, cin] = dz W^T, gW [cin, cout] += t^T dz. bn_bwd_finalize must have run. slabs (fp32, at least
    pw_bwd_bn_slabs(M) * cin * cout): the weight gradient goes through per-CTA slabs added in a fixed order."""
    _chk(g, z, t, W, gA, gW, slabs)
    n = pw_bwd_bn_slabs(M, g.device) if slabs is not None else 0
    lib().pw_bwd_bn(_p(g), _p(z), _p(t), _p(W), _p(a), _p(save_mean), _p(save_rstd), _p(c1), _p(c2), _p(gA), _p(gW),
                    _p(slabs), n, M, cin, cout, _s())
    if slabs is not None:
        slab_reduce(slabs, n, cin, cout, gW, accumulate=True)
    return gA


def augment_on_the_fly(x_orig, x, seed, max_regions=6, minsize=11, maxsize=75, sp_prob=0.5, sp_amount=0.004,
                       salt_vs_pepper=0.2):
    """x[n,H,W,C] = cutout + salt-and-pepper copy of the pristine frames x_orig (fp32, on the device)."""
    _chk(x_orig, x)
    assert x_orig.dtype == torch.float32 and x.dtype == torch.float32 and x.shape == x_orig.shape
    n, H, W, C = x.shape
    lib().augment_on_the_fly(_p(x_orig), _p(x), n, H, W, C, int(seed) & (2 ** 63 - 1), max_regions, minsize, maxsize,
                             sp_prob, sp_amount, salt_vs_pepper, _s())
    return x


def calc_errors(yp, yt):
    """-> (counters int32 [7], pix_err fp32 [n]); yp / yt denormalised fp32 [n, ncols] on the device."""
    _chk(yp, yt)
    n, ncols = yp.shape
    counters = torch.zeros(7, device=yp.device, dtype=torch.int32)
    pix_err = torch.empty(n, device=yp.device, dtype=torch.float32)
    lib().calc_errors(_p(yp), _p(yt), n, ncols, _p(counters), _p(pix_err), _s())
    return counters, pix_err


def ellipse_iou(yp, yt):
    """-> int32 [n, ncols/8, 2] = (intersection, union) pixel counts of the reference's raster; union = 0 marks a pair
    the reference scores -1."""
    _chk(yp, yt)
    n, ncols = yp.shape
    cnt = torch.empty(n, ncols // 8, 2, device=yp.device, dtype=torch.int32)
    lib().ellipse_iou(_p(yp), _p(yt), n, ncols, _p(cnt), _s())
    return cnt


# ----------------------------------------------------------------------------- pooling
def maxpool3s2_add_fwd(z, a=None, b=None, res=None, ra=None, rb=None, out=None, argmax=None):
    _chk(z, res, out, argmax)
    B, H, W, C = z.shape
    if out is None:
        out = torch.empty(B, (H + 1) // 2, (W + 1) // 2, C, device=z.device, dtype=z.dtype)
    lib().maxpool3s2_add_fwd(_p(z), _p(a), _p(b), _p(res), _p(ra), _p(rb), _p(out), _p(argmax), dtype_code(z), B, H,
                             W, C, _s())
    return out


def maxpool3s2_bwd(gout, argmax, H, W, out=None, z=None, mean=None, rstd=None, stats=None):
    """gin; with z (the raw input of the BatchNorm whose output was pooled) also that BatchNorm's backward sums
    (sum gin, sum gin*xhat) into stats, over gin as stored."""
    _chk(gout, argmax, out, z, mean, rstd, stats)
    B, OH, OW, C = gout.shape
    if out is None:
        out = torch.empty(B, H, W, C, device=gout.device, dtype=gout.dtype)
    lib().maxpool3s2_bwd(_p(gout), _p(argmax), _p(out), dtype_code(gout), B, H, W, C, _p(z), _p(mean), _p(rstd),
                         _p(stats), _s())
    return out


def _off2(off):
    return (off, off) if isinstance(off, int) else (int(off[0]), int(off[1]))


def gather_s2(x, out=None, off=0):
    """out[b,oh,ow] = x[b, 2*oh+off_h, 2*ow+off_w]; off = int or (off_h, off_w)."""
    _chk(x, out)
    B, H, W, C = x.shape
    oh, ow = _off2(off)
    if out is None:
        out = torch.empty(B, (H + 1 - oh) // 2, (W + 1 - ow) // 2, C, device=x.device, dtype=x.dtype)
    lib().gather_s2(_p(x), _p(out), dtype_code(x), B, H, W, C, oh, ow, _s())
    return out


def scatter_s2(x, out, off=0):
    """Adjoint of gather_s2: x [B,OH,OW,C] -> out [B,H,W,C] (zero where nothing lands)."""
    _chk(x, out)
    B, H, W, C = out.shape
    oh, ow = _off2(off)
    lib().scatter_s2(_p(x), _p(out), dtype_code(x), B, H, W, C, oh, ow, _s())
    return out


def colstats(z, stats):
    _chk(z, stats)
    C = z.shape[-1]
    lib().colstats(_p(z), _p(stats), dtype_code(z), z.numel() // C, C, _s())


# ----------------------------------------------------------------------------- stem / block1
def conv_small_fwd(which, x, w, out, skip=None, in_a=None, in_b=None, act=0, stats=None):
    _chk(x, w, out, skip, stats)
    B, H, W = x.shape[0], x.shape[1], x.shape[2]
    lib().conv_small_fwd(which, _p(x), _p(w), _p(in_a), _p(in_b), act, _p(out), _p(skip), _p(stats), dtype_code(out),
                         B, H, W, _s())
    return out


def conv_small_wgrad(which, x, g, dw, in_a=None, in_b=None, act=0, acc=None):
    """dw += weight gradient. acc: accumulator scratch (stats_alloc, >= dw.numel() entries, all zero): the cross-CTA sums
    then go through the order-independent accumulators (bit-identical run to run) and are added into dw afterwards."""
    _chk(x, g, dw, acc)
    B, H, W = x.shape[0], x.shape[1], x.shape[2]
    lib().conv_small_wgrad(which, _p(x), _p(in_a), _p(in_b), act, _p(g), _p(dw), _p(acc), dtype_code(g), B, H, W, _s())
    if acc is not None:
        lib().acc_to_f32(_p(acc), _p(dw), dw.numel(), 1, 1, _s())
    return dw


def conv_small_dgrad(which, g, w, gin, mask_z=None, mask_a=None, mask_b=None, act=0):
    _chk(g, w, gin, mask_z)
    B, H, W = gin.shape[0], gin.shape[1], gin.shape[2]
    lib().conv_small_dgrad(which, _p(g), _p(w), _p(mask_z), _p(mask_a), _p(mask_b), act, _p(gin), dtype_code(g), B, H,
                           W, _s())
    return gin


def stem_k3_to_k4(k3, k4):
    lib().stem_k3_to_k4(_p(k3), _p(k4), k3.shape[-1], _s())


def stem_k4grad_to_k3grad(g4, g3):
    lib().stem_k4grad_to_k3grad(_p(g4), _p(g3), g3.shape[-1], _s())


def stem_out_fwd(c3, a, b, skip, out, rate=0.0, seed=None):
    lib().stem_out_fwd(_p(c3), _p(a), _p(b), _p(skip), _p(out), dtype_code(c3), c3.numel() // 3, rate, _p(seed), _s())
    return out


def stem_out_bwd(g, out, rate=0.0, seed=None):
    lib().stem_out_bwd(_p(g), _p(out), dtype_code(g), g.numel() // 3, rate, _p(seed), _s())
    return out


def bn3_bwd_reduce(g, z, save_mean, save_rstd, stats):
    lib().bn3_bwd_reduce(_p(g), _p(z), _p(save_mean), _p(save_rstd), _p(stats), dtype_code(z), z.numel() // 3, _s())


def bn3_bwd_dz(g, z, a, save_mean, save_rstd, c1, c2, out):
    lib().bn3_bwd_dz(_p(g), _p(z), _p(a), _p(save_mean), _p(save_rstd), _p(c1), _p(c2), _p(out), dtype_code(z),
                     z.numel() // 3, _s())
    return out


# ----------------------------------------------------------------------------- optimiser
def adam_keras_step(p, g, m, v, lr_t_dev, n_l2=0, l2=1e-4, beta1=0.9, beta2=0.999, eps=1e-7, grad_scale=1.0,
                    p_bf16=None, frozen8=None, g_bf16=None):
    """Keras-2.1.3 Adam on a flat range. frozen8: uint8 per 8 parameters (non-zero = not trainable);
    g_bf16: read the gradients from this bf16 buffer instead of g."""
    lib().adam_keras_step(_p(p), _p(g), _p(m), _p(v), p.numel(), n_l2, l2, _p(lr_t_dev), beta1, beta2, eps,
                          grad_scale, _p(p_bf16), _p(frozen8), _p(g_bf16), _s())


def sumsq(p, n, scale, acc):
    """acc (stats accumulator, 1 entry) += scale * sum(p[:n]^2); read it with acc_to_f32."""
    lib().sumsq(_p(p), n, scale, _p(acc), _s())


def acc_to_f32(acc, out, accumulate=False, clear=True):
    lib().acc_to_f32(_p(acc), _p(out), out.numel(), int(accumulate), int(clear), _s())
    return out


# ---- order-independent accumulators (csrc/common.cuh stat_add / stat_get): 2 int64 words per entry
def stats_alloc(n_entries, device):
    return torch.zeros(2 * n_entries, device=device, dtype=torch.int64)


def stats_values(st):
    """Decode an accumulator buffer into float64 values (host-side helper for tests / diagnostics)."""
    w = st.detach().cpu().view(-1, 2)
    return (w[:, 0].double() + w[:, 1].double() / 4294967296.0) / 16777216.0


def stats_from_values(vals, device):
    """Encode float64 values as accumulators (tests feed bn_finalize directly)."""
    t = vals.detach().cpu().double() * 16777216.0
    hi = torch.floor(t)
    lo = torch.floor((t - hi) * 4294967296.0)
    return torch.stack([hi.long(), lo.long()], 1).reshape(-1).contiguous().to(device)


# ----------------------------------------------------------------------------- host-path kernels
def assign_grid(ann, counts, defaults, means, ranges, nx=6, ny=6, ppc=2):
    """true_to_pred_grid + norm_Y on the device. ann [n, max_obj, 8] float64, counts [n] int32.
    Returns (Y [n, nx*ny*ppc*8] fp32, err [n] int32)."""
    _chk(ann, counts, defaults, means, ranges)
    assert ann.dtype == torch.float64 and counts.dtype == torch.int32
    n, max_obj = ann.shape[0], ann.shape[1]
    Y = torch.empty(n, nx * ny * ppc * 8, device=ann.device, dtype=torch.float32)
    err = torch.zeros(n, device=ann.device, dtype=torch.int32)
    lib().assign_grid(_p(ann), _p(counts), n, max_obj, nx, ny, ppc, _p(defaults), _p(means), _p(ranges), _p(Y), _p(err), _s())
    return Y, err


def yolo_ellipse_loss_ann(ann, counts, defaults, means, ranges, y_pred, nx=6, ny=6, ppc=2, hybrid=False, sel_sigmoid=False,
                          out6=None, grad=None, y_true_out=None):
    """custom_loss straight from the annotations (assignment + normalisation + loss + gradient in one launch).
    Returns (out6, err)."""
    _chk(ann, counts, defaults, means, ranges, y_pred, out6, grad, y_true_out)
    assert ann.dtype == torch.float64 and counts.dtype == torch.int32
    B, max_obj = ann.shape[0], ann.shape[1]
    assert y_pred.shape == (B, nx * ny * ppc * 8)
    if out6 is None:
        out6 = torch.empty(6, device=y_pred.device, dtype=torch.float32)
    err = torch.zeros(B, device=y_pred.device, dtype=torch.int32)
    lib().yolo_ellipse_loss_ann(_p(ann), _p(counts), max_obj, nx, ny, ppc, _p(defaults), _p(means), _p(ranges), _p(y_pred), B,
                                int(hybrid), int(sel_sigmoid), _p(y_true_out), _p(out6), _p(grad), _p(err), _s())
    return out6, err


_U8_LUT = {}


def normalize_u8(x_u8, out=None):
    """(v/255 - 0.5)*2 of spnet/utils.py:340-342 on uint8 frames, bit-exact to numpy's fp32 arithmetic (the 256
    possible results are computed by numpy itself and looked up on the device)."""
    _chk(x_u8, out)
    assert x_u8.dtype == torch.uint8
    if out is None:
        out = torch.empty(x_u8.shape, device=x_u8.device, dtype=torch.float32)
    lib().normalize_u8(_p(x_u8), _p(_u8_lut(x_u8.device)), _p(out), x_u8.numel(), _s())
    return out


def _u8_lut(device):
    """The 256 values of (v/255 - 0.5)*2 as numpy computes them in fp32, one device copy per device."""
    import numpy as np
    key = str(device)
    if key not in _U8_LUT:
        lut = np.arange(256, dtype=np.float32)
        lut = lut / 255.0
        lut -= 0.5
        lut *= 2.0
        _U8_LUT[key] = torch.from_numpy(lut.astype(np.float32)).to(device)
    return _U8_LUT[key]


_PB_ONE = float(1 << 22)  # Pillow's PRECISION_BITS = 32 - 8 - 2


def _lanczos(t):
    """Pillow's lanczos_filter (libImaging/Resample.c): sinc(t) * sinc(t/3) on [-3, 3), sinc(x) = sin(pi x) / (pi x)."""
    def sinc(x):
        if x == 0.0:
            return 1.0
        x = x * math.pi
        return math.sin(x) / x
    return sinc(t) * sinc(t / 3.0) if -3.0 <= t < 3.0 else 0.0


def lanczos_tables(in_size, out_size):
    """Pillow's LANCZOS coefficients for one axis in its 8-bit fixed point (precompute_coeffs + normalize_coeffs_8bpc
    of libImaging/Resample.c, float64 in Pillow's operation order): bounds int32 [out_size, 2] = (first input index,
    tap count), coeffs int32 [out_size, ksize] in units of 2^-22. Host only; resize_lanczos_u8 applies them."""
    import numpy as np
    if in_size < 1 or out_size < 1:
        raise ValueError("lanczos_tables: sizes must be positive, got %r -> %r" % (in_size, out_size))
    scale = in_size / out_size
    fs = max(scale, 1.0)
    support = 3.0 * fs
    ss = 1.0 / fs  # Pillow multiplies by 1/filterscale; dividing by filterscale can differ in the last bit
    ksize = int(math.ceil(support)) * 2 + 1
    bounds = np.zeros((out_size, 2), np.int32)
    coeffs = np.zeros((out_size, ksize), np.int32)
    for xx in range(out_size):
        center = (xx + 0.5) * scale
        xmin = max(int(center - support + 0.5), 0)
        count = min(int(center + support + 0.5), in_size) - xmin
        w = [_lanczos((x + xmin - center + 0.5) * ss) for x in range(count)]
        ww = 0.0
        for v in w:
            ww += v
        if ww != 0.0:
            w = [v / ww for v in w]
        bounds[xx] = (xmin, count)
        coeffs[xx, :count] = [int(v * _PB_ONE + (0.5 if v >= 0 else -0.5)) for v in w]
    return bounds, coeffs


_LANCZOS = {}


def resize_lanczos_u8(x_u8, OH, OW, out=None):
    """LANCZOS resize of uint8 frames [n, H, W] (or [n, H, W, 1]) to [n, OH, OW], fused with normalize_u8's
    (v/255 - 0.5)*2: out fp32 [n, OH, OW] (or any contiguous tensor of that many elements) = lut[resized byte]. The
    bytes are those of PIL's Image.resize((OW, OH), Image.LANCZOS) on each frame (spnet/utils.py:325-349)."""
    _chk(x_u8, out)
    if x_u8.dtype != torch.uint8:
        raise TypeError("resize_lanczos_u8 takes uint8 frames, got %s" % x_u8.dtype)
    if x_u8.dim() == 4 and x_u8.shape[3] == 1:
        x_u8 = x_u8.view(x_u8.shape[:3])
    if x_u8.dim() != 3:
        raise ValueError("resize_lanczos_u8 takes frames [n, H, W] or [n, H, W, 1], got %s" % (tuple(x_u8.shape),))
    n, H, W = x_u8.shape
    OH, OW = int(OH), int(OW)
    if out is None:
        out = torch.empty((n, OH, OW), device=x_u8.device, dtype=torch.float32)
    if out.dtype != torch.float32 or out.numel() != n * OH * OW:
        raise ValueError("resize_lanczos_u8: out must be fp32 with %d elements" % (n * OH * OW))
    key = (H, W, OH, OW, str(x_u8.device))
    if key not in _LANCZOS:
        xb, xc = lanczos_tables(W, OW)
        yb, yc = lanczos_tables(H, OH)
        _LANCZOS[key] = tuple(torch.from_numpy(a).to(x_u8.device) for a in (xb, xc, yb, yc))
    xb, xc, yb, yc = _LANCZOS[key]
    lib().resize_lanczos_u8(_p(x_u8), n, H, W, _p(xb), _p(xc), xc.shape[1], _p(yb), _p(yc), yc.shape[1],
                            _p(_u8_lut(x_u8.device)), _p(out), OH, OW, _s())
    return out


def png_decode_u8(streams, offsets, H, W, bpp, out, scratch=None):
    """Channel 0 of n PNG frames of one size and colour type (csrc/png.cu): streams uint8 = the frames' zlib streams
    (concatenated IDAT payloads) back to back, offsets int64 [n + 1], bpp bytes per pixel (1, 2, 3, 4 for colour
    types 0, 4, 2, 6), out uint8 [n, H, W] (or [n, H, W, 1]). Returns the int32 status per frame (0, or one of the
    header's SPNET_PNG_ERR_* codes; that frame's out bytes are then undefined). spnet_b200.png hides the container."""
    _chk(streams, offsets, out, scratch)
    if streams.dtype != torch.uint8 or out.dtype != torch.uint8 or offsets.dtype != torch.int64:
        raise TypeError("png_decode_u8 takes uint8 streams and out and int64 offsets")
    n = offsets.numel() - 1
    if n < 1 or out.numel() != n * H * W:
        raise ValueError("png_decode_u8: %d offsets for out %s of %dx%d frames" % (offsets.numel(), tuple(out.shape), H, W))
    if scratch is None:
        scratch = torch.empty(n * H * (1 + W * bpp), dtype=torch.uint8, device=out.device)
    status = torch.empty(n, dtype=torch.int32, device=out.device)
    lib().png_decode_u8(_p(streams), streams.numel(), _p(offsets), n, H, W, bpp, _p(scratch), scratch.numel(), _p(out),
                        _p(status), _s())
    return status


def cast_f32_to_bf16(src, dst):
    lib().cast_f32_to_bf16(_p(src), _p(dst), src.numel(), _s())


def colsum(g, out):
    rows, cols = g.shape
    lib().colsum(_p(g), _p(out), rows, cols, _s())


# ----------------------------------------------------------------------------- dense-convolution backbone pieces
def im2col(x, col, kh, kw, stride, pt, pl, oh, ow):
    _chk(x, col)
    B, H, W, C = x.shape
    lib().im2col(_p(x), _p(col), dtype_code(x), B, H, W, C, kh, kw, stride, stride, pt, pl, oh, ow, _s())
    return col


def col2im(gcol, gin, kh, kw, stride, pt, pl, oh, ow, accumulate=False):
    _chk(gcol, gin)
    B, H, W, C = gin.shape
    lib().col2im(_p(gcol), _p(gin), int(accumulate), dtype_code(gin), B, H, W, C, kh, kw, stride, stride, pt, pl, oh, ow, _s())
    return gin


def maxpool3s2_valid_fwd(x, out, argmax=None):
    _chk(x, out, argmax)
    B, H, W, C = x.shape
    lib().maxpool3s2_valid_fwd(_p(x), _p(out), _p(argmax), dtype_code(x), B, H, W, C, _s())
    return out


def maxpool3s2_valid_bwd(gout, argmax, gin):
    _chk(gout, argmax, gin)
    B, H, W, C = gin.shape
    lib().maxpool3s2_valid_bwd(_p(gout), _p(argmax), _p(gin), dtype_code(gin), B, H, W, C, _s())
    return gin


def avgpool3s1(x, out, bwd=False, accumulate=False):
    _chk(x, out)
    B, H, W, C = x.shape
    lib().avgpool3s1(_p(x), _p(out), int(bwd), int(accumulate), dtype_code(x), B, H, W, C, _s())
    return out


def copy2d(src, src_col, ld_src, dst, dst_col, ld_dst, rows, cols, accumulate=False):
    """dst[r, dst_col:dst_col+cols] (+)= src[r, src_col:src_col+cols] on row-major buffers with pitches ld_*."""
    es = src.element_size()
    lib().copy2d(src.data_ptr() + src_col * es, ld_src, dst.data_ptr() + dst_col * es, ld_dst, int(accumulate),
                 dtype_code(src), rows, cols, _s())


def residual_fwd(x, u, bias, scale, relu, out):
    _chk(x, u, out)
    C = x.shape[-1]
    lib().residual_fwd(_p(x), _p(u), _p(bias), float(scale), int(relu), _p(out), dtype_code(x), x.numel() // C, C, _s())
    return out


def residual_bwd(gy, y, scale, relu, gx, accumulate_gx, gu):
    _chk(gy, y, gx, gu)
    C = y.shape[-1]
    lib().residual_bwd(_p(gy), _p(y), float(scale), int(relu), _p(gx), int(accumulate_gx), _p(gu), dtype_code(y),
                       y.numel() // C, C, _s())


def colsum_rows(g, out, acc=None):
    """out[C] += column sums of g [rows, C]. acc: accumulator scratch (stats_alloc, >= C entries, all zero): the sums
    then go through the order-independent accumulators (bit-identical whatever the order of the rows) and are added
    into out afterwards."""
    _chk(g, out, acc)
    C = g.shape[-1]
    lib().colsum_rows(_p(g), _p(out), _p(acc), dtype_code(g), g.numel() // C, C, _s())
    if acc is not None:
        lib().acc_to_f32(_p(acc), _p(out), C, 1, 1, _s())
    return out
