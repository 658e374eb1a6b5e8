"""Xception-SPNet execution engine: owns the device buffers and sequences the sm_100a kernels
of libspnet_b200.so for inference, and for the training step
    forward (train-mode BN, dropout) -> YOLO-ellipse loss (+L2) -> backward -> Keras Adam.

This replaces what the reference gets from keras Model.predict / Model.fit's train_function
on the graph built by create_model_functional (spnet/models.py:302-424, compiled at :494-502).
All arithmetic happens in the CUDA kernels; torch only provides memory, streams and graphs.

Data layout in HBM: activations NHWC, bf16 (or fp32 in fp32 mode); every convolution output is
stored RAW (pre-BatchNorm) together with fp64 per-channel sum / sum-of-squares accumulated by
the producing kernel; BatchNorm (+ReLU) is applied by the consumer on load as y = a*z + b.
Parameters: one flat fp32 master buffer (L2-regularised kernels first, Dense head at offset 0
so its gradient is the first all-reduce bucket), flat fp32 grad / Adam m / Adam v buffers with
the same layout and a flat bf16 working copy refreshed by the Adam kernel.
"""
import math
from collections import OrderedDict

import numpy as np
import os

import torch

from . import arch, irv2, ops
from ._lib import lib


class _BN:
    __slots__ = ("name", "C", "gamma", "beta", "ggamma", "gbeta", "mm", "mv", "a", "b", "mean", "rstd", "c1", "c2",
                 "stats")


class _Sep:
    __slots__ = ("name", "cin", "cout", "dwk", "gdwk", "pw", "pwl", "gpw", "bn", "t", "z", "H", "W")


class SPNetEngineBase:
    """Stem, Dense head, loss, optimiser and step plumbing shared by the backbones. A backbone
    subclass provides: _arch() -> (shapes, param spec), _build_backbone(), _alloc_backbone()
    (must set self.feat_dims = (fh, fw, C)), _backbone_fwd(training) (stem output self.d ->
    self.feat) and _backbone_bwd(ga) (self.gfeat -> gradient w.r.t. self.d in ga)."""

    def __init__(self, H, W, batch, n_out=576, dtype="bf16", device="cuda:0", weights=None, seed=1,
                 loss_type="same", dropout_rate=arch.DROPOUT_RATE, use_l2=True, unbiased_moving_var=True,
                 training=True, deterministic=False):
        """deterministic: also make the WEIGHT GRADIENTS bit-identical from run to run (split-K partial products go to
        slabs that are added in a fixed order instead of fp32 reduce-adds). The forward pass, the BatchNorm
        statistics, the loss and the predictions are order-independent in either mode."""
        assert dtype in ("bf16", "fp32")
        self.deterministic = bool(deterministic)
        self._slabs = None
        self._affine_fixed = False
        self._gacc = None  # accumulator scratch of the deterministic weight-gradient paths (allocated with the activations)
        self.device = torch.device(device)
        torch.cuda.set_device(self.device)
        lib().check_device()
        self.H, self.W, self.B, self.n_out = H, W, batch, n_out
        self.lowp = dtype == "bf16"
        self.adt = torch.bfloat16 if self.lowp else torch.float32
        self.loss_type = loss_type
        self.dropout_rate = float(dropout_rate)
        self.use_l2 = use_l2
        self.unbiased = unbiased_moving_var
        self.can_train = training
        self.shapes, self.spec = self._arch()
        self._alloc_params(weights if weights is not None else arch.glorot_init(self.spec, seed))
        self._build_layers()
        self._alloc_activations()
        self.step_count = 0
        self.graph = None
        self.lr_t_dev = torch.zeros(1, device=self.device, dtype=torch.float32)
        self.seed_dev = torch.zeros(1, device=self.device, dtype=torch.int64)
        self.base_seed = int(seed)
        self.grad_hook = None  # called between backward and the optimiser (data-parallel all-reduce)
        # which BatchNorms normalise with their moving statistics inside a training step: "none" (Keras 2.1.3: even a
        # frozen BN uses the batch statistics in the training phase), "frozen" (modern tf.keras semantics), "all"
        self.bn_use_moving = "none"
        self.frozen8 = None    # uint8 per 8 parameters: non-zero = frozen (set_frozen)
        self.frozen_layers = frozenset()

    # ------------------------------------------------------------------ parameters
    def _alloc_params(self, weights):
        dev = self.device
        train = [(k, s, r) for k, s, t, r in self.spec if t]
        # Dense head first, then the other L2-regularised kernels, then everything else
        order = ([e for e in train if e[0] == "FinalOutput/kernel"] + [e for e in train if e[2] and e[0] != "FinalOutput/kernel"]
                 + [e for e in train if not e[2]])
        self.offsets = OrderedDict()
        off = 0
        for k, s, r in order:
            n = int(np.prod(s))
            self.offsets[k] = (off, n, s)
            off += (n + 7) // 8 * 8  # keep every tensor 32-byte aligned (16 B in bf16) for TMA / vector loads
        self.n_params_padded = off
        self.n_l2 = sum((int(np.prod(s)) + 7) // 8 * 8 for k, s, r in order if r)
        self.params = torch.zeros(off, device=dev, dtype=torch.float32)
        self.w = OrderedDict((k, self.params[o:o + n].view(*s)) for k, (o, n, s) in self.offsets.items())
        if self.can_train:
            self.grads = torch.zeros(off, device=dev, dtype=torch.float32)
            self.adam_m = torch.zeros(off, device=dev, dtype=torch.float32)
            self.adam_v = torch.zeros(off, device=dev, dtype=torch.float32)
            self.g = OrderedDict((k, self.grads[o:o + n].view(*s)) for k, (o, n, s) in self.offsets.items())
        if self.lowp:
            self.params_lp = torch.zeros(off, device=dev, dtype=torch.bfloat16)
            self.wl = OrderedDict((k, self.params_lp[o:o + n].view(*s)) for k, (o, n, s) in self.offsets.items())
        else:
            self.params_lp, self.wl = None, self.w
        nt = [(k, s) for k, s, t, _ in self.spec if not t]
        self.nt_offsets = OrderedDict()
        off = 0
        for k, s in nt:
            self.nt_offsets[k] = (off, int(np.prod(s)), s)
            off += int(np.prod(s))
        self.nontrainable = torch.zeros(off, device=dev, dtype=torch.float32)
        self.nt = OrderedDict((k, self.nontrainable[o:o + n].view(*s)) for k, (o, n, s) in self.nt_offsets.items())
        self.set_weights(weights)

    def set_weights(self, weights):
        """weights: {'<layer>/<weight>': array in Keras layout}."""
        for k, _, t, _ in self.spec:
            src = torch.as_tensor(np.asarray(weights[k], dtype=np.float32))
            dst = self.w[k] if t else self.nt[k]
            assert tuple(src.shape) == tuple(dst.shape), (k, tuple(src.shape), tuple(dst.shape))
            dst.copy_(src)
        self.refresh_lowp()

    def get_weights(self):
        torch.cuda.synchronize(self.device)
        out = OrderedDict()
        for k, _, t, _ in self.spec:
            out[k] = (self.w[k] if t else self.nt[k]).detach().cpu().numpy().copy()
        return out

    def refresh_lowp(self):
        self._affine_fixed = False  # the weights changed: inference-mode BatchNorm affines must be rebuilt
        if self.lowp:
            ops.cast_f32_to_bf16(self.params, self.params_lp)

    # ------------------------------------------------------------------ layers
    def _f32(self, n):
        return torch.zeros(n, device=self.device, dtype=torch.float32)

    def _mk_bn(self, name, C, scale=True):
        bn = _BN()
        bn.name, bn.C = name, C
        bn.gamma, bn.beta = (self.w[name + "/gamma"] if scale else None), self.w[name + "/beta"]
        if self.can_train:
            bn.ggamma, bn.gbeta = (self.g[name + "/gamma"] if scale else None), self.g[name + "/beta"]
        else:
            bn.ggamma = bn.gbeta = None
        bn.mm, bn.mv = self.nt[name + "/moving_mean"], self.nt[name + "/moving_variance"]
        bn.a, bn.b, bn.mean, bn.rstd, bn.c1, bn.c2 = (self._f32(C) for _ in range(6))
        bn.stats = ops.stats_alloc(2 * C, self.device)  # order-independent accumulators (sum | sum of squares)
        self.bns.append(bn)
        return bn

    def _mk_sep(self, name, cin, cout, hw):
        s = _Sep()
        s.name, s.cin, s.cout = name, cin, cout
        s.H, s.W = hw
        s.dwk = self.w[name + "/depthwise_kernel"].view(3, 3, cin)
        s.pw = self.w[name + "/pointwise_kernel"].view(cin, cout)
        s.pwl = self.wl[name + "/pointwise_kernel"].view(cin, cout)
        if self.can_train:
            s.gdwk = self.g[name + "/depthwise_kernel"].view(3, 3, cin)
            s.gpw = self.g[name + "/pointwise_kernel"].view(cin, cout)
        s.bn = self._mk_bn(name + "_bn", cout)
        return s

    def _build_layers(self):
        self.bns = []
        self.stem_bn = [self._mk_bn("batch_normalization_%d" % i, 3) for i in (1, 2, 3)]
        self._build_backbone()
        self.k4 = self._f32(48).view(4, 4, 1, 3)
        self.gk4 = self._f32(48).view(4, 4, 1, 3)
        self.l2_out = self._f32(1)
        self.l2_acc = ops.stats_alloc(1, self.device)

    def _act(self, *shape, dtype=None):
        t = torch.empty(*shape, device=self.device, dtype=dtype or self.adt)
        if os.environ.get("SPNET_B200_POISON") and t.is_floating_point():
            t.fill_(float("nan"))  # debug: a kernel that reads a buffer before anything wrote it now fails loudly
        return t

    def _alloc_activations(self):
        B, sh, A = self.B, self.shapes, self._act
        H, W = self.H, self.W
        self.x0 = torch.zeros(B, H, W, 1, device=self.device, dtype=torch.float32)
        self.y_true = torch.zeros(B, self.n_out, device=self.device, dtype=torch.float32)
        h, w = sh["stem"]
        self.p1, self.c2, self.c3, self.d = (A(B, h, w, 3) for _ in range(4))
        self.s0 = A(B, h, w, 1)
        self._alloc_backbone()
        fh, fw, fc = self.feat_dims
        self.feat = A(B, fh * fw * fc)
        self.y_pred = torch.zeros(B, self.n_out, device=self.device, dtype=torch.float32)
        self.loss6 = self._f32(6)
        if self.can_train:
            self.gy = torch.zeros(B, self.n_out, device=self.device, dtype=torch.float32)
            self.gyl = A(B, self.n_out) if self.lowp else self.gy
            self.gfeat = A(B, fh * fw * fc)
            sp = B * sh["stem"][0] * sh["stem"][1] * 3
            self.gstem = [A(sp) for _ in range(2)]
        if self.deterministic and self.can_train:
            self._gacc = ops.stats_alloc(9 * 2048, self.device)
        self.n_sms = torch.cuda.get_device_properties(self.device).multi_processor_count
        # Dense head forward = split-K over the features: ONE wave of the persistent GEMM (bf16: 128 x 256 tiles when
        # n_out >= 512, else 128 x 128 / 128 x 64) - a second, nearly empty wave doubled its time
        if self.lowp:
            tile_n = 256 if self.n_out >= 512 else (64 if self.n_out <= 64 else 128)
            tiles = -(-self.n_out // tile_n) * -(-B // 128)
            self.dense_splits = max(1, min(64, self.n_sms // max(1, tiles)))
        else:  # the fp32 kernel is not persistent: a few CTAs per SM hide its latency
            self.dense_splits = max(1, min(64, (2 * self.n_sms) // max(1, -(-self.n_out // 128))))
        self.head_slabs = torch.zeros(self.dense_splits, B, self.n_out, device=self.device, dtype=torch.float32)

    # ------------------------------------------------------------------ helpers
    def _view(self, buf, *shape):
        n = int(np.prod(shape))
        return buf[:n].view(*shape)

    def _uses_moving(self, bn):
        """Whether bn normalises with its moving statistics inside a training step (see bn_use_moving)."""
        return self.bn_use_moving == "all" or (self.bn_use_moving == "frozen" and bn.name in self.frozen_layers)

    def _bn_ready(self, bn, count, training):
        if training:
            # a frozen BatchNormalization (layer.trainable = False under Keras 2.1.3) still normalises with the batch
            # statistics in the training phase; what stops is the update of its moving averages (Layer.updates is
            # empty for a non-trainable layer) and of gamma / beta (Adam mask)
            frozen = bn.name in self.frozen_layers
            moving = self._uses_moving(bn)
            ops.bn_finalize(bn.stats, count, bn.gamma, bn.beta, bn.a, bn.b, bn.mean, bn.rstd, None if (frozen or moving) else bn.mm,
                            None if (frozen or moving) else bn.mv, eps=arch.BN_EPS, momentum=arch.BN_MOMENTUM, unbiased=self.unbiased)
            if moving:
                # this BatchNorm normalises with its MOVING statistics inside the training step (modern-Keras frozen-BN
                # semantics, and the N-GPU == 1-GPU gradient test where the batch must not couple the samples): the
                # affine and the statistics saved for backward come from the moving averages; backward then runs with
                # count = 0, which drops the batch-statistics terms (c1 = c2 = 0) and leaves dz = a * g
                ops.bn_inference_affine(bn.gamma, bn.beta, bn.mm, bn.mv, bn.a, bn.b, eps=arch.BN_EPS, save_mean=bn.mean,
                                        save_rstd=bn.rstd)
        elif not self._affine_fixed:
            ops.bn_inference_affine(bn.gamma, bn.beta, bn.mm, bn.mv, bn.a, bn.b, eps=arch.BN_EPS)

    def _pw_fwd(self, A, Wl, D, M, K, N, bn, training):
        ops.gemm(A, False, Wl, True, D, M, N, K, out_mode=ops.OUT_T, colstats=bn.stats if training else None)
        self._bn_ready(bn, M, training)

    def _wgrad_splits(self, rows_out, cols_out, K):
        tile = 128 if self.lowp else 64
        tiles = -(-rows_out // tile) * -(-cols_out // tile)
        kb = max(1, K // (64 if self.lowp else 16))
        return int(max(1, min(kb // 4 if kb >= 8 else 1, -(-(2 * self.n_sms) // tiles))))

    def _slab_buf(self, nslabs, rows, cols):
        n = nslabs * rows * cols
        if self._slabs is None or self._slabs.numel() < n:
            assert not torch.cuda.is_current_stream_capturing(), "slab scratch must be sized by an eager warm-up step"
            self._slabs = torch.zeros(n, device=self.device, dtype=torch.float32)
        return self._slabs

    def _pw_bwd(self, A, Wl, gW, gz, gA, M, K, N):
        """gz [M,N] -> gW [K,N] += A^T gz ;  gA [M,K] = gz W^T. gW None: the weight gradient is computed elsewhere
        (the batched launch over the middle flow)."""
        if gW is not None:
            if self.deterministic:
                # fixed-order split-K: partial products to slabs, added in split order (bit-identical run to run)
                sp = self._wgrad_splits(K, N, M)
                slabs = self._slab_buf(sp, K, N)
                if sp > 1:
                    slabs[:sp * K * N].zero_()  # a slab the GEMM does not need must read as zero
                ops.gemm(A, True, gz, True, slabs, K, N, M, out_mode=ops.OUT_SLAB, splits=sp, lda=K, ldb=N)
                ops.slab_reduce(slabs, sp, K, N, gW, accumulate=True)
            else:
                sp = 0 if self.lowp else self._wgrad_splits(K, N, M)  # 0 = let the tcgen05 GEMM pick (fills the SMs once)
                ops.gemm(A, True, gz, True, gW, K, N, M, out_mode=ops.OUT_ATOMIC, splits=sp, lda=K, ldb=N)
        if gA is not None:
            ops.gemm(gz, False, Wl, False, gA, M, K, N, out_mode=ops.OUT_T, ldb=N)

    def _pw_bwd_fusable(self, K, N):
        """The BatchNorm backward and both pointwise GEMMs of a K -> N layer run as one kernel (csrc/pw_bwd.cu)."""
        return self.lowp and N == 128 and K in (64, 128)

    def _bn_pw_bwd(self, g, z, bn, A, Wl, gW, gA, M, K, N, dz=None):
        """g = grad wrt the output of BatchNorm bn of z = A W, its sums already in bn.stats -> gA [M,K] = dz W^T and
        gW [K,N] += A^T dz (gW None: computed elsewhere from the stored dz). One kernel where _pw_bwd_fusable, dz never
        leaving the chip and g left as it is; otherwise dz is stored in dz, or over g when dz is None."""
        if gW is not None and self._pw_bwd_fusable(K, N):
            ops.bn_bwd_finalize(bn.stats, self._bwd_count(bn, M), bn.ggamma, bn.gbeta, bn.c1, bn.c2)
            slabs = self._slab_buf(ops.pw_bwd_bn_slabs(M, self.device), K, N) if self.deterministic else None
            ops.pw_bwd_bn(g, z, A, Wl, bn.a, bn.mean, bn.rstd, bn.c1, bn.c2, gA, gW, M, K, N, slabs=slabs)
        else:
            dz = self._bn_bwd(g, z, bn, M, out=dz)
            self._pw_bwd(A, Wl, gW, dz.view(M, N), gA, M, K, N)

    def _sep_fwd(self, s, x, in_bn, relu, training):
        B = self.B
        ops.dwconv3x3_fwd(x, s.dwk, in_bn.a if in_bn else None, in_bn.b if in_bn else None, relu, out=s.t)
        M = B * s.H * s.W
        self._pw_fwd(s.t, s.pwl, s.z, M, s.cin, s.cout, s.bn, training)

    def _bwd_count(self, bn, rows):
        # count 0: bn_bwd_finalize drops the batch-statistics terms (c1 = c2 = 0)
        return 0 if self._uses_moving(bn) else rows

    def _bn_bwd_sums(self, g, z, bn, act=None):
        """Accumulates bn's backward sums over g into bn.stats: the step for a gradient whose producer does not. g = grad
        wrt the BN output; with act (1 = ReLU, 3 = ReLU6) g = grad wrt act(BN output), masked in place by act' first."""
        if act is None:
            ops.bn_bwd_reduce(g, z, bn.mean, bn.rstd, bn.stats)
        else:
            ops.bn_bwd_reduce(g, z, bn.mean, bn.rstd, bn.stats, relu_a=bn.a, relu_b=bn.b, act=act)

    def _bn_bwd(self, g, z, bn, rows, out=None):
        """g = grad wrt the BN output, its backward sums already in bn.stats (accumulated by the producer of g or by
        _bn_bwd_sums) -> grad wrt z, stored in out (default: over g)."""
        ops.bn_bwd_finalize(bn.stats, self._bwd_count(bn, rows), bn.ggamma, bn.gbeta, bn.c1, bn.c2)
        return ops.bn_bwd_dz(g, z, bn.a, bn.mean, bn.rstd, bn.c1, bn.c2, out=out if out is not None else g)

    # ------------------------------------------------------------------ forward
    def forward(self, training=False):
        """Runs the network on self.x0 (already on the device). Result in self.y_pred."""
        B, sh = self.B, self.shapes
        w = self.w
        bn1, bn2, bn3 = self.stem_bn
        H2, W2 = sh["stem"]
        npx = B * H2 * W2
        st = (lambda bn: bn.stats) if training else (lambda bn: None)
        # ---- stem (spnet/models.py:321-338)
        ops.stem_k3_to_k4(w["conv2d_1/kernel"], self.k4)
        ops.conv_small_fwd(0, self.x0, self.k4, self.p1, skip=self.s0, stats=st(bn1))
        self._bn_ready(bn1, npx, training)
        ops.conv_small_fwd(1, self.p1, w["conv2d_2/kernel"], self.c2, in_a=bn1.a, in_b=bn1.b, act=2, stats=st(bn2))
        self._bn_ready(bn2, npx, training)
        ops.conv_small_fwd(1, self.c2, w["conv2d_3/kernel"], self.c3, in_a=bn2.a, in_b=bn2.b, act=2, stats=st(bn3))
        self._bn_ready(bn3, npx, training)
        drop = training and self.dropout_rate > 0
        ops.stem_out_fwd(self.c3, bn3.a, bn3.b, self.s0, self.d, rate=self.dropout_rate if drop else 0.0,
                         seed=self.seed_dev if drop else None)
        self._backbone_fwd(training)
        F = self.feat.shape[1]
        # split-K over the 98,304 features with a FIXED summation order: every split stores its partial product in its
        # own slab, one small kernel adds bias + slabs in order -> two predict() calls give bit-identical outputs
        ops.gemm(self.feat, False, self.wl["FinalOutput/kernel"], True, self.head_slabs, B, self.n_out, F,
                 out_mode=ops.OUT_SLAB, splits=self.dense_splits)
        ops.slab_reduce(self.head_slabs, self.dense_splits, B, self.n_out, self.y_pred, bias=w["FinalOutput/bias"])
        return self.y_pred

    def _entry_fwd(self, e, x, training):
        B = self.B
        oh, ow = e["ohw"]
        ops.gather_s2(x, out=e["xs"])
        self._pw_fwd(e["xs"].view(-1, e["cin"]), self.wl[e["res"] + "/kernel"].view(e["cin"], e["c"]),
                     e["zr"].view(-1, e["c"]), B * oh * ow, e["cin"], e["c"], e["res_bn"], training)
        s1, s2 = e["sep1"], e["sep2"]
        self._sep_fwd(s1, x, None, e["relu_in"], training)
        self._sep_fwd(s2, s1.z, s1.bn, True, training)
        ops.maxpool3s2_add_fwd(s2.z, s2.bn.a, s2.bn.b, e["zr"], e["res_bn"].a, e["res_bn"].b, out=e["out"],
                               argmax=e["argmax"] if training else None)
        return e["out"]

    # ------------------------------------------------------------------ loss
    def loss(self, with_grad):
        ops.yolo_ellipse_loss(self.y_true, self.y_pred, hybrid=(self.loss_type != "same"), out6=self.loss6,
                              grad=self.gy if with_grad else None)
        if self.use_l2:
            ops.sumsq(self.params, self.n_l2, arch.L2_COEF, self.l2_acc)
            ops.acc_to_f32(self.l2_acc, self.l2_out)

    # ------------------------------------------------------------------ backward
    def _sep_bwd(self, s, g, x, in_bn, relu, g_t, g_in, add_src=None, add_strided=None, wgrad=True, out_bn=None,
                 dz=None):
        """g: grad wrt the output of s.bn [M,cout], its backward sums already in s.bn.stats. The BatchNorm and pointwise
        backward run as _bn_pw_bwd (grad wrt s.t in g_t; dz as there; wgrad=False: the pointwise weight gradient is
        computed elsewhere from dz). Produces the gradient wrt the sepconv's input tensor x (before its on-load BN/ReLU
        transform) in g_in; for a BN'd input in_bn this is the grad wrt in_bn's OUTPUT (masked by relu'), with in_bn's
        backward sums accumulated.
        out_bn = (z, bn, relu_mask): x = [relu](bn(z)) [+ ...], the BN that produced the UNtransformed input x. The
        depthwise backward then accumulates that BN's backward sums on the final g_in (masked by the ReLU when
        relu_mask), so the caller can go straight to _bn_bwd on g_in's residual path."""
        B = self.B
        M = B * s.H * s.W
        self._bn_pw_bwd(g, s.z, s.bn, s.t, s.pwl, s.gpw if wgrad else None, g_t, M, s.cin, s.cout, dz=dz)
        gt4 = g_t.view(B, s.H, s.W, s.cin)
        zo, zbn, zmask = out_bn if out_bn else (None, None, False)
        ops.dwconv3x3_bwd_fused(gt4, x, s.dwk, s.gdwk, in_a=in_bn.a if in_bn else None, in_b=in_bn.b if in_bn else None,
                                relu=relu, bn_mean=in_bn.mean if in_bn else None, bn_rstd=in_bn.rstd if in_bn else None,
                                stats=in_bn.stats if in_bn else None, add_src=add_src, add_strided=add_strided,
                                out=g_in.view(B, s.H, s.W, s.cin), acc=self._gacc,
                                zo=zo, zo_mean=zbn.mean if zbn else None, zo_rstd=zbn.rstd if zbn else None,
                                zo_stats=zbn.stats if zbn else None, mask_a=zbn.a if zmask else None,
                                mask_b=zbn.b if zmask else None)

    def _entry_bwd(self, e, x, g_out, bufs, x_bn):
        """g_out: grad wrt block output [B,oh,ow,c], the backward sums of its residual BN already accumulated (by the
        producer of g_out); it is left as it is. Returns grad wrt block input x, with the sums of x's BN
        x_bn = (z, bn, relu_mask) accumulated."""
        B = self.B
        (H, W), (oh, ow) = e["hw"], e["ohw"]
        cin, c = e["cin"], e["c"]
        G1, G2, G3, S, R = bufs
        Mo = B * oh * ow
        M = B * H * W
        s1, s2 = e["sep1"], e["sep2"]
        # residual branch (g_out is read again by the max-pool backward: dz goes to G1, not over g_out)
        g_xs = self._view(S, Mo, cin)
        self._bn_pw_bwd(g_out, e["zr"], e["res_bn"], e["xs"].view(Mo, cin), self.wl[e["res"] + "/kernel"].view(cin, c),
                        self.g[e["res"] + "/kernel"].view(cin, c), g_xs, Mo, cin, c, dz=self._view(G1, Mo, c))
        # main branch
        g_y2 = ops.maxpool3s2_bwd(g_out, e["argmax"], H, W, out=self._view(G1, B, H, W, c), z=s2.z, mean=s2.bn.mean,
                                  rstd=s2.bn.rstd, stats=s2.bn.stats)
        g_y1 = self._view(G3, B, H, W, s2.cin)
        self._sep_bwd(s2, g_y2.view(M, c), s1.z, s1.bn, True, self._view(G2, M, s2.cin), g_y1)
        g_x = self._view(R, B, H, W, cin)
        self._sep_bwd(s1, g_y1.view(M, s1.cout), x, None, e["relu_in"], self._view(G1, M, cin), g_x,
                      add_strided=g_xs.view(B, oh, ow, cin), out_bn=x_bn)
        return g_x

    def backward_head(self):
        """Dense head: consumes self.gy (dL/dy_pred) -> FinalOutput gradients + dL/dfeatures.
        Its weight gradient is 73 % of all gradient bytes and is complete first: under data
        parallelism its all-reduce is launched right after this and overlaps backward_body()."""
        B, g = self.B, self.g
        F = self.feat.shape[1]
        if self.lowp:
            ops.cast_f32_to_bf16(self.gy, self.gyl)
        ops.colsum(self.gy, g["FinalOutput/bias"])
        # under bf16 data-parallel communication the 226 MB fp32 weight gradient of the head is written as bf16
        # straight into the all-reduce buffer (multi_gpu.GradAllReduce sets head_grad_lp); Adam reads it from there
        gk = getattr(self, "head_grad_lp", None)
        ops.gemm(self.feat, True, self.gyl, True, gk if gk is not None else g["FinalOutput/kernel"], F, self.n_out, B,
                 out_mode=ops.OUT_T if gk is not None else ops.OUT_F32, lda=F, ldb=self.n_out)
        ops.gemm(self.gyl, False, self.wl["FinalOutput/kernel"], False, self.gfeat, B, F, self.n_out,
                 out_mode=ops.OUT_T, ldb=self.n_out)

    def backward(self):
        """Consumes self.gy; accumulates into self.grads (zeroed by the caller)."""
        self.backward_head()
        self.backward_body()

    # Backward of the backbone in two parts, so that under data parallelism the gradients that are
    # final after part A (everything from `tail_param_key` to the end of the flat buffer) can be
    # all-reduced while part B and the stem still run. Backbones without such a split do all of it in B.
    tail_param_key = None

    def _backbone_bwd_a(self):
        pass

    def _backbone_bwd_b(self, ga):
        self._backbone_bwd(ga)

    def backward_body(self):
        self.backward_body_a()
        self.backward_body_b()

    def backward_body_a(self):
        self._backbone_bwd_a()

    def backward_body_b(self):
        B, sh, w, g = self.B, self.shapes, self.w, self.g
        H2, W2 = sh["stem"]
        npx = B * H2 * W2
        ga, gb = (self._view(t, B, H2, W2, 3) for t in self.gstem)
        self._backbone_bwd_b(ga)
        # ---- stem
        bn1, bn2, bn3 = self.stem_bn
        drop = self.dropout_rate > 0
        ops.stem_out_bwd(ga, gb, rate=self.dropout_rate if drop else 0.0, seed=self.seed_dev if drop else None)
        self._bn3_bwd(gb, self.c3, bn3, npx)                      # gb = grad wrt c3
        ops.conv_small_wgrad(1, self.c2, gb, g["conv2d_3/kernel"], in_a=bn2.a, in_b=bn2.b, act=2, acc=self._gacc)
        ops.conv_small_dgrad(1, gb, w["conv2d_3/kernel"], ga, mask_z=self.c2, mask_a=bn2.a, mask_b=bn2.b, act=2)
        self._bn3_bwd(ga, self.c2, bn2, npx)                      # ga = grad wrt c2
        ops.conv_small_wgrad(1, self.p1, ga, g["conv2d_2/kernel"], in_a=bn1.a, in_b=bn1.b, act=2, acc=self._gacc)
        ops.conv_small_dgrad(1, ga, w["conv2d_2/kernel"], gb, mask_z=self.p1, mask_a=bn1.a, mask_b=bn1.b, act=2)
        self._bn3_bwd(gb, self.p1, bn1, npx)                      # gb = grad wrt p1
        self.gk4.zero_()
        ops.conv_small_wgrad(0, self.x0, gb, self.gk4, acc=self._gacc)
        ops.stem_k4grad_to_k3grad(self.gk4, g["conv2d_1/kernel"])

    def _bn3_bwd(self, gbuf, z, bn, npx):
        ops.bn3_bwd_reduce(gbuf, z, bn.mean, bn.rstd, bn.stats)
        ops.bn_bwd_finalize(bn.stats, self._bwd_count(bn, npx), bn.ggamma, bn.gbeta, bn.c1, bn.c2)
        ops.bn3_bwd_dz(gbuf, z, bn.a, bn.mean, bn.rstd, bn.c1, bn.c2, gbuf)

    # ------------------------------------------------------------------ optimiser / step
    def set_frozen(self, layer_names):
        """Layers whose weights must not train (Keras layer.trainable = False; spnet/models.py:361-372): Adam skips
        every tensor of those layers (no update, no L2 pull) and their BatchNormalization moving averages stop."""
        self.frozen_layers = frozenset(layer_names or ())
        if not self.frozen_layers:
            self.frozen8 = None
            return
        mask = np.zeros(self.n_params_padded // 8, np.uint8)
        for k, (o, n, _) in self.offsets.items():
            if k.split("/")[0] in self.frozen_layers:
                mask[o // 8:(o + n + 7) // 8] = 1
        self.frozen8 = torch.from_numpy(mask).to(self.device)
        self.graph = None  # the mask pointer is baked into a captured step

    def optimizer_step(self, grad_scale=1.0, lo=0, hi=None, g_bf16=None):
        """Keras Adam (+ L2 pull) on the flat parameter range [lo, hi) (multiples of 8; default: everything)."""
        hi = self.n_params_padded if hi is None else hi
        n_l2 = min(max((self.n_l2 if self.use_l2 else 0) - lo, 0), hi - lo)
        ops.adam_keras_step(self.params[lo:hi], self.grads[lo:hi], self.adam_m[lo:hi], self.adam_v[lo:hi], self.lr_t_dev,
                            n_l2=n_l2, l2=arch.L2_COEF, grad_scale=grad_scale,
                            p_bf16=self.params_lp[lo:hi] if self.params_lp is not None else None,
                            frozen8=self.frozen8[lo // 8:] if self.frozen8 is not None else None,
                            g_bf16=g_bf16[lo:hi] if g_bf16 is not None else None)

    def _step_part1(self):
        # the Dense-head weight gradient (73 % of the buffer, at offset 0) is written in overwrite mode
        o, n, _ = self.offsets["FinalOutput/kernel"]
        assert o == 0
        self.grads[(n + 7) // 8 * 8:].zero_()
        self.forward(training=True)
        self.loss(with_grad=True)
        self.backward_head()

    def _step_body(self):
        self._step_part1()
        self._bucket_ready("head")
        self.backward_body_a()
        self._bucket_ready("tail")
        self.backward_body_b()
        if self.grad_hook is None:
            self.optimizer_step()

    def _bucket_ready(self, which):
        fn = getattr(self.grad_hook, "bucket_ready", None)
        if fn is not None:
            fn(self, which)

    def set_lr(self, lr, beta1=0.9, beta2=0.999):
        """Host side of Keras Adam: t += 1, lr_t = lr*sqrt(1-b2^t)/(1-b1^t) -> device scalar."""
        self.step_count += 1
        t = self.step_count
        # by-value kernel arguments (fill), not asynchronous copies from a reused pinned scalar: the host may be several
        # steps ahead of the GPU, and a pinned buffer is read when the copy EXECUTES
        self.lr_t_dev.fill_(lr * math.sqrt(1.0 - beta2 ** t) / (1.0 - beta1 ** t))
        self.seed_dev.fill_((self.base_seed * 1000003 + t) & 0x7FFFFFFFFFFFFFFF)

    def capture(self):
        """Capture fwd+loss+bwd(+Adam) into one CUDA graph (call after one eager warm-up step)."""
        if getattr(self.grad_hook, "bucket_ready", None) is None:
            gph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gph):
                self._step_body()
            self.graph = (gph,)
        else:
            # three graphs so that the Dense-head and the tail-bucket all-reduces can be launched between them
            g1, g2, g3 = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            with torch.cuda.graph(g1):
                self._step_part1()
            with torch.cuda.graph(g2, pool=g1.pool()):
                self.backward_body_a()
            with torch.cuda.graph(g3, pool=g1.pool()):
                self.backward_body_b()
            self.graph = (g1, g2, g3)

    def train_step(self, lr):
        """One optimiser step on the batch currently in self.x0 / self.y_true.
        Returns the device tensor [total, center, size, angle, noobj, class] (data loss) —
        the L2 term is in self.l2_out."""
        self.set_lr(lr)
        fn = getattr(self.grad_hook, "step_begin", None)
        if fn is not None:
            fn(self)
        if self.graph is not None:
            self.graph[0].replay()
            if len(self.graph) > 1:
                self._bucket_ready("head")
                self.graph[1].replay()
                self._bucket_ready("tail")
                self.graph[2].replay()
        else:
            self._step_body()
        if self.grad_hook is not None:
            self.skip_default_optimizer = False
            self.grad_hook(self)          # e.g. multi_gpu.GradAllReduce (runs its own optimiser step)
            if not self.skip_default_optimizer:
                self.optimizer_step()
        return self.loss6

    # ---- asynchronous input path: the NEXT batch travels host -> device on a copy stream into a staging
    #      buffer while the current step computes; take_prefetched() moves it into the step's (graph-captured)
    #      input buffers with a device-to-device copy.
    def _ensure_stage(self):
        if getattr(self, "_copy_stream", None) is None:
            self._xs = torch.empty_like(self.x0)
            self._xs_u8 = None
            self._ys = torch.empty_like(self.y_true)
            self._copy_stream = torch.cuda.Stream(device=self.device)
            self._stage_ready = torch.cuda.Event()
            self._stage_free = torch.cuda.Event()
            self._stage_free.record()
            self._h2d_done = torch.cuda.Event()
            self._staged_u8 = False

    def prefetch_batch(self, x_host, y_host=None):
        """Start the H2D copy of a batch (pinned torch tensors) without blocking the compute stream.
        uint8 frames (raw pixel values 0..255) travel as bytes - a quarter of the PCIe traffic of fp32 - and are
        normalised on the device by take_prefetched(). Returns an event that fires when the host buffers may be reused."""
        self._ensure_stage()
        cs = self._copy_stream
        u8 = x_host.dtype == torch.uint8
        if u8 and (self._xs_u8 is None or self._xs_u8.shape[1:3] != x_host.shape[1:3]):
            self._xs_u8 = torch.empty((self.B,) + tuple(x_host.shape[1:3]), device=self.device, dtype=torch.uint8)
        with torch.cuda.stream(cs):
            cs.wait_event(self._stage_free)  # the previous staged batch has been taken
            if u8:
                self._xs_u8.copy_(x_host.view(self._xs_u8.shape), non_blocking=True)
            else:
                self._xs.copy_(x_host.view(self._xs.shape), non_blocking=True)
            if y_host is not None:
                self._ys.copy_(y_host.view(self._ys.shape), non_blocking=True)
            done = torch.cuda.Event()
            done.record(cs)
            self._stage_ready.record(cs)
        self._has_y = y_host is not None
        self._staged_u8 = u8
        return done

    def take_prefetched(self):
        """Make the staged batch the current one (compute stream waits for its H2D copy only)."""
        main = torch.cuda.current_stream()
        main.wait_event(self._stage_ready)
        if self._staged_u8:
            self.frames_to_x0(self._xs_u8)
        else:
            self.x0.copy_(self._xs)
        if self._has_y:
            self.y_true.copy_(self._ys)
        self._stage_free.record(main)

    def frames_to_x0(self, x_u8):
        """uint8 frames [m, h, w(, 1)] on the device -> self.x0[:m]: (v/255 - 0.5)*2 of spnet/utils.py:340-342, after a
        LANCZOS resize to the engine's (H, W) when (h, w) differs - the bytes of the host's PIL resize (:325-349)."""
        m = x_u8.shape[0]
        if m > self.B or x_u8.dim() < 3 or x_u8.numel() != m * x_u8.shape[1] * x_u8.shape[2]:
            raise ValueError("frames %s for an engine of batch %d: want [<= %d, h, w(, 1)] uint8" % (tuple(x_u8.shape), self.B, self.B))
        if tuple(x_u8.shape[1:3]) == (self.H, self.W):
            if x_u8.data_ptr() % 16:  # normalize_u8 reads 16-byte vectors; a slice of odd-sized frames may start anywhere
                x_u8 = x_u8.clone()
            ops.normalize_u8(x_u8, self.x0[:m])
        else:
            ops.resize_lanczos_u8(x_u8, self.H, self.W, out=self.x0[:m])

    def load_batch(self, x_host, y_host=None):
        """H2D copy of one batch (numpy or pinned torch tensors; uint8 frames are normalised - and resized when their size
        is not the engine's - on the device)."""
        if (torch.is_tensor(x_host) and x_host.dtype == torch.uint8) or (not torch.is_tensor(x_host) and np.asarray(x_host).dtype == np.uint8):
            xt = x_host if torch.is_tensor(x_host) else torch.from_numpy(np.ascontiguousarray(x_host))
            self.frames_to_x0(xt.to(self.device, non_blocking=True).contiguous())
        else:
            xt = x_host if torch.is_tensor(x_host) else torch.from_numpy(np.ascontiguousarray(x_host, dtype=np.float32))
            self.x0.copy_(xt.view(self.x0.shape), non_blocking=True)
        if y_host is not None:
            yt = y_host if torch.is_tensor(y_host) else torch.from_numpy(np.ascontiguousarray(y_host, dtype=np.float32))
            self.y_true.copy_(yt.view(self.y_true.shape), non_blocking=True)

    # ---- inference: the forward pass as one CUDA graph
    def capture_forward(self):
        """Capture forward(training=False) into a CUDA graph (call after one eager forward)."""
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self.forward(training=False)
        self.fwd_graph = g

    def prepare_inference(self):
        """Inference-only engines: build every BatchNorm's moving-statistics affine once per set of weights instead of
        once per forward pass (about a hundred tiny launches per batch)."""
        self._affine_fixed = False
        for bn in self.bns:
            self._bn_ready(bn, 0, False)
        self._affine_fixed = not self.can_train  # a training step overwrites bn.a / bn.b with batch-statistics affines

    def infer(self):
        """Inference-mode forward on the batch in self.x0 (graph replay once captured). Result in self.y_pred."""
        if not self._affine_fixed and not self.can_train:
            self.prepare_inference()
        g = getattr(self, "fwd_graph", None)
        if g is not None:
            g.replay()
        else:
            self.forward(training=False)
        return self.y_pred


class XceptionSPNetEngine(SPNetEngineBase):
    """keras.applications.Xception backbone (reference default, spnet/config.py:52)."""

    def _arch(self):
        return arch.shape_walk(self.H, self.W), arch.param_spec(self.H, self.W, self.n_out)

    def _build_backbone(self):
        sh = self.shapes
        self.b1_bn1 = self._mk_bn("block1_conv1_bn", 32)
        self.b1_bn2 = self._mk_bn("block1_conv2_bn", 64)
        self.entry = []
        for n, (blk, cin, c) in enumerate(arch.ENTRY_BLOCKS):
            hw = sh["in%d" % blk]
            e = dict(blk=blk, cin=cin, c=c, hw=hw, ohw=sh["out%d" % blk], res="conv2d_%d" % (4 + n),
                     res_bn=self._mk_bn("batch_normalization_%d" % (4 + n), c),
                     sep1=self._mk_sep("block%d_sepconv1" % blk, cin, c, hw),
                     sep2=self._mk_sep("block%d_sepconv2" % blk, c, c, hw), relu_in=(blk != 2))
            self.entry.append(e)
        self.middle = []
        for blk in arch.MIDDLE_BLOCKS:
            self.middle.append([self._mk_sep("block%d_sepconv%d" % (blk, j), 728, 728, sh["middle"]) for j in (1, 2, 3)])
        hw = sh["in13"]
        self.exit13 = dict(blk=13, cin=728, c=1024, hw=hw, ohw=sh["out13"], res="conv2d_7",
                           res_bn=self._mk_bn("batch_normalization_7", 1024),
                           sep1=self._mk_sep("block13_sepconv1", 728, 728, hw),
                           sep2=self._mk_sep("block13_sepconv2", 728, 1024, hw), relu_in=True)
        self.sep14 = [self._mk_sep("block14_sepconv1", 1024, 1536, sh["out13"]),
                      self._mk_sep("block14_sepconv2", 1536, 2048, sh["out13"])]

    def _alloc_backbone(self):
        B, sh, A = self.B, self.shapes, self._act
        h1, w1 = sh["b1c1"]
        self.z11 = A(B, h1, w1, 32)
        h2, w2 = sh["b1c2"]
        # block1_conv2 (3x3 'valid', 32 -> 64) reads the materialised activation a11 = relu(BN(z11)): bf16 runs it as
        # an implicit GEMM (csrc/gemm_tc.cu kw-fold entry points); fp32 and the deterministic mode as im2col + GEMM
        self.b1_fold = self.lowp and not self.deterministic
        self.a11 = A(B, h1, w1, 32)
        if not self.b1_fold:
            self.col = A(B * h2 * w2, 288)
        self.z12 = A(B, h2, w2, 64)
        self.x2 = A(B, h2, w2, 64)
        train = self.can_train
        maxel = B * h2 * w2 * 128
        for e in self.entry + [self.exit13]:
            (eh, ew), (oh, ow) = e["hw"], e["ohw"]
            e["xs"] = A(B, oh, ow, e["cin"])
            e["zr"] = A(B, oh, ow, e["c"])
            for s in (e["sep1"], e["sep2"]):
                s.t = A(B, eh, ew, s.cin)
                s.z = A(B, eh, ew, s.cout)
                maxel = max(maxel, B * eh * ew * max(s.cin, s.cout))
            e["out"] = A(B, oh, ow, e["c"])
            e["argmax"] = A(B, oh, ow, e["c"], dtype=torch.uint8) if train else None
        mh, mw = sh["middle"]
        # the depthwise outputs t (the A operand of every pointwise weight gradient) of the 24 identical middle-flow
        # layers are ONE contiguous [24, Mpad, 728] tensor, and so are the gradients dz reaching their pointwise
        # convolutions: the 24 weight gradients dW_i = t_i^T dz_i are then a single GEMM launch whose K range is cut
        # into 24 slabs (ops.gemm out_mode OUT_SLAB), each stored straight into the flat gradient buffer. Each layer's
        # M = B*mh*mw rows are padded to Mpad, a multiple of the GEMM's k-block (64 rows bf16, 16 fp32), so that no
        # k-block straddles two layers; the pad rows are zero (nothing writes them) and add nothing to dW_i
        nmid, M = 3 * len(self.middle), B * mh * mw
        kb = 64 if self.lowp else 16
        Mpad = -(-M // kb) * kb
        self.mid_t = torch.zeros(nmid, Mpad, 728, device=self.device, dtype=self.adt)
        self.mid_dz = torch.zeros(nmid, Mpad, 728, device=self.device, dtype=self.adt) if train else None
        for bi, blk in enumerate(self.middle):
            for j, s in enumerate(blk):
                s.t = self.mid_t[3 * bi + j, :M].view(B, mh, mw, 728)
                s.z = A(B, mh, mw, 728)
        self.mid_out = [A(B, mh, mw, 728) for _ in self.middle]
        fh, fw = sh["out13"]
        for s in self.sep14:
            s.t = A(B, fh, fw, s.cin)
            s.z = A(B, fh, fw, s.cout)
        self.feat_dims = (fh, fw, 2048)
        if train:
            self.gcol = None if self.lowp else A(B * h2 * w2, 288)  # bf16: the data gradient is an implicit GEMM
            self.scratch = [A(maxel) for _ in range(6)]
            # batched middle-flow weight gradient: the 24 pointwise kernels are equally spaced in the flat gradient
            # buffer (every layer contributes dw kernel + pw kernel + gamma + beta, 728 * 739 parameters)
            o0 = self.offsets["block5_sepconv1/pointwise_kernel"][0]
            stride = self.offsets["block5_sepconv2/pointwise_kernel"][0] - o0
            names = ["block%d_sepconv%d/pointwise_kernel" % (b, j) for b in arch.MIDDLE_BLOCKS for j in (1, 2, 3)]
            assert all(self.offsets[n][0] == o0 + i * stride for i, n in enumerate(names))
            self.mid_gw_off, self.mid_gw_stride = o0, stride

    def _backbone_fwd(self, training):
        B, sh, w = self.B, self.shapes, self.w
        st = (lambda bn: bn.stats) if training else (lambda bn: None)
        # ---- block 1
        h1, w1 = sh["b1c1"]
        ops.conv_small_fwd(2, self.d, w["block1_conv1/kernel"], self.z11, stats=st(self.b1_bn1))
        self._bn_ready(self.b1_bn1, B * h1 * w1, training)
        h2, w2 = sh["b1c2"]
        ops.bn_apply(self.z11, self.b1_bn1.a, self.b1_bn1.b, act=1, out=self.a11)
        if self.b1_fold:
            ops.conv_tc_fwd_kwfold(self.a11, self.wl["block1_conv2/kernel"], self.z12, colstats=st(self.b1_bn2))
            self._bn_ready(self.b1_bn2, B * h2 * w2, training)
        else:
            ops.im2col(self.a11, self.col, 3, 3, 1, 0, 0, h2, w2)
            self._pw_fwd(self.col, self.wl["block1_conv2/kernel"].view(288, 64), self.z12.view(-1, 64), B * h2 * w2, 288,
                         64, self.b1_bn2, training)
        ops.bn_apply(self.z12, self.b1_bn2.a, self.b1_bn2.b, act=1, out=self.x2)
        # ---- entry blocks 2-4, middle 5-12, exit 13
        x = self.x2
        for e in self.entry:
            x = self._entry_fwd(e, x, training)
        for blk, out in zip(self.middle, self.mid_out):
            self._sep_fwd(blk[0], x, None, True, training)
            self._sep_fwd(blk[1], blk[0].z, blk[0].bn, True, training)
            self._sep_fwd(blk[2], blk[1].z, blk[1].bn, True, training)
            ops.bn_apply(blk[2].z, blk[2].bn.a, blk[2].bn.b, act=0, x=x, out=out)
            x = out
        x = self._entry_fwd(self.exit13, x, training)
        # ---- block 14 + head
        s1, s2 = self.sep14
        self._sep_fwd(s1, x, None, False, training)
        self._sep_fwd(s2, s1.z, s1.bn, True, training)
        ops.bn_apply(s2.z.view(B, -1, 2048), s2.bn.a, s2.bn.b, act=1, out=self.feat.view(B, -1, 2048))

    tail_param_key = "block5_sepconv1/depthwise_kernel"  # flat-buffer suffix that is final after part A

    def _backbone_bwd_a(self):
        """Block 14, exit block 13, middle blocks 12..5."""
        B, sh, w, g = self.B, self.shapes, self.w, self.g
        G1, G2, G3, S, R0, R1 = self.scratch
        # ---- block 14
        s1, s2 = self.sep14
        fh, fw = sh["out13"]
        M = B * fh * fw
        x13 = self.exit13["out"]
        g_feat = self.gfeat.view(M, 2048)
        self._bn_bwd_sums(g_feat, s2.z, s2.bn, act=1)
        g_y = self._view(G3, B, fh, fw, 1536)
        self._sep_bwd(s2, g_feat, s1.z, s1.bn, True, self._view(G2, M, 1536), g_y)
        g_x = self._view(R0, B, fh, fw, 1024)
        self._sep_bwd(s1, g_y.view(M, 1536), x13, None, False, self._view(G1, M, 1024), g_x,
                      out_bn=(self.exit13["zr"], self.exit13["res_bn"], False))
        # ---- exit block 13
        R_cur, R_nxt = R0, R1
        x_in13 = self.mid_out[-1]
        g_x = self._entry_bwd(self.exit13, x_in13, g_x, (G1, G2, G3, S, R_nxt),
                              (self.middle[-1][2].z, self.middle[-1][2].bn, False))
        R_cur, R_nxt = R_nxt, R_cur
        # ---- middle blocks 12..5
        mh, mw = sh["middle"]
        M = B * mh * mw
        for i in range(len(self.middle) - 1, -1, -1):
            blk = self.middle[i]
            x_in = self.mid_out[i - 1] if i > 0 else self.entry[-1]["out"]
            # the BN on x_in's residual path: the previous middle block's sepconv3 BN or entry block 4's residual BN
            x_bn = (self.middle[i - 1][2].z, self.middle[i - 1][2].bn, False) if i > 0 else \
                (self.entry[-1]["zr"], self.entry[-1]["res_bn"], False)
            # every dz is kept (mid_dz) for the batched weight gradient at the end of the middle flow (g_x is read again
            # as blk[0]'s add_src)
            dz = [self.mid_dz[3 * i + j, :M] for j in range(3)]
            g_t = self._view(G2, M, 728)
            gy2, gy1 = self._view(G3, B, mh, mw, 728), self._view(G1, B, mh, mw, 728)
            self._sep_bwd(blk[2], g_x.view(M, 728), blk[1].z, blk[1].bn, True, g_t, gy2, wgrad=False, dz=dz[2])
            self._sep_bwd(blk[1], gy2.view(M, 728), blk[0].z, blk[0].bn, True, g_t, gy1, wgrad=False, dz=dz[1])
            g_new = self._view(R_nxt, B, mh, mw, 728)
            self._sep_bwd(blk[0], gy1.view(M, 728), x_in, None, True, g_t, g_new, add_src=g_x, wgrad=False, out_bn=x_bn,
                          dz=dz[0])
            g_x = g_new
            R_cur, R_nxt = R_nxt, R_cur
        # dW_i = t_i^T dz_i for the 24 layers in ONE launch: both operands stacked along K (pixel rows, Mpad per layer),
        # split s of the K range = layer s, its [728, 728] product stored at the layer's place in the flat gradient
        # buffer. No split-K reduce-adds (every output tile has ONE writer: also bit-identical run to run), 192 k-blocks
        # per tile instead of 24 launches with ~10 k-blocks per CTA each
        n, Mpad = self.mid_t.shape[:2]
        ops.gemm(self.mid_t.view(n * Mpad, 728), True, self.mid_dz.view(n * Mpad, 728), True, self.grads[self.mid_gw_off:], 728,
                 728, n * Mpad, out_mode=ops.OUT_SLAB, splits=n, lda=728, ldb=728, ldd=728, slab_stride=self.mid_gw_stride)
        self._bwd_state = (g_x, R_cur, R_nxt)

    def _backbone_bwd_b(self, ga):
        """Entry blocks 4..2 and block 1."""
        B, sh, w, g = self.B, self.shapes, self.w, self.g
        G1, G2, G3, S, R0, R1 = self.scratch
        g_x, R_cur, R_nxt = self._bwd_state
        # ---- entry blocks 4..2
        for i in range(len(self.entry) - 1, -1, -1):
            e = self.entry[i]
            x_in = self.entry[i - 1]["out"] if i > 0 else self.x2
            x_bn = (self.entry[i - 1]["zr"], self.entry[i - 1]["res_bn"], False) if i > 0 else \
                (self.z12, self.b1_bn2, True)  # x2 = relu(BN(z12))
            g_x = self._entry_bwd(e, x_in, g_x, (G1, G2, G3, S, R_nxt), x_bn)
            R_cur, R_nxt = R_nxt, R_cur
        # ---- block 1
        h2, w2 = sh["b1c2"]
        h1, w1 = sh["b1c1"]
        M2 = B * h2 * w2
        # masked by the block-1 ReLU, with its sums, by block2_sepconv1's depthwise backward
        g_z12 = self._bn_bwd(g_x, self.z12, self.b1_bn2, M2)
        W2l = self.wl["block1_conv2/kernel"].view(288, 64)
        g_y11 = self._view(G1, B, h1, w1, 32)
        if self.b1_fold:
            ops.conv_tc_wgrad_kwfold(self.a11, g_z12.view(B, h2, w2, 64), g["block1_conv2/kernel"].view(3, 3, 32, 64))
        else:  # weight gradient from the forward's im2col buffer; fp32 also forms the column gradient (gcol)
            self._pw_bwd(self.col, W2l, g["block1_conv2/kernel"].view(288, 64), g_z12.view(M2, 64), self.gcol, M2, 288, 64)
        if self.lowp:
            # data gradient as implicit GEMM (csrc/gemm_tc.cu CONV mode: 95 us instead of a 120 us GEMM into a 428 MB
            # column-gradient buffer + 97 us col2im)
            ops.conv_tc_dgrad(g_z12.view(B, h2, w2, 64), self.wl["block1_conv2/kernel"], g_y11, 0, 0)
        else:
            ops.col2im(self.gcol, g_y11, 3, 3, 1, 0, 0, h2, w2)
        # the ReLU mask of block1_conv1_act is applied by the BatchNorm-backward reduction
        self._bn_bwd_sums(g_y11, self.z11, self.b1_bn1, act=1)
        g_z11 = self._bn_bwd(g_y11, self.z11, self.b1_bn1, B * h1 * w1)
        ops.conv_small_wgrad(2, self.d, g_z11, g["block1_conv1/kernel"], acc=self._gacc)
        ops.conv_small_dgrad(2, g_z11, w["block1_conv1/kernel"], ga)


class MobileNetSPNetEngine(SPNetEngineBase):
    """keras.applications.mobilenet.MobileNet (alpha 1, depth multiplier 1) backbone, BASELINE
    configs[2] (reference call site spnet/models.py:349-355). Post-activation blocks:
    DepthwiseConv2D 3x3 'same' stride s -> BN -> ReLU6 -> Conv 1x1 -> BN -> ReLU6.

    The depthwise stages run on the same packed kernels as Xception's (BN + ReLU6 of the
    previous stage applied on load). A stride-2 'same' depthwise convolution equals the stride-1
    'same' result sampled at odd positions of an even-sized dimension (TF pads only at the end)
    and at even positions of an odd-sized one (TF pads one on each side), so the four stride-2
    stages run the stride-1 kernel followed by a subsample (and its adjoint in backward)."""

    def _arch(self):
        return arch.mobilenet_shape_walk(self.H, self.W), arch.mobilenet_param_spec(self.H, self.W, self.n_out)

    def _build_backbone(self):
        sh = self.shapes
        self.c1_bn = self._mk_bn("conv1_bn", 32)
        self.blocks = []
        for i, (cin, cout, stride) in enumerate(arch.MOBILENET_BLOCKS, start=1):
            hw = sh["in%d" % i]
            b = dict(i=i, cin=cin, cout=cout, s=stride, hw=hw, ohw=sh["out%d" % i],
                     off=(1 - hw[0] % 2, 1 - hw[1] % 2),  # even size: odd positions; odd size: even positions
                     dwk=self.w["conv_dw_%d/depthwise_kernel" % i].view(3, 3, cin),
                     pw=self.w["conv_pw_%d/kernel" % i].view(cin, cout),
                     pwl=self.wl["conv_pw_%d/kernel" % i].view(cin, cout),
                     bn_dw=self._mk_bn("conv_dw_%d_bn" % i, cin), bn_pw=self._mk_bn("conv_pw_%d_bn" % i, cout))
            if self.can_train:
                b["gdwk"] = self.g["conv_dw_%d/depthwise_kernel" % i].view(3, 3, cin)
                b["gpw"] = self.g["conv_pw_%d/kernel" % i].view(cin, cout)
            self.blocks.append(b)

    def _alloc_backbone(self):
        B, sh, A = self.B, self.shapes, self._act
        h, w = sh["conv1"]
        self.zc1 = A(B, h, w, 32)
        maxel = B * h * w * 32
        for b in self.blocks:
            (h, w), (oh, ow) = b["hw"], b["ohw"]
            b["zd_full"] = A(B, h, w, b["cin"]) if b["s"] == 2 else None
            b["zd"] = A(B, oh, ow, b["cin"])
            b["t"] = A(B, oh, ow, b["cin"])
            b["zp"] = A(B, oh, ow, b["cout"])
            maxel = max(maxel, B * h * w * b["cin"], B * oh * ow * b["cout"])
        fh, fw = self.blocks[-1]["ohw"]
        self.feat_dims = (fh, fw, 1024)
        if self.can_train:
            self.scratch = [A(maxel) for _ in range(4)]

    def _backbone_fwd(self, training):
        B, w = self.B, self.w
        h, wd = self.shapes["conv1"]
        ops.conv_small_fwd(3, self.d, w["conv1/kernel"], self.zc1, stats=self.c1_bn.stats if training else None)
        self._bn_ready(self.c1_bn, B * h * wd, training)
        x, xbn = self.zc1, self.c1_bn
        for b in self.blocks:
            (oh, ow) = b["ohw"]
            M = B * oh * ow
            if b["s"] == 2:
                ops.dwconv3x3_fwd(x, b["dwk"], xbn.a, xbn.b, 2, out=b["zd_full"])
                ops.gather_s2(b["zd_full"], out=b["zd"], off=b["off"])
            else:
                ops.dwconv3x3_fwd(x, b["dwk"], xbn.a, xbn.b, 2, out=b["zd"])
            if training:
                ops.colstats(b["zd"], b["bn_dw"].stats)
            self._bn_ready(b["bn_dw"], M, training)
            ops.bn_apply(b["zd"], b["bn_dw"].a, b["bn_dw"].b, act=3, out=b["t"])
            self._pw_fwd(b["t"].view(M, b["cin"]), b["pwl"], b["zp"].view(M, b["cout"]), M, b["cin"], b["cout"],
                         b["bn_pw"], training)
            x, xbn = b["zp"], b["bn_pw"]
        fh, fw, fc = self.feat_dims
        ops.bn_apply(x.view(B, -1, fc), xbn.a, xbn.b, act=3, out=self.feat.view(B, -1, fc))

    def _backbone_bwd(self, ga):
        B, w, g = self.B, self.w, self.g
        bufs = self.scratch
        last = self.blocks[-1]
        fh, fw, fc = self.feat_dims
        # gradient w.r.t. relu6(BN(zp13)) -> masked in place, BN-backward sums accumulated
        g_y = self.gfeat.view(B, fh, fw, fc)
        self._bn_bwd_sums(g_y, last["zp"], last["bn_pw"], act=3)
        cur = None  # scratch buffer holding g_y (None: self.gfeat)
        for idx in range(len(self.blocks) - 1, -1, -1):
            b = self.blocks[idx]
            (h, wd), (oh, ow) = b["hw"], b["ohw"]
            M = B * oh * ow
            cin, cout = b["cin"], b["cout"]
            x, xbn = (self.blocks[idx - 1]["zp"], self.blocks[idx - 1]["bn_pw"]) if idx > 0 else (self.zc1, self.c1_bn)
            tb, fb, nb = [i for i in range(4) if i != cur][:3]
            # pointwise BN + 1x1 (g_y already carries the ReLU6 mask and this BN's backward sums)
            g_zp = self._bn_bwd(g_y, b["zp"], b["bn_pw"], M)
            g_t = self._view(bufs[tb], B, oh, ow, cin)
            self._pw_bwd(b["t"].view(M, cin), b["pwl"], b["gpw"], g_zp.view(M, cout), g_t.view(M, cin), M, cin, cout)
            # depthwise BN (+ReLU6 mask)
            self._bn_bwd_sums(g_t, b["zd"], b["bn_dw"], act=3)
            g_zd = self._bn_bwd(g_t, b["zd"], b["bn_dw"], M)
            g_full = ops.scatter_s2(g_zd, self._view(bufs[fb], B, h, wd, cin), off=b["off"]) if b["s"] == 2 else g_zd
            # depthwise 3x3: gradient w.r.t. relu6(BN_prev(x)) (masked) + BN_prev backward sums + dk
            g_y = self._view(bufs[nb], B, h, wd, cin)
            ops.dwconv3x3_bwd_fused(g_full, x, b["dwk"], b["gdwk"], in_a=xbn.a, in_b=xbn.b, relu=2, bn_mean=xbn.mean,
                                    bn_rstd=xbn.rstd, stats=xbn.stats, out=g_y, acc=self._gacc)
            cur = nb
        h, wd = self.shapes["conv1"]
        g_zc1 = self._bn_bwd(g_y, self.zc1, self.c1_bn, B * h * wd)
        ops.conv_small_wgrad(3, self.d, g_zc1, g["conv1/kernel"], acc=self._gacc)
        ops.conv_small_dgrad(3, g_zc1, w["conv1/kernel"], ga)


class InceptionResNetV2SPNetEngine(SPNetEngineBase):
    """keras.applications.InceptionResNetV2 backbone, BASELINE configs[3] (reference: the generic backbone
    branch, spnet/models.py:18,357-359). The architecture is a static program of layer records
    (spnet_b200/irv2.py); this class allocates one buffer per activation (+ its gradient) and walks the
    program forwards / backwards. Every convolution is a GEMM on the tcgen05 kernel (1x1: directly on the
    NHWC activation; k x k: through a generic im2col, recomputed in backward) with the BatchNorm
    statistics in its epilogue; BN(scale=False)+ReLU outputs are materialised because they are GEMM
    operands."""

    def _arch(self):
        return irv2.shape_walk(self.H, self.W), irv2.param_spec(self.H, self.W, self.n_out)

    def _build_backbone(self):
        h, w = self.shapes["stem"]
        self.prog = irv2.build_program(h, w)
        for op in self.prog.ops:
            if op["kind"] == "conv_bn":
                op["bnrec"] = self._mk_bn(op["bn"], op["cout"], scale=False)
        for op in self.prog.ops:
            if op["kind"] == "residual":  # the bias of the 1x1 "up" convolution is added here
                op["bias_name"] = next(p_ for p_ in self.prog.ops if p_["out"] is op["inputs"][1])["name"] + "/bias"
        # which backward contribution to an activation's gradient comes first (writes) vs later (accumulates)
        seen = set()
        for op in reversed(self.prog.ops):
            op["first"] = []
            for x in op["inputs"]:
                op["first"].append(x.idx not in seen)
                seen.add(x.idx)

    def _alloc_backbone(self):
        B, A, prog = self.B, self._act, self.prog
        train = self.can_train
        self.data, self.grad = {}, {}
        out = prog.output
        self.feat_dims = (out.h, out.w, out.c)
        for sy in prog.syms:
            if sy is prog.input or sy is out:
                continue
            self.data[sy.idx] = A(B, sy.h, sy.w, sy.c)
            if train:
                self.grad[sy.idx] = A(B, sy.h, sy.w, sy.c)
        col_el, tmp_el = 8, 8
        for op in prog.ops:
            o = op["out"]
            if op["kind"] == "conv_bn":
                op["z"] = A(B, o.h, o.w, o.c)
                if not (op["kh"] == 1 and op["kw"] == 1 and op["stride"] == 1) and op["cin"] != 3 and not self._implicit(op):
                    col_el = max(col_el, B * o.h * o.w * op["kh"] * op["kw"] * op["cin"])
            elif op["kind"] == "maxpool":
                op["argmax"] = A(B, o.h, o.w, o.c, dtype=torch.uint8) if train else None
            for x in op["inputs"]:
                tmp_el = max(tmp_el, B * x.h * x.w * x.c)
        self.col = A(col_el)
        if train:
            self.gcol = A(col_el)
            self.tmp = A(tmp_el)

    def _alloc_activations(self):
        super()._alloc_activations()
        B, out = self.B, self.prog.output
        self.data[self.prog.input.idx] = self.d
        self.data[out.idx] = self.feat.view(B, out.h, out.w, out.c)
        if self.can_train:
            self.grad[out.idx] = self.gfeat.view(B, out.h, out.w, out.c)

    # ---- helpers
    def _implicit(self, op):
        """k x k stride-1 convolutions of the bf16 engine run as implicit GEMM (csrc/gemm_tc.cu CONV modes): no
        im2col / col2im buffers. fp32, the few stride-2 convolutions and the deterministic mode (the implicit weight
        gradient reduce-adds fp32 partials from many CTAs) keep the im2col + GEMM route."""
        return (self.lowp and not self.deterministic and op["stride"] == 1 and (op["kh"] > 1 or op["kw"] > 1)
                and op["cin"] != 3)

    def _conv_operand(self, op, x):
        """GEMM A operand [M, K] of a convolution: the activation itself for 1x1, an im2col buffer otherwise."""
        o = op["out"]
        M, K = self.B * o.h * o.w, op["kh"] * op["kw"] * op["cin"]
        if op["kh"] == 1 and op["kw"] == 1 and op["stride"] == 1:
            return x.view(M, K), M, K
        col = self.col[:M * K].view(M, K)
        ops.im2col(x, col, op["kh"], op["kw"], op["stride"], op["pt"], op["pl"], o.h, o.w)
        return col, M, K

    def _backbone_fwd(self, training):
        B, w, wl = self.B, self.w, self.wl
        for op in self.prog.ops:
            kind, o = op["kind"], op["out"]
            xs = [self.data[x.idx] for x in op["inputs"]]
            y = self.data[o.idx]
            if kind == "conv_bn":
                bn, z = op["bnrec"], op["z"]
                M = B * o.h * o.w
                if op["cin"] == 3:  # first convolution: 3x3 stride 2 'valid' on the 3-channel stem output
                    ops.conv_small_fwd(2, xs[0], w[op["name"] + "/kernel"], z, stats=bn.stats if training else None)
                    self._bn_ready(bn, M, training)
                elif self._implicit(op):
                    ops.conv_tc_fwd(xs[0], wl[op["name"] + "/kernel"], z, op["pt"], op["pl"],
                                    colstats=bn.stats if training else None)
                    self._bn_ready(bn, M, training)
                else:
                    A_, M, K = self._conv_operand(op, xs[0])
                    self._pw_fwd(A_, wl[op["name"] + "/kernel"].view(K, o.c), z.view(M, o.c), M, K, o.c, bn, training)
                ops.bn_apply(z, bn.a, bn.b, act=1 if op["act"] else 0, out=y)
            elif kind == "conv_bias":
                M = B * o.h * o.w
                ops.gemm(xs[0].view(M, op["cin"]), False, wl[op["name"] + "/kernel"].view(op["cin"], o.c), True, y.view(M, o.c),
                         M, o.c, op["cin"], out_mode=ops.OUT_T)
            elif kind == "maxpool":
                ops.maxpool3s2_valid_fwd(xs[0], y, op["argmax"] if training else None)
            elif kind == "avgpool":
                ops.avgpool3s1(xs[0], y)
            elif kind == "concat":
                M, off = B * o.h * o.w, 0
                for x, t in zip(op["inputs"], xs):
                    ops.copy2d(t, 0, x.c, y, off, o.c, M, x.c)
                    off += x.c
            elif kind == "residual":
                ops.residual_fwd(xs[0], xs[1], w[op["bias_name"]], op["scale"], op["relu"], y)

    def _into(self, x, first):
        """Where a full-tensor gradient contribution for activation x goes: its gradient buffer when it is the
        first contribution, a temporary (added afterwards by _merge) otherwise."""
        g = self.grad[x.idx]
        return g if first else self.tmp[:g.numel()].view(g.shape)

    def _merge(self, x, first):
        if not first:
            g = self.grad[x.idx]
            n = g.numel()
            ops.copy2d(self.tmp, 0, x.c, g, 0, x.c, n // x.c, x.c, accumulate=True)

    def _backbone_bwd(self, ga):
        B, w, wl, g_ = self.B, self.w, self.wl, self.g
        self.grad[self.prog.input.idx] = ga
        for op in reversed(self.prog.ops):
            kind, o = op["kind"], op["out"]
            ins = op["inputs"]
            xs = [self.data[x.idx] for x in ins]
            gy = self.grad[o.idx]
            M = B * o.h * o.w
            if kind == "conv_bn":
                bn, z = op["bnrec"], op["z"]
                self._bn_bwd_sums(gy, z, bn, act=1 if op["act"] else None)
                dz = self._bn_bwd(gy, z, bn, M)
                gW = g_[op["name"] + "/kernel"]
                if op["cin"] == 3:
                    ops.conv_small_wgrad(2, xs[0], dz, gW, acc=self._gacc)
                    ops.conv_small_dgrad(2, dz, w[op["name"] + "/kernel"], ga)
                    continue
                if self._implicit(op):
                    ops.conv_tc_wgrad(xs[0], dz, gW, op["pt"], op["pl"])
                    tgt = self._into(ins[0], op["first"][0])
                    ops.conv_tc_dgrad(dz, wl[op["name"] + "/kernel"], tgt, op["pt"], op["pl"])
                    self._merge(ins[0], op["first"][0])
                    continue
                A_, M, K = self._conv_operand(op, xs[0])
                Wl = wl[op["name"] + "/kernel"].view(K, o.c)
                if K == op["cin"]:  # 1x1: the data gradient is the input gradient itself
                    tgt = self._into(ins[0], op["first"][0])
                    self._pw_bwd(A_, Wl, gW.view(K, o.c), dz.view(M, o.c), tgt.view(M, K), M, K, o.c)
                    self._merge(ins[0], op["first"][0])
                else:
                    gcol = self.gcol[:M * K].view(M, K)
                    self._pw_bwd(A_, Wl, gW.view(K, o.c), dz.view(M, o.c), gcol, M, K, o.c)
                    ops.col2im(gcol, self.grad[ins[0].idx], op["kh"], op["kw"], op["stride"], op["pt"], op["pl"], o.h, o.w,
                               accumulate=not op["first"][0])
            elif kind == "conv_bias":
                K = op["cin"]
                tgt = self._into(ins[0], op["first"][0])
                self._pw_bwd(xs[0].view(M, K), wl[op["name"] + "/kernel"].view(K, o.c), g_[op["name"] + "/kernel"].view(K, o.c),
                             gy.view(M, o.c), tgt.view(M, K), M, K, o.c)
                self._merge(ins[0], op["first"][0])
                assert self._gacc is None or o.c <= self._gacc.numel() // 2
                ops.colsum_rows(gy.view(M, o.c), g_[op["name"] + "/bias"], acc=self._gacc)
            elif kind == "maxpool":
                tgt = self._into(ins[0], op["first"][0])
                ops.maxpool3s2_valid_bwd(gy, op["argmax"], tgt)
                self._merge(ins[0], op["first"][0])
            elif kind == "avgpool":
                ops.avgpool3s1(gy, self.grad[ins[0].idx], bwd=True, accumulate=not op["first"][0])
            elif kind == "concat":
                off = 0
                for x, first in zip(ins, op["first"]):
                    ops.copy2d(gy, off, o.c, self.grad[x.idx], 0, x.c, M, x.c, accumulate=not first)
                    off += x.c
            elif kind == "residual":
                ops.residual_bwd(gy, self.data[o.idx], op["scale"], op["relu"], self.grad[ins[0].idx],
                                 not op["first"][0], self.grad[ins[1].idx])
