"""The bf16 backward pass of one Xception-SPNet training step, layer by layer, against fp64.

test_bf16_kernels_layer_by_layer_teacher_forced (test_parity_configs_gpu.py) does this for the forward pass; here every
layer of the backward pass is recomputed in fp64 from the engine's stored forward tensors (x, t, z, a11, feat, argmax
positions), its BatchNorm mean / rstd / a / b, and the gradient that reached the layer in the step, captured while
the step runs. The reference follows the network's definition (which input a layer reads, which BatchNorm + ReLU
sits on it, which residual gradient joins it), not the engine's call arguments, so a kernel that is fed the wrong
mask, sum, residual or buffer fails here even when it computes its own operation correctly. Where one layer's output
gradient is the next layer's input, the two captures must be equal bit for bit.

Cases: the route bench.py trains with (bf16, deterministic=False: kw-fold block1_conv2, slab-free fused pointwise
backward, reduce-added weight gradients), deterministic=True (slabs, accumulators, im2col for block1_conv2), and every
BatchNorm on its moving statistics, set to those of the batch (backward count 0: c1 = c2 = 0, dz = a * g).

Tolerances are the forward test's: a bf16 output is at most one bf16 ulp beyond 1e-5 x sum|terms| of the fp64 value
and differs from its rounding on fewer than 2 % of the elements; an fp32 weight gradient is within 1e-5 x sum|terms|
of the fp64 value built from the same bf16 operands. The per-layer figures are written by the parity tests' record()
as bf16_backward_layer_by_layer_<case>.json."""
import inspect

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from oracle import xception_torch as xt  # noqa: E402
from test_parity_configs_gpu import frames, perturbed_weights, record  # noqa: E402

CASES = {"default": dict(deterministic=False, moving=False),
         "deterministic": dict(deterministic=True, moving=False),
         "moving_statistics": dict(deterministic=False, moving=True)}


def _nchw(t):
    return t.permute(0, 3, 1, 2).contiguous()


def _nhwc(t):
    return t.permute(0, 2, 3, 1)


def _oihw(k):  # Keras kernel [kh, kw, cin, cout] -> torch [cout, cin, kh, kw]
    return k.permute(3, 2, 0, 1).contiguous()


def _keras(k):  # torch [cout, cin, kh, kw] -> Keras [kh, kw, cin, cout]
    return k.permute(2, 3, 1, 0)


def _capture(eng):
    """Wraps the engine's backward helpers on this instance: each clones the gradient it receives before the original
    method runs and the gradients it produced afterwards (stream-ordered clones, so no synchronisation)."""
    cap = {"sums": {}, "bn_bwd": {}, "sep": {}, "entry": {}, "bn3": {}}

    def wrap(meth, before, after):
        orig = getattr(eng, meth)
        sig = inspect.signature(orig)

        def wrapped(*args, **kw):
            a = sig.bind(*args, **kw)
            a.apply_defaults()
            rec = before(a.arguments)
            out = orig(*args, **kw)
            after(a.arguments, out, rec)
            return out
        setattr(eng, meth, wrapped)

    def put(kind, key, rec):
        assert key not in cap[kind], (kind, key)  # every layer runs its backward once per step
        cap[kind][key] = rec

    def clone(t):
        return None if t is None else t.clone()

    wrap("_bn_bwd_sums", lambda a: {"g": a["g"].clone()},
         lambda a, out, r: put("sums", a["bn"].name, dict(r, g_masked=a["g"].clone())))
    wrap("_bn_bwd", lambda a: {"g": a["g"].clone()},
         lambda a, out, r: put("bn_bwd", a["bn"].name, dict(r, dz=out.clone())))
    wrap("_sep_bwd", lambda a: {"g": a["g"].clone(), "add_strided": clone(a["add_strided"])},
         lambda a, out, r: put("sep", a["s"].name, dict(r, g_t=a["g_t"].clone(), g_in=a["g_in"].clone())))
    wrap("_entry_bwd", lambda a: {"g_out": a["g_out"].clone()},
         lambda a, out, r: put("entry", a["e"]["blk"], dict(r, g_x=out.clone())))
    wrap("_bn3_bwd", lambda a: {"g": a["gbuf"].clone()},
         lambda a, out, r: put("bn3", a["bn"].name, dict(r, dz=a["gbuf"].clone())))
    wrap("_backbone_bwd_b", lambda a: {}, lambda a, out, r: cap.__setitem__("ga", a["ga"].clone()))
    return cap


def _dw_bwd_ref(g_t, xin, k):
    """Depthwise 3x3 'same' (stride 1) backward in fp64, NHWC: the transposed convolution of g_t, the kernel gradient
    sum_p g_t[p] xin[p + tap], and the sums of |terms| of both."""
    B, H, W, C = g_t.shape
    gp, xp = F.pad(g_t, (0, 0, 1, 1, 1, 1)), F.pad(xin, (0, 0, 1, 1, 1, 1))
    gin, sgin = torch.zeros_like(g_t), torch.zeros_like(g_t)
    dk, sdk = torch.zeros(3, 3, C, dtype=torch.float64, device=g_t.device), torch.zeros(3, 3, C, dtype=torch.float64, device=g_t.device)
    for kh in range(3):
        for kw in range(3):
            gs = gp[:, 2 - kh:2 - kh + H, 2 - kw:2 - kw + W]
            gin += gs * k[kh, kw]
            sgin += gs.abs() * k[kh, kw].abs()
            xs = xp[:, kh:kh + H, kw:kw + W]
            dk[kh, kw] = (xs * g_t).sum((0, 1, 2))
            sdk[kh, kw] = (xs.abs() * g_t.abs()).sum((0, 1, 2))
    return gin, sgin, dk, sdk


@pytest.mark.parametrize("case", sorted(CASES))
def test_bf16_backward_layer_by_layer_teacher_forced(case):
    from spnet_b200 import arch, ops
    from spnet_b200.engine import XceptionSPNetEngine
    cfg = CASES[case]
    H, W, B = 384, 512, 8
    X, Y = frames(B, 7300)
    w = perturbed_weights(xt.xception_spnet_spec, H, W, 113)
    eng = XceptionSPNetEngine(H, W, B, dtype="bf16", weights=w, dropout_rate=0.0, deterministic=cfg["deterministic"])
    eng.load_batch(X, Y)
    if cfg["moving"]:
        # moving statistics that describe this batch, as a trained model's do. With the perturbed ones the activations
        # shrink layer after layer and the gradients reach 1e-15 by block 3, below the 2^-56 quantum of the BatchNorm
        # sum accumulators (csrc/common.cuh stat_add), where no relative bound means anything
        eng.forward(training=True)
        for bn in eng.bns:
            bn.mm.copy_(bn.mean)
            bn.mv.copy_((1.0 / bn.rstd.double() ** 2 - arch.BN_EPS).clamp_min(0.0))
        eng.bn_use_moving = "all"
    cap = _capture(eng)
    # eager step, stopped before Adam: the weights stay those the step used (a hook that returns without setting
    # skip_default_optimizer would still let train_step run the optimiser)
    eng.grad_hook = lambda e: setattr(e, "skip_default_optimizer", True)
    eng.train_step(lr=1e-5)
    torch.cuda.synchronize()
    assert eng.b1_fold == (not cfg["deterministic"])

    rep, bad, checked = {}, [], set()

    def check(name, got, ref64, scale64):
        """bf16 output: at most 1 bf16 ulp beyond 1e-5 x sum|terms|, on under 2 % of the elements."""
        got = got.reshape(ref64.shape)
        ref = ref64.to(torch.bfloat16)
        ulp = torch.pow(2.0, torch.floor(torch.log2(ref.double().abs().clamp_min(1e-30))) - 7)
        excess = ((got.double() - ref.double()).abs() - 1e-5 * scale64) / ulp
        frac = float((got != ref).double().mean())
        worst = float(excess.max())
        rep[name] = {"mismatch_fraction": frac, "max_ulps": max(worst, 0.0)}
        if not (worst <= 1.0 + 1e-9 and frac < 2e-2):
            bad.append((name, frac, worst))

    def check_f32(name, got, ref64, scale64):
        """fp32 result: within 1e-5 x sum|terms| of the fp64 value."""
        err = (got.double().reshape(ref64.shape) - ref64).abs()
        q = float((err / (1e-5 * scale64).clamp_min(1e-300)).max())
        rep[name] = {"max_error_over_bound": q}
        if not q <= 1.0:
            bad.append((name, q))

    def grad(key, ref64, scale64):
        checked.add(key)
        check_f32(key, eng.g[key], ref64, scale64)

    def same(name, produced, consumed):
        """A gradient handed from one layer to the next: what the consumer read is what the producer wrote."""
        ok = produced is not None and consumed is not None and torch.equal(produced, consumed.view(produced.shape))
        rep[name + "/handoff"] = {"equal": ok}
        if not ok:
            bad.append((name + "/handoff",))

    def bn_backward(bn, z, g, rows, stored=None):
        """g = gradient wrt the output of BatchNorm bn of z. Checks its gamma / beta gradients, c1, c2 and dz (the
        engine's stored dz when stored, else ops.bn_bwd_dz of g, which is what the fused pointwise backward forms on
        chip, bit for bit); returns that dz."""
        C = bn.C
        zd, gd = z.double().reshape(-1, C), g.double().reshape(-1, C)
        mu, rs = bn.mean.double(), bn.rstd.double()
        sg, sgx = gd.sum(0), (gd * (zd - mu) * rs).sum(0)
        ag, agx = gd.abs().sum(0), (gd.abs() * (zd.abs() + mu.abs()) * rs).sum(0)
        grad(bn.name + "/beta", sg, ag)
        grad(bn.name + "/gamma", sgx, agx)
        if cfg["moving"]:
            ok = not bool(bn.c1.any()) and not bool(bn.c2.any())
            rep[bn.name + "/c1_c2_zero"] = {"equal": ok}
            if not ok:
                bad.append((bn.name + "/c1_c2_zero",))
        else:
            check_f32(bn.name + "/c1", bn.c1, sg / rows, ag / rows)
            check_f32(bn.name + "/c2", bn.c2, sgx / rows, agx / rows)
        if stored is not None:
            same(bn.name + "/bn_backward_input", g, stored["g"])
            dz = stored["dz"]
        else:
            dz = ops.bn_bwd_dz(g.reshape(-1, C).contiguous(), z, bn.a, bn.mean, bn.rstd, bn.c1, bn.c2)
        a, c1, c2 = bn.a.double(), bn.c1.double(), bn.c2.double()
        check(bn.name + "/dz", dz.reshape(-1, C), a * (gd - c1 - (zd - mu) * rs * c2),
              a.abs() * (gd.abs() + c1.abs() + (zd.abs() + mu.abs()) * rs * c2.abs()))
        return dz.reshape(-1, C)

    def pointwise(name, t, Wl, dz, gA, key):
        """z = t W: data gradient dz W^T (bf16) and weight gradient t^T dz (fp32)."""
        K, N = Wl.shape
        t2, dz2, W2 = t.double().reshape(-1, K), dz.double().reshape(-1, N), Wl.double()
        if gA is None:
            rep[name + "/data_grad"] = {"missing": True}
            bad.append((name + "/data_grad", "missing"))
        else:
            check(name + "/data_grad", gA, dz2 @ W2.T, dz2.abs() @ W2.abs().T)
        grad(key, t2.T @ dz2, t2.abs().T @ dz2.abs())
        return dz2 @ W2.T

    def sep(s, g_in_expected, x, in_bn, relu, add_src=None, add_strided=None, out_mask=None):
        """SeparableConv2D s = pointwise(depthwise(relu?(in_bn(x)))) followed by BatchNorm s.bn. g_in_expected: the
        gradient wrt s.bn's output as the layer above produced it. add_src / add_strided (fp64 reference when the
        engine's own is missing): residual gradients joining the input gradient; out_mask: the ReLU mask of the
        BatchNorm that produced x (block 2 only)."""
        r = cap["sep"][s.name]
        same(s.name + "/incoming", g_in_expected, r["g"])
        M = B * s.H * s.W
        dz = bn_backward(s.bn, s.z, r["g"], M, cap["bn_bwd"].get(s.bn.name))
        pointwise(s.name + "/pointwise", s.t, s.pwl, dz, r["g_t"], s.name + "/pointwise_kernel")
        xin = x.double()
        if in_bn is not None:
            xin = xin * in_bn.a.double() + in_bn.b.double()
        live = xin > 0
        if relu:
            xin = xin * live
        gin, sgin, dk, sdk = _dw_bwd_ref(r["g_t"].double().view(B, s.H, s.W, s.cin), xin, s.dwk.double())
        if relu:
            gin, sgin = gin * live, sgin * live
        if add_src is not None:
            gin, sgin = gin + add_src.double(), sgin + add_src.double().abs()
        if add_strided is not None:
            gin[:, ::2, ::2] += add_strided.double()
            sgin[:, ::2, ::2] += add_strided.double().abs()
        if out_mask is not None:
            gin, sgin = gin * out_mask, sgin * out_mask
        check(s.name + "/input_grad", r["g_in"], gin, sgin)
        grad(s.name + "/depthwise_kernel", dk, sdk)
        return r

    def entry(e, x_in, g_expected, out_mask=None):
        """Entry / exit block: sepconv1 -> sepconv2 -> max-pool 3x3 s2 'same', plus the 1x1 stride-2 residual conv."""
        r = cap["entry"][e["blk"]]
        same("block%d/incoming" % e["blk"], g_expected, r["g_out"])
        (eh, ew), (oh, ow) = e["hw"], e["ohw"]
        cin, c = e["cin"], e["c"]
        s1, s2 = e["sep1"], e["sep2"]
        g_out = r["g_out"]
        # residual branch: its data gradient reaches x through sepconv1's depthwise backward (add_strided)
        dz_r = bn_backward(e["res_bn"], e["zr"], g_out, B * oh * ow, cap["bn_bwd"].get(e["res_bn"].name))
        g_xs = cap["sep"][s1.name]["add_strided"]
        ref_xs = pointwise(e["res"], e["xs"], eng.wl[e["res"] + "/kernel"].view(cin, c), dz_r, g_xs, e["res"] + "/kernel")
        if g_xs is None:
            g_xs = ref_xs.to(torch.bfloat16)
        # max-pool: the gradient goes to the first maximum of each window of fma(z, a, b)
        y2 = (s2.z.double() * s2.bn.a.double() + s2.bn.b.double()).permute(0, 3, 1, 2).requires_grad_(True)
        pooled = xt.maxpool3s2_same(y2)
        go = _nchw(g_out.double().view(B, oh, ow, c))
        gref, = torch.autograd.grad(pooled, y2, go, retain_graph=True)
        gabs, = torch.autograd.grad(pooled, y2, go.abs())
        check("block%d_pool/input_grad" % e["blk"], cap["sep"][s2.name]["g"], _nhwc(gref), _nhwc(gabs))
        r2 = sep(s2, cap["sep"][s2.name]["g"], s1.z, s1.bn, True)
        r1 = sep(s1, r2["g_in"], x_in, None, e["relu_in"], add_strided=g_xs.view(B, oh, ow, cin), out_mask=out_mask)
        same("block%d/outgoing" % e["blk"], r1["g_in"], r["g_x"])
        return r["g_x"]

    # ---- Dense head: y = feat W + bias
    g_feat = cap["sums"]["block14_sepconv2_bn"]["g"]
    gy, gyl = eng.gy.double(), eng.gyl
    same("FinalOutput/gy_bf16", eng.gy.to(torch.bfloat16), gyl)
    Wd, feat = eng.wl["FinalOutput/kernel"].double(), eng.feat.double()
    check("FinalOutput/input_grad", g_feat.view(B, -1), gyl.double() @ Wd.T, gyl.double().abs() @ Wd.abs().T)
    grad("FinalOutput/kernel", feat.T @ gyl.double(), feat.abs().T @ gyl.double().abs())
    grad("FinalOutput/bias", gy.sum(0), gy.abs().sum(0))
    # ---- block 14: feat = relu(BN(sepconv2)), sepconv2 reads relu(BN(sepconv1)), sepconv1 reads block 13's output
    s1, s2 = eng.sep14
    rec = cap["sums"][s2.bn.name]
    live = (s2.z.double() * s2.bn.a.double() + s2.bn.b.double() > 0).view(-1, 2048)
    same("block14_sepconv2_act/mask", (g_feat.view(-1, 2048) * live).to(torch.bfloat16), rec["g_masked"])
    r2 = sep(s2, rec["g_masked"], s1.z, s1.bn, True)
    r1 = sep(s1, r2["g_in"], eng.exit13["out"], None, False)
    # ---- exit block 13, middle blocks 12..5 (x + sepconv3(sepconv2(sepconv1(relu(x))))), entry blocks 4..2
    g_x = entry(eng.exit13, eng.mid_out[-1], r1["g_in"])
    for i in range(len(eng.middle) - 1, -1, -1):
        blk = eng.middle[i]
        x_in = eng.mid_out[i - 1] if i > 0 else eng.entry[-1]["out"]
        r3 = sep(blk[2], g_x, blk[1].z, blk[1].bn, True)
        r2 = sep(blk[1], r3["g_in"], blk[0].z, blk[0].bn, True)
        r1 = sep(blk[0], r2["g_in"], x_in, None, True, add_src=r3["g"].view(x_in.shape))
        g_x = r1["g_in"]
    for i in range(len(eng.entry) - 1, -1, -1):
        e = eng.entry[i]
        if i > 0:
            g_x = entry(e, eng.entry[i - 1]["out"], g_x)
        else:  # block 2 reads x2 = relu(BN(z12)): its input gradient carries that ReLU's mask
            bn = eng.b1_bn2
            g_x = entry(e, eng.x2, g_x, out_mask=eng.z12.double() * bn.a.double() + bn.b.double() > 0)
    # ---- block 1: conv1 3x3 s2 'valid' 3 -> 32, BN, ReLU (a11 stored), conv2 3x3 'valid' 32 -> 64, BN, ReLU (= x2)
    b1, b2 = eng.b1_bn1, eng.b1_bn2
    h1, w1 = eng.z11.shape[1:3]
    h2, w2 = eng.z12.shape[1:3]
    dz12 = bn_backward(b2, eng.z12, g_x, B * h2 * w2, cap["bn_bwd"].get(b2.name))
    dz12 = _nchw(dz12.double().view(B, h2, w2, 64))
    k2 = _oihw(eng.wl["block1_conv2/kernel"].double())
    rec = cap["sums"][b1.name]
    check("block1_conv2/data_grad", rec["g"], _nhwc(torch.nn.grad.conv2d_input((B, 32, h1, w1), k2, dz12)),
          _nhwc(torch.nn.grad.conv2d_input((B, 32, h1, w1), k2.abs(), dz12.abs())))
    a11 = _nchw(eng.a11.double())
    grad("block1_conv2/kernel", _keras(torch.nn.grad.conv2d_weight(a11, k2.shape, dz12)),
         _keras(torch.nn.grad.conv2d_weight(a11.abs(), k2.shape, dz12.abs())))
    live = eng.z11.double() * b1.a.double() + b1.b.double() > 0
    same("block1_conv1_act/mask", (rec["g"].double().view(live.shape) * live).to(torch.bfloat16), rec["g_masked"])
    dz11 = bn_backward(b1, eng.z11, rec["g_masked"], B * h1 * w1, cap["bn_bwd"].get(b1.name))
    dz11 = _nchw(dz11.double().view(B, h1, w1, 32))
    k1 = _oihw(eng.w["block1_conv1/kernel"].double())
    d = _nchw(eng.d.double())
    H2, W2 = eng.d.shape[1:3]
    check("block1_conv1/data_grad", cap["ga"], _nhwc(torch.nn.grad.conv2d_input((B, 3, H2, W2), k1, dz11, stride=2)),
          _nhwc(torch.nn.grad.conv2d_input((B, 3, H2, W2), k1.abs(), dz11.abs(), stride=2)))
    grad("block1_conv1/kernel", _keras(torch.nn.grad.conv2d_weight(d, k1.shape, dz11, stride=2)),
         _keras(torch.nn.grad.conv2d_weight(d.abs(), k1.shape, dz11.abs(), stride=2)))
    # ---- stem: d = BN3(conv3(act(BN2(conv2(act(BN1(avgpool2(conv1(x0)))))))) + avgpool2(x0), act = LeakyReLU(0.1)
    bn1, bn2, bn3 = eng.stem_bn
    npx = B * H2 * W2
    r = cap["bn3"][bn3.name]
    same("stem_out/grad", cap["ga"], r["g"])   # dropout rate 0: the gradient wrt BN3's output is dL/dd
    dz = bn_backward(bn3, eng.c3, r["g"], npx, r)
    for conv, x, bn_in, bn_out in (("conv2d_3", eng.c2, bn2, bn3), ("conv2d_2", eng.p1, bn1, bn2)):
        dzn = _nchw(dz.double().view(B, H2, W2, 3))
        k = _oihw(eng.w[conv + "/kernel"].double())
        y = _nchw(x.double() * bn_in.a.double() + bn_in.b.double())
        slope = torch.where(y > 0, 1.0, 0.1)
        grad(conv + "/kernel", _keras(torch.nn.grad.conv2d_weight(y * slope, k.shape, dzn, padding=1)),
             _keras(torch.nn.grad.conv2d_weight((y * slope).abs(), k.shape, dzn.abs(), padding=1)))
        r = cap["bn3"][bn_in.name]
        check(conv + "/data_grad", r["g"], _nhwc(torch.nn.grad.conv2d_input(y.shape, k, dzn, padding=1) * slope),
              _nhwc(torch.nn.grad.conv2d_input(y.shape, k.abs(), dzn.abs(), padding=1) * slope))
        dz = bn_backward(bn_in, x, r["g"], npx, r)
    # conv2d_1 (3x3 'same', 1 -> 3) followed by AveragePooling2D(2): the engine runs it as one 4x4 stride-2 convolution
    g1 = _nchw(dz.double().view(B, H2, W2, 3)).repeat_interleave(2, 2).repeat_interleave(2, 3) * 0.25
    x0 = _nchw(eng.x0.double())
    grad("conv2d_1/kernel", _keras(torch.nn.grad.conv2d_weight(x0, (3, 1, 3, 3), g1, padding=1)),
         _keras(torch.nn.grad.conv2d_weight(x0.abs(), (3, 1, 3, 3), g1.abs(), padding=1)))

    rep["summary"] = {"checks": len(rep), "failed": len(bad),
                      "worst_mismatch_fraction": max(v.get("mismatch_fraction", 0.0) for v in rep.values()),
                      "worst_ulps": max(v.get("max_ulps", 0.0) for v in rep.values()),
                      "worst_fp32_error_over_bound": max(v.get("max_error_over_bound", 0.0) for v in rep.values())}
    record("bf16_backward_layer_by_layer_" + case, rep)
    assert checked == set(eng.g), (sorted(set(eng.g) - checked), sorted(checked - set(eng.g)))
    assert not bad, bad[:20]
