"""One InceptionResNetV2-SPNet training step, op by op, against fp64.

The backbone is a static program (spnet_b200/irv2.py) of conv_bn, conv_bias, maxpool, avgpool, concat and residual
ops. After one eager training step every op is recomputed in fp64 from the engine's own stored tensors: its inputs
(eng.data), z, argmax, the BatchNorm affines and statistics, the low-precision weights, and, for the backward pass,
the gradients that reached the op during the step. Those are captured by walking the program backwards through a
list whose reversed() takes stream-ordered clones around every op: the op's output gradient and the gradient buffer
of each input before the op runs, and the same buffers (plus the column / temporary buffer the op wrote its
contribution to) after it ran. For every input the reference is `after = (0 if first else before) + contribution`,
so a dropped, doubled or misplaced gradient contribution, a wrong `accumulate` flag, a wrong residual scale or mask
fails here even where every kernel computes its own operation correctly. Where one op's gradient is the next op's
input, the two captures must be equal bit for bit.

Cases: the route bench.py trains with (bf16, implicit-GEMM convolutions, reduce-added weight gradients), the bf16
deterministic mode (im2col + slab GEMMs, accumulator bias gradients) and the fp32 deterministic mode (im2col + the
SIMT GEMM). The engine is built with SPNET_B200_POISON=1: every activation, gradient and scratch buffer starts as NaN,
so a read of memory that nothing wrote shows up.

Tolerances are those of the Xception layer-by-layer tests: a bf16 output is at most one bf16 ulp beyond
1e-5 x sum|terms| of its fp64 value and differs from its rounding on fewer than 2 % of the elements; an fp32 output
(every weight gradient, every output of the fp32 engine) is within 1e-5 x sum|terms|; copies, routes, masks and
argmax positions are bit-exact. Where the engine stores an intermediate (a column gradient, a contribution waiting in
the temporary buffer to be added), that intermediate is checked on its own and the next step is rebuilt from it as
stored, so that each check covers one rounding. The per-op figures are written by the parity tests' record() as
irv2_layer_by_layer_<case>.json."""
import time

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from oracle import xception_torch as xt  # noqa: E402
from test_parity_configs_gpu import frames, perturbed_weights, record  # noqa: E402

CASES = {"bf16_default": dict(dtype="bf16", deterministic=False, implicit=98),
         "bf16_deterministic": dict(dtype="bf16", deterministic=True, implicit=0),
         "fp32_deterministic": dict(dtype="fp32", deterministic=True, implicit=0)}

# gradients this test does not rebuild: the SPNet stem (base-class code, checked layer by layer for Xception in
# test_backward_layer_by_layer_gpu.py) and the Dense head
EXCLUDED = ({"conv2d_%d/kernel" % i for i in (1, 2, 3)} | {"batch_normalization_%d/%s" % (i, p) for i in (1, 2, 3)
                                                          for p in ("gamma", "beta")}
            | {"FinalOutput/kernel", "FinalOutput/bias"})


def _nchw(t):
    return t.double().permute(0, 3, 1, 2).contiguous()


def _nhwc(t):
    return t.permute(0, 2, 3, 1)


def _conv(x, k, s, pt, pl, oh, ow):
    """TF convolution of x (NCHW fp64) with the Keras kernel k [kh, kw, cin, cout]: leading pads (pt, pl), trailing
    pads implied by (oh, ow) - negative for the 'valid' reductions that leave the last row or column unread."""
    kh, kw = k.shape[0], k.shape[1]
    h, w = x.shape[2], x.shape[3]
    pb, pr = (oh - 1) * s + kh - h - pt, (ow - 1) * s + kw - w - pl
    return F.conv2d(F.pad(x, (pl, pr, pt, pb)), k.permute(3, 2, 0, 1), stride=s)


class _Tap(list):
    """The program's op list. Iterating it is plain (the forward pass); reversed() (the backward pass) yields each
    op between clones of the gradient buffers it reads and writes, taken on the current stream."""

    def __init__(self, ops, eng):
        super().__init__(ops)
        self.eng, self.cap = eng, {}

    def __reversed__(self):
        eng = self.eng
        for i in range(len(self) - 1, -1, -1):
            op = self[i]
            ins = op["inputs"]
            rec = {"gy": eng.grad[op["out"].idx].clone(), "before": [eng.grad[x.idx].clone() for x in ins]}
            yield op
            rec["after"] = [eng.grad[x.idx].clone() for x in ins]
            g0 = eng.grad[ins[0].idx]
            if op["kind"] == "conv_bn" and _route(eng, op) == "im2col":
                o = op["out"]
                n = eng.B * o.h * o.w * op["kh"] * op["kw"] * op["cin"]
                rec["gcol"] = eng.gcol[:n].clone()
            elif op["kind"] in ("conv_bn", "conv_bias", "maxpool") and not op["first"][0] and op.get("cin") != 3:
                rec["tmp"] = eng.tmp[:g0.numel()].view(g0.shape).clone()
            assert i not in self.cap
            self.cap[i] = rec


def _route(eng, op):
    if op["cin"] == 3:
        return "small"
    if eng._implicit(op):
        return "implicit"
    if op["kh"] == 1 and op["kw"] == 1 and op["stride"] == 1:
        return "1x1"
    return "im2col"


@pytest.mark.parametrize("case", sorted(CASES))
def test_irv2_train_step_op_by_op_teacher_forced(case, monkeypatch):
    from spnet_b200 import arch
    from spnet_b200.engine import InceptionResNetV2SPNetEngine
    cfg = CASES[case]
    t0 = time.time()
    H, W, B = 260, 330, 4
    X, Y = frames(B, 7000)
    X = X[:, 62:322, 91:421, :].copy()   # the 260x330 window of the bf16 parity case
    w = perturbed_weights(xt.irv2_spnet_spec, H, W, 131)
    monkeypatch.setenv("SPNET_B200_POISON", "1")
    eng = InceptionResNetV2SPNetEngine(H, W, B, dtype=cfg["dtype"], weights=w, dropout_rate=0.0,
                                       deterministic=cfg["deterministic"])
    prog = eng.prog
    n_impl = sum(1 for op in prog.ops if op["kind"] == "conv_bn" and eng._implicit(op))
    assert n_impl == cfg["implicit"], (case, n_impl)
    kinds = [op["kind"] for op in prog.ops]
    assert {k: kinds.count(k) for k in set(kinds)} == {"conv_bn": 204, "concat": 43, "conv_bias": 40, "residual": 40,
                                                       "maxpool": 4, "avgpool": 1}
    lowp = eng.lowp
    tap = _Tap(prog.ops, eng)
    prog.ops = tap
    bncap = {}
    orig_sums, orig_bwd = eng._bn_bwd_sums, eng._bn_bwd

    def sums(g, z, bn, act=None):
        orig_sums(g, z, bn, act=act)
        assert bn.name not in bncap
        bncap[bn.name] = {"g_masked": g.clone()}

    def bwd(g, z, bn, rows, out=None):
        dz = orig_bwd(g, z, bn, rows, out=out)
        bncap[bn.name]["dz"] = dz.clone()
        return dz
    eng._bn_bwd_sums, eng._bn_bwd = sums, bwd
    eng.load_batch(X, Y)
    # eager step, stopped before Adam: the weights stay those the step used
    eng.grad_hook = lambda e: setattr(e, "skip_default_optimizer", True)
    eng.train_step(lr=1e-5)
    torch.cuda.synchronize()
    t_step = time.time()
    assert len(tap.cap) == len(prog.ops)

    rep, bad, checked = {}, [], set()

    def check(name, got, ref64, scale64):
        """bf16: at most 1 bf16 ulp beyond 1e-5 x sum|terms|, on under 2 % of the elements; fp32: within
        1e-5 x sum|terms|."""
        got = got.reshape(ref64.shape)
        if got.dtype == torch.bfloat16:
            ref = ref64.to(torch.bfloat16)
            ulp = torch.pow(2.0, torch.floor(torch.log2(ref.double().abs().clamp_min(1e-30))) - 7)
            excess = ((got.double() - ref.double()).abs() - 1e-5 * scale64) / ulp
            frac = float((got != ref).double().mean())
            worst = float(excess.max())
            rep[name] = {"mismatch_fraction": frac, "max_ulps": max(worst, 0.0)}
            if not (worst <= 1.0 + 1e-9 and frac < 2e-2):
                bad.append((name, frac, worst))
        else:
            err = (got.double() - ref64).abs()
            q = float((err / (1e-5 * scale64).clamp_min(1e-300)).max())
            rep[name] = {"max_error_over_bound": q}
            if not q <= 1.0:
                bad.append((name, q))

    def exact(name, got, ref):
        ok = got.shape == ref.shape and torch.equal(got, ref)
        rep[name] = {"equal": ok}
        if not ok:
            bad.append((name, "not bit-exact"))

    def grad(key, ref64, scale64):
        checked.add(key)
        check(key, eng.g[key], ref64, scale64)

    def into(name, j, op, rec, contrib, cabs, stored=None):
        """Input j's gradient after the op: (0 if first else before) + contribution. stored: the contribution as the
        engine stored it before adding it (the temporary buffer), checked on its own first."""
        if stored is not None:
            check(name + "/contribution", stored, contrib, cabs)
            contrib, cabs = stored.double(), stored.double().abs()
        if op["first"][j]:
            check(name, rec["after"][j], contrib, cabs)
        else:
            b = rec["before"][j].double()
            check(name, rec["after"][j], b + contrib, b.abs() + cabs)

    def affine(bn, z, name):
        """bn.a / bn.b / bn.mean / bn.rstd against fp64 statistics of the stored z: within 2e-6 relative. In fp32 the
        variance comes from fp32 partial sums of z^2 (E[z^2] - mean^2), so there the bound is 2e-6 of its sum of
        |terms|: relative to the variance, scaled by (mean^2 + var) / (var + eps). (Measured on a B200, fp32: up to
        5.7e-6 relative on the 2x3 maps of the block8 layers, 24 rows per channel, against 5.3e-7 in bf16.)"""
        zd = z.double().reshape(-1, bn.C)
        mean, var = zd.mean(0), zd.var(0, unbiased=False)
        rstd = 1.0 / torch.sqrt(var + arch.BN_EPS)
        b = bn.beta.double() - mean * rstd        # scale=False: gamma = 1, a = rstd
        cond = (mean * mean + var) / (var + arch.BN_EPS) if not lowp else torch.ones_like(var)
        ea = float(((bn.a.double() - rstd).abs() / rstd / cond).max())
        er = float(((bn.rstd.double() - rstd).abs() / rstd / cond).max())
        # b = beta - mean * a: the mean is known to 2e-6 of |mean| + std, and std * a is about 1
        eb = float(((bn.b.double() - b).abs() / (bn.beta.double().abs() + (mean.abs() + var.sqrt()) * rstd) / cond).max())
        em = float(((bn.mean.double() - mean).abs() / (mean.abs() + var.sqrt() + 1e-12)).max())
        rep[name + "/affine"] = {"a_rel_max": ea, "b_rel_max": eb, "rstd_rel_max": er, "mean_rel_max": em}
        if not (ea < 2e-6 and eb < 2e-6 and er < 2e-6 and em < 2e-6):
            bad.append((name + "/affine", ea, eb, er, em))

    # ------------------------------------------------------------------ forward
    for op in prog.ops:
        kind, o = op["kind"], op["out"]
        xs = [eng.data[x.idx] for x in op["inputs"]]
        y = eng.data[o.idx]
        if kind == "conv_bn":
            name, bn, z = op["name"], op["bnrec"], op["z"]
            k = (eng.w if op["cin"] == 3 else eng.wl)[name + "/kernel"].double()
            geo = (op["stride"], op["pt"], op["pl"], o.h, o.w)
            x = _nchw(xs[0])
            check(name + "/z", z, _nhwc(_conv(x, k, *geo)), _nhwc(_conv(x.abs(), k.abs(), *geo)))
            affine(bn, z, name)
            az = z.double() * bn.a.double()
            ref = az + bn.b.double()
            check(name + "/y", y, torch.relu(ref) if op["act"] else ref, az.abs() + bn.b.double().abs())
        elif kind == "conv_bias":
            K = op["cin"]
            x2, W2 = xs[0].double().reshape(-1, K), eng.wl[op["name"] + "/kernel"].double().reshape(K, o.c)
            check(op["name"] + "/u", y.reshape(-1, o.c), x2 @ W2, x2.abs() @ W2.abs())
        elif kind == "maxpool":
            x = _nchw(xs[0])
            win = F.unfold(x, 3, stride=2).view(B, o.c, 9, o.h * o.w)
            mx, am = win.max(2)   # the first maximum in window order kh*3+kw
            tag = "maxpool_%dx%d" % (op["inputs"][0].h, op["inputs"][0].w)
            exact(tag + "/out", y, _nhwc(mx.view(B, o.c, o.h, o.w)).to(y.dtype))
            exact(tag + "/argmax", op["argmax"], _nhwc(am.view(B, o.c, o.h, o.w)).to(torch.uint8))
        elif kind == "avgpool":
            x = _nchw(xs[0])
            check("avgpool/out", y, _nhwc(F.avg_pool2d(x, 3, 1, 1, count_include_pad=False)),
                  _nhwc(F.avg_pool2d(x.abs(), 3, 1, 1, count_include_pad=False)))
        elif kind == "concat":
            off = 0
            for j, x in enumerate(xs):
                exact("concat_%d/slice%d" % (o.idx, j), y[..., off:off + x.shape[-1]].contiguous(), x)
                off += x.shape[-1]
        elif kind == "residual":
            s, bias = op["scale"], eng.w[op["bias_name"]].double()
            ud = xs[1].double() + bias
            ref = xs[0].double() + s * ud
            check(op["bias_name"].split("/")[0] + "/residual_out", y, torch.relu(ref) if op["relu"] else ref,
                  xs[0].double().abs() + s * (xs[1].double().abs() + bias.abs()))

    # ------------------------------------------------------------------ backward
    # the head's data gradient is the incoming gradient of conv_7b (the last op)
    gyl = eng.gyl.double()
    Wd = eng.wl["FinalOutput/kernel"].double()
    out = prog.output
    check("FinalOutput/input_grad", tap.cap[len(prog.ops) - 1]["gy"].reshape(B, -1), gyl @ Wd.T, gyl.abs() @ Wd.abs().T)
    # wiring: every contribution to an activation's gradient, in backward order, starts from what the previous one
    # left (first: from nothing), and the producer reads what the last one left
    contributors = {}
    for i in range(len(prog.ops) - 1, -1, -1):
        for j, x in enumerate(prog.ops[i]["inputs"]):
            contributors.setdefault(x.idx, []).append((i, j))
    for i, op in enumerate(prog.ops):
        o = op["out"]
        if o is out:
            continue
        chain = contributors[o.idx]
        assert [prog.ops[c]["first"][j] for c, j in chain] == [True] + [False] * (len(chain) - 1), o.idx
        for (c0, j0), (c1, j1) in zip(chain, chain[1:]):
            exact("act%d/handoff_%d_to_%d" % (o.idx, c0, c1), tap.cap[c1]["before"][j1], tap.cap[c0]["after"][j0])
        c, j = chain[-1]
        exact("act%d/incoming" % o.idx, tap.cap[i]["gy"], tap.cap[c]["after"][j])

    counts = {}
    for i, op in enumerate(prog.ops):
        kind, o, rec = op["kind"], op["out"], tap.cap[i]
        ins = op["inputs"]
        xs = [eng.data[x.idx] for x in ins]
        gy = rec["gy"]
        M = B * o.h * o.w
        counts[kind] = counts.get(kind, 0) + 1
        if kind == "conv_bn":
            name, bn, z = op["name"], op["bnrec"], op["z"]
            C = bn.C
            r = bncap[bn.name]
            assert op["act"]
            ref_mask = z.double() * bn.a.double() + bn.b.double() > 0
            exact(name + "/relu_mask", r["g_masked"], torch.where(ref_mask, gy, torch.zeros_like(gy)))
            zd, gd = z.double().reshape(-1, C), r["g_masked"].double().reshape(-1, C)
            mu, rs = bn.mean.double(), bn.rstd.double()
            sg, sgx = gd.sum(0), (gd * (zd - mu) * rs).sum(0)
            ag, agx = gd.abs().sum(0), (gd.abs() * (zd.abs() + mu.abs()) * rs).sum(0)
            grad(bn.name + "/beta", sg, ag)
            check(bn.name + "/c1", bn.c1, sg / M, ag / M)
            check(bn.name + "/c2", bn.c2, sgx / M, agx / M)
            a, c1, c2 = bn.a.double(), bn.c1.double(), bn.c2.double()
            check(name + "/dz", r["dz"].reshape(-1, C), a * (gd - c1 - (zd - mu) * rs * c2),
                  a.abs() * (gd.abs() + c1.abs() + (zd.abs() + mu.abs()) * rs * c2.abs()))
            dz = r["dz"].view(B, o.h, o.w, C)
            route = _route(eng, op)
            key = name + "/kernel"
            k = (eng.w if route == "small" else eng.wl)[key].double()
            geo = (op["stride"], op["pt"], op["pl"], o.h, o.w)
            x = _nchw(xs[0]).requires_grad_(True)
            kk = k.clone().requires_grad_(True)
            gx, gk = torch.autograd.grad(_conv(x, kk, *geo), (x, kk), _nchw(dz))
            xa = _nchw(xs[0]).abs().requires_grad_(True)
            ka = k.abs().requires_grad_(True)
            gxa, gka = torch.autograd.grad(_conv(xa, ka, *geo), (xa, ka), _nchw(dz).abs())
            grad(key, gk, gka)
            gx, gxa = _nhwc(gx), _nhwc(gxa)
            if route == "im2col":
                # column gradient (one GEMM), then col2im: its fold, added to the gradient there when not first
                kh, kw, cin = op["kh"], op["kw"], op["cin"]
                K = kh * kw * cin
                gcol = rec["gcol"].view(M, K)
                Wm, dz2 = eng.wl[key].double().reshape(K, C), dz.double().reshape(M, C)
                check(name + "/column_grad", gcol, dz2 @ Wm.T, dz2.abs() @ Wm.abs().T)
                h, wd = ins[0].h, ins[0].w
                pb, pr = (o.h - 1) * op["stride"] + kh - h - op["pt"], (o.w - 1) * op["stride"] + kw - wd - op["pl"]
                cols = gcol.double().view(B, o.h * o.w, kh * kw, cin).permute(0, 3, 2, 1).reshape(B, cin * kh * kw, -1)

                def fold(t):
                    f = F.fold(t, (h + op["pt"] + pb, wd + op["pl"] + pr), (kh, kw), stride=op["stride"])
                    return _nhwc(F.pad(f, (-op["pl"], -pr, -op["pt"], -pb)))
                into(name + "/input_grad", 0, op, rec, fold(cols), fold(cols.abs()))
            else:
                into(name + "/input_grad", 0, op, rec, gx, gxa, rec.get("tmp"))
        elif kind == "conv_bias":
            name, K = op["name"], op["cin"]
            g2 = gy.double().reshape(M, o.c)
            x2, W2 = xs[0].double().reshape(M, K), eng.wl[name + "/kernel"].double().reshape(K, o.c)
            grad(name + "/kernel", x2.T @ g2, x2.abs().T @ g2.abs())
            grad(name + "/bias", g2.sum(0), g2.abs().sum(0))
            into(name + "/input_grad", 0, op, rec, (g2 @ W2.T).view(xs[0].shape), (g2.abs() @ W2.abs().T).view(xs[0].shape),
                 rec.get("tmp"))
        elif kind == "maxpool":
            xi = ins[0]
            tag = "maxpool_%dx%d" % (xi.h, xi.w)
            win = F.unfold(_nchw(xs[0]), 3, stride=2).view(B, o.c, 9, M // B)
            hot = F.one_hot(win.argmax(2), 9).permute(0, 1, 3, 2).double()      # [B, C, 9, L]
            g = _nchw(gy).reshape(B, o.c, 1, M // B)

            def scatter(t):
                return _nhwc(F.fold((hot * t).reshape(B, o.c * 9, -1), (xi.h, xi.w), 3, stride=2))
            into(tag + "/input_grad", 0, op, rec, scatter(g), scatter(g.abs()), rec.get("tmp"))
            # rows / columns no window covers (62 -> 30, 28 -> 13 leave the last one) keep what was there
            keep = rec["before"][0] if not op["first"][0] else torch.zeros_like(rec["after"][0])
            if (xi.h - 3) % 2:
                exact(tag + "/uncovered_row", rec["after"][0][:, -1], keep[:, -1])
            if (xi.w - 3) % 2:
                exact(tag + "/uncovered_col", rec["after"][0][:, :, -1], keep[:, :, -1])
        elif kind == "avgpool":
            g = _nchw(gy)
            x = torch.zeros_like(g, requires_grad=True)
            pooled = F.avg_pool2d(x, 3, 1, 1, count_include_pad=False)
            gin, = torch.autograd.grad(pooled, x, g, retain_graph=True)
            gabs, = torch.autograd.grad(pooled, x, g.abs())
            into("avgpool/input_grad", 0, op, rec, _nhwc(gin), _nhwc(gabs))
        elif kind == "concat":
            off = 0
            for j, x in enumerate(ins):
                sl = gy[..., off:off + x.c].contiguous()
                if op["first"][j]:
                    exact("concat_%d/input_grad%d" % (o.idx, j), rec["after"][j], sl)
                else:
                    into("concat_%d/input_grad%d" % (o.idx, j), j, op, rec, sl.double(), sl.double().abs())
                off += x.c
        elif kind == "residual":
            tag = op["bias_name"].split("/")[0] + "/residual"
            gm = torch.where(eng.data[o.idx] > 0, gy, torch.zeros_like(gy)) if op["relu"] else gy
            if op["first"][0]:
                exact(tag + "/x_grad", rec["after"][0], gm)
            else:
                into(tag + "/x_grad", 0, op, rec, gm.double(), gm.double().abs())
            assert op["first"][1]   # the 1x1 "up" convolution's output is read by its residual only
            check(tag + "/up_grad", rec["after"][1], op["scale"] * gm.double(), op["scale"] * gm.double().abs())
    assert counts == {"conv_bn": 204, "concat": 43, "conv_bias": 40, "residual": 40, "maxpool": 4, "avgpool": 1}

    rep["summary"] = {"checks": len(rep), "failed": len(bad), "implicit_convolutions": n_impl,
                      "seconds_step": t_step - t0, "seconds_reference": time.time() - t_step,
                      "worst_mismatch_fraction": max(v.get("mismatch_fraction", 0.0) for v in rep.values()),
                      "worst_ulps": max(v.get("max_ulps", 0.0) for v in rep.values()),
                      "worst_fp32_error_over_bound": max(v.get("max_error_over_bound", 0.0) for v in rep.values())}
    record("irv2_layer_by_layer_" + case, rep)
    assert set(eng.g) - checked == EXCLUDED, (sorted(set(eng.g) - checked - EXCLUDED), sorted(EXCLUDED - set(eng.g)))
    assert checked <= set(eng.g)
    assert not bad, bad[:20]
