"""Drop-in surface of the reference's spnet/models.py for the hot path (SURVEY.md §8b):
setup_model(...) -> (model, serial_model), custom_loss, my_loss, SelectiveSigmoid,
unfreeze_model — same names, argument meaning and error behaviour — on top of the B200 engine
(spnet_b200/engine.py -> libspnet_b200.so). `model` is a small Keras-Model look-alike exposing
what the reference's callers use: fit / predict / compile / save_weights / load_weights / save /
get_weights / set_weights / layers / optimizer.lr / trainable_weights / non_trainable_weights /
losses, and the Keras callback protocol.

There is no CPU path: arrays come in and go out as numpy float32 (NHWC), everything in between
runs in the CUDA kernels.
"""
import os
import sys
import time
from collections import OrderedDict
from os.path import isfile

import numpy as np

from . import arch
from . import config as cf
from . import multi_gpu

# Loss constants (spnet/models.py:557-562); the kernels carry the same values.
lambda_center = 2.0
lambda_size = 1.0
lambda_angle = 3.0
lambda_noobj = 0.3
lambda_class = 5.0
logeps = 1e-10


def _torch():
    import torch
    return torch


def _dev_f32(a):
    torch = _torch()
    if torch.is_tensor(a):
        return a.to("cuda", torch.float32).contiguous()
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


def _loss6(y_true, y_pred, sel_sigmoid=False):
    from . import ops
    yt, yp = _dev_f32(y_true), _dev_f32(y_pred)
    if yt.shape != yp.shape or yt.dim() != 2:
        raise ValueError("y_true and y_pred must both be (batch, ncols); got %s and %s" % (tuple(yt.shape), tuple(yp.shape)))
    return ops.yolo_ellipse_loss(yt, yp, hybrid=(cf.loss_type != "same"), sel_sigmoid=sel_sigmoid).cpu().numpy()


def custom_loss(y_true, y_pred):
    """MSE-like YOLO-ellipse loss with the angle term weighted by (a-b)^2 (spnet/models.py:564-589);
    cf.loss_type is read at call time. Returns the scalar batch mean."""
    return float(_loss6(y_true, y_pred)[0])


def my_loss(y_true, y_pred, verbosity=0):
    """Diagnostic twin (spnet/models.py:594-633): (total, [center, size, angle, noobj, class])."""
    out = _loss6(y_true, y_pred)
    losses = out[1:6].astype(np.float64)
    if verbosity > 0:
        print("    my_loss: [   center,        size,      angle,     noobj,      class ].  loss_type =", cf.loss_type)
        print("    losses =", losses, ", ind_max =", int(np.argmax(losses)))
    return float(np.sum(losses)), losses


class SelectiveSigmoid:
    """Sigmoid on the strided columns start:end:skip, identity elsewhere (spnet/models.py:277-298).
    Callable on (batch, ncols) arrays; `grad` gives the backward."""

    def __init__(self, **kwargs):
        self.start = kwargs.get("start", cf.ind_noobj)
        self.end = kwargs.get("end", None)
        self.skip = kwargs.get("skip", cf.vars_per_pred)
        self.sigmoid_stretch = 1
        self.name = kwargs.get("name", "selective_sigmoid")

    def build(self, input_shape):
        self.indices = np.zeros(input_shape[-1])
        self.indices[self.start:self.end:self.skip] = 1

    def _bounds(self, n):
        # python-slice semantics of start:end:skip on n columns -> explicit [start, end)
        start, end, _ = slice(self.start, self.end, self.skip).indices(n)
        return start, end

    def call(self, x):
        from . import ops
        xd = _dev_f32(x)
        s, e = self._bounds(xd.shape[1])
        return ops.selective_sigmoid_fwd(xd, s, e, self.skip).cpu().numpy()

    __call__ = call

    def grad(self, y, dy):
        from . import ops
        yd, gd = _dev_f32(y), _dev_f32(dy)
        s, e = self._bounds(yd.shape[1])
        return ops.selective_sigmoid_bwd(yd, gd, s, e, self.skip).cpu().numpy()

    def compute_output_shape(self, input_shape):
        return input_shape


def selective_activation(x, start=1, end=-1, skip_every=6):
    """selective_activation.py:6-9 (the snippet's own defaults)."""
    return SelectiveSigmoid(start=start, end=end, skip=skip_every)(x)


# ------------------------------------------------------------------------------------------------
class Adam:
    """Hyper-parameter holder with the Keras 2.1.3 defaults; `lr` is read before every step
    (OneCycleScheduler overwrites it per batch, spnet/callbacks.py:396-399)."""

    def __init__(self, lr=0.001, beta_1=0.9, beta_2=0.999, epsilon=1e-7, decay=0.0):
        self.lr, self.beta_1, self.beta_2, self.epsilon, self.decay = lr, beta_1, beta_2, epsilon, decay


class _Layer:
    def __init__(self, model, name, keys):
        self._model, self.name, self._keys, self.trainable = model, name, keys, True

    def get_weights(self):
        w = self._model._weights_dict()
        return [w[k] for k in self._keys]

    def count_params(self):
        return int(sum(np.prod(self._model._shape[k]) for k in self._keys))


class History:
    def __init__(self):
        self.history = {}
        self.epoch = []


class SPNetModel:
    """Xception-SPNet behind a Keras-Model-like interface."""

    def __init__(self, input_shape, Y0size=576, quick_setup=False, weights=None, seed=1, name="spnet",
                 backbone="Xception"):
        H, W = int(input_shape[0]), int(input_shape[1])
        self.backbone = backbone
        if len(input_shape) > 2 and int(input_shape[2]) != 1:
            raise ValueError("Xception-SPNet takes single-channel (grayscale) input; got shape %s" % (tuple(input_shape),))
        if Y0size % cf.vars_per_pred != 0:
            raise ValueError("Y0size (=" + str(Y0size) + ") must be a multiple of cf.vars_per_pred (=" + str(cf.vars_per_pred) + ")")
        self.name = name
        self.input_shape = (None, H, W, 1)
        self.output_shape = (None, Y0size)
        self.H, self.W, self.Y0size = H, W, Y0size
        from . import irv2
        self.spec = {"MobileNet": arch.mobilenet_param_spec, "InceptionResNetV2": irv2.param_spec}.get(backbone, arch.param_spec)(H, W, Y0size)
        self._shape = OrderedDict((k, s) for k, s, _, _ in self.spec)
        self._host_weights = weights if weights is not None else arch.glorot_init(self.spec, seed)
        self.use_l2 = not quick_setup          # add_regularization is skipped by quick_setup (spnet/models.py:398-399)
        self.losses = [] if quick_setup else [k for k, _, _, r in self.spec if r]
        self.optimizer = None
        self.loss = None
        self.parallel = False
        self.serial_model = self
        self.stop_training = False
        self.frozen_layers = set()
        self._engines = {}
        self._master = None       # engine holding the newest weights
        self._version = 0
        by_layer = OrderedDict()
        for k, _, _, _ in self.spec:
            by_layer.setdefault(k.split("/")[0], []).append(k)
        self.layers = [_Layer(self, n, ks) for n, ks in by_layer.items()]

    # ---- weights ------------------------------------------------------------------------------
    @property
    def trainable_weights(self):
        return [k for k, _, t, _ in self.spec if t and k.split("/")[0] not in self.frozen_layers]

    @property
    def non_trainable_weights(self):
        return [k for k, _, t, _ in self.spec if not t or k.split("/")[0] in self.frozen_layers]

    def count_params(self):
        return arch.count_params(self.spec)[0]

    def _count_trainable(self):
        """(trainable, non-trainable) parameter counts as Keras reports them: weights of frozen layers count as
        non-trainable (spnet/models.py:415-423)."""
        tr = sum(int(np.prod(self._shape[k])) for k in self.trainable_weights)
        return tr, arch.count_params(self.spec)[0] - tr

    def _weights_dict(self):
        if self._master is not None:
            self._host_weights = self._master.get_weights()
        return self._host_weights

    def get_weights(self):
        w = self._weights_dict()
        return [w[k] for k, _, _, _ in self.spec]

    def set_weights(self, weights):
        if len(weights) != len(self.spec):
            raise ValueError("set_weights: expected %d arrays, got %d" % (len(self.spec), len(weights)))
        new = OrderedDict()
        for (k, s, _, _), a in zip(self.spec, weights):
            a = np.asarray(a, dtype=np.float32)
            if tuple(a.shape) != tuple(s):
                raise ValueError("set_weights: %s has shape %s, expected %s" % (k, a.shape, s))
            new[k] = a
        self._load_dict(new)

    def _load_dict(self, d):
        self._host_weights = OrderedDict((k, np.asarray(d[k], np.float32)) for k, _, _, _ in self.spec)
        self._master = None
        self._version += 1
        for eng in self._engines.values():
            eng.set_weights(self._host_weights)
            eng._version = self._version

    # ---- checkpoint files -------------------------------------------------------------------------
    # The reference's checkpoints are Keras HDF5 files (weights.hdf5 / spnet.model / full_model.h5: spnet/models.py:
    # 475-485, spnet/callbacks.py:35-41, train_spnet.py:145-150). Files whose name ends in .h5 / .hdf5 / .model are
    # written in that format (spnet_b200/hdf5_min.py: h5py is not in this image); any other name gets an .npz container
    # keyed by the Keras weight names. Reading sniffs the file's magic bytes, whatever its name.
    def _keras_layers(self):
        by_layer = OrderedDict()
        for k, _, _, _ in self.spec:
            by_layer.setdefault(k.split("/")[0], []).append(k)
        order = {"Xception": arch.xception_keras_layers, "MobileNet": arch.mobilenet_keras_layers}.get(self.backbone)
        names = (order() + ["flatten_1", "FinalOutput"]) if order else list(by_layer)
        names += [n for n in by_layer if n not in names]
        return [(n, by_layer.get(n, [])) for n in names]

    @staticmethod
    def _is_hdf5_name(filepath):
        return str(filepath).lower().endswith((".h5", ".hdf5", ".model"))

    def save_weights(self, filepath):
        w = self._weights_dict()
        if self._is_hdf5_name(filepath):
            from . import hdf5_min
            hdf5_min.write_keras_weights(filepath, self._keras_layers(), w)
            return
        with open(filepath, "wb") as f:
            np.savez(f, **{k.replace("/", "::"): v for k, v in w.items()})

    @staticmethod
    def _read_weight_file(filepath):
        """-> ({key: array}, config dict or None) from an HDF5 (Keras) or .npz file."""
        with open(filepath, "rb") as f:
            magic = f.read(8)
        if magic.startswith(b"\x89HDF"):
            import json
            from . import hdf5_min
            d, attrs = hdf5_min.read_keras_weights(filepath)
            cfg = attrs.get("model_config")
            if cfg is not None:
                cfg = json.loads(cfg.decode("utf8") if isinstance(cfg, bytes) else cfg)
            return d, cfg
        z = np.load(filepath)
        d = {k.replace("::", "/"): z[k] for k in z.files if not k.startswith("__")}
        cfg = None
        if "__config__" in z.files:
            H, W, Y0, use_l2 = (int(v) for v in z["__config__"])
            cfg = {"spnet_b200": {"H": H, "W": W, "Y0size": Y0, "use_l2": bool(use_l2),
                                  "backbone": str(z["__backbone__"]) if "__backbone__" in z.files else "Xception",
                                  "loss_type": str(z["__loss_type__"]) if "__loss_type__" in z.files else None}}
        return d, cfg

    def load_weights(self, filepath, by_name=False):
        d, _ = self._read_weight_file(filepath)
        missing = [k for k, _, _, _ in self.spec if k not in d]
        if missing and not by_name:
            raise ValueError("load_weights: %d tensors missing from %s (first: %s)" % (len(missing), filepath, missing[0]))
        for k, shp, _, _ in self.spec:
            if k in d and tuple(d[k].shape) != tuple(shp):
                raise ValueError("load_weights: %s has shape %s in %s, the model expects %s" % (k, tuple(d[k].shape), filepath, tuple(shp)))
        cur = self._weights_dict()
        self._load_dict({k: d.get(k, cur[k]) for k, _, _, _ in self.spec})

    def save(self, filepath):
        """Full-model save: weights + architecture config (+ Adam state is not stored by the reference's resume path either:
        spnet/models.py:475-485 reloads weights only)."""
        w = self._weights_dict()
        cfg = {"H": self.H, "W": self.W, "Y0size": self.Y0size, "use_l2": bool(self.use_l2), "backbone": self.backbone,
               "loss_type": cf.loss_type}
        if self._is_hdf5_name(filepath):
            import json
            from . import hdf5_min
            hdf5_min.write_keras_weights(filepath, self._keras_layers(), w, full_model_config=json.dumps({"spnet_b200": cfg}))
            return
        with open(filepath, "wb") as f:
            np.savez(f, __config__=np.array([self.H, self.W, self.Y0size, int(self.use_l2)]),
                     __backbone__=np.array(self.backbone), __loss_type__=np.array(cf.loss_type),
                     **{k.replace("/", "::"): v for k, v in w.items()})

    def summary(self):
        tot, tr, nt = arch.count_params(self.spec)
        print("%s-SPNet  input (%d,%d,1) -> %d outputs; %d layers with weights" % (self.backbone, self.H, self.W, self.Y0size, len(self.layers)))
        print("Total params: {:,}\nTrainable params: {:,}\nNon-trainable params: {:,}".format(tot, tr, nt))

    # ---- engines ------------------------------------------------------------------------------
    def compile(self, loss=None, optimizer=None):
        self.loss = loss if loss is not None else custom_loss
        self.optimizer = optimizer if optimizer is not None else Adam(lr=0.00001)

    def _engine(self, batch, training):
        from .engine import InceptionResNetV2SPNetEngine, MobileNetSPNetEngine, XceptionSPNetEngine
        Engine = {"MobileNet": MobileNetSPNetEngine, "InceptionResNetV2": InceptionResNetV2SPNetEngine}.get(self.backbone, XceptionSPNetEngine)
        key = (batch, training)
        eng = self._engines.get(key)
        if eng is None:
            torch = _torch()
            dev = "cuda:%d" % torch.cuda.current_device()
            eng = Engine(self.H, self.W, batch, n_out=self.Y0size, dtype=cf.compute_dtype, device=dev,
                                      weights=self._weights_dict(), loss_type=cf.loss_type, use_l2=self.use_l2,
                                      training=training)
            eng._version = self._version
            self._engines[key] = eng
        elif eng._version != self._version:
            if self._master is not None and self._master is not eng:
                eng.params.copy_(self._master.params)
                eng.nontrainable.copy_(self._master.nontrainable)
                eng.refresh_lowp()
            eng._version = self._version
        eng.loss_type = cf.loss_type
        if training and eng.frozen_layers != frozenset(self.frozen_layers):
            eng.set_frozen(self.frozen_layers)
        return eng

    # ---- inference ----------------------------------------------------------------------------
    def predict(self, X, batch_size=32, verbose=0, resize=False):
        """Keras Model.predict (reference call site predict_spnet.py:85): inference-mode forward over X in batches.
        X: numpy / torch array (n, H, W, 1), float32 already normalised, or uint8 raw pixel values (normalised on the
        device, (v/255 - 0.5)*2 of spnet/utils.py:340-342 bit for bit; a quarter of the host->device bytes).
        resize=True: X holds uint8 frames (n, h, w, 1) as decoded (utils.build_X(..., defer_resize=True)), on the host
        or the device; each is LANCZOS-resized to the model's (H, W) on the device, the bytes of the host's PIL resize
        (:325-349), so the result is predict() of the frames utils.build_X(force_dim=...) returns.
        The forward pass of a batch is one CUDA-graph replay; batch k+1 travels host -> device on a copy stream
        (from X itself when X is a pinned torch tensor, through a pinned staging pair filled by a helper thread
        otherwise) while batch k computes, and the results come back through one pinned buffer."""
        torch = _torch()
        if resize and (X.dtype != torch.uint8 if torch.is_tensor(X) else np.asarray(X).dtype != np.uint8):
            raise ValueError("predict(resize=True) takes uint8 frames as decoded, got %s" % (X.dtype,))
        if torch.is_tensor(X):
            Xt = X if X.dtype in (torch.uint8, torch.float32) else X.float()
        else:
            Xn = np.asarray(X)
            if Xn.dtype not in (np.uint8, np.float32):
                Xn = Xn.astype(np.float32)
            Xt = torch.from_numpy(np.ascontiguousarray(Xn))
        n = Xt.shape[0]
        if Xt.dtype == torch.uint8 and not resize and tuple(Xt.shape[1:3]) != (self.H, self.W):
            raise ValueError("predict: %s frames for a %dx%d model (resize=True resizes them on the device)"
                             % ("x".join(map(str, Xt.shape[1:3])), self.H, self.W))
        out = np.empty((n, self.Y0size), np.float32)
        if n == 0:
            return out
        bs = min(batch_size, n)
        eng = self._engine(bs, False)
        nb = -(-n // bs)
        frame = tuple(Xt.shape[1:])
        res = torch.empty((nb * bs, self.Y0size), dtype=torch.float32).pin_memory()
        if os.environ.get("SPNET_B200_NO_GRAPH") is None and getattr(eng, "fwd_graph", None) is None:
            eng.x0.zero_()
            eng.prepare_inference()
            eng.forward(training=False)   # eager warm-up (sizes every lazily allocated buffer), then capture
            torch.cuda.synchronize()
            eng.capture_forward()
        if Xt.is_cuda:
            for j in range(nb):
                m = min(bs, n - j * bs)
                if m < bs:
                    eng.x0.zero_()
                src = Xt[j * bs:j * bs + m]
                if src.dtype == torch.uint8:
                    eng.frames_to_x0(src.contiguous())
                else:
                    eng.x0[:m].copy_(src.reshape((m,) + tuple(eng.x0.shape[1:])))
                res[j * bs:(j + 1) * bs].copy_(eng.infer(), non_blocking=True)
        else:
            direct = Xt.is_pinned() and Xt.is_contiguous()
            pin = None if direct else [torch.empty((bs,) + frame, dtype=Xt.dtype).pin_memory() for _ in range(2)]
            pin_free = [None, None]

            def fill(j):
                """Host side of batch j: a full pinned batch to copy from (X itself, or a staging buffer)."""
                m = min(bs, n - j * bs)
                if direct and m == bs:
                    return Xt[j * bs:(j + 1) * bs]
                k = j % 2
                if pin is None:
                    return torch.cat([Xt[j * bs:j * bs + m], torch.zeros((bs - m,) + frame, dtype=Xt.dtype)]).pin_memory()
                if pin_free[k] is not None:
                    pin_free[k].synchronize()  # the H2D copy that last read this staging buffer is done
                pin[k][:m].copy_(Xt[j * bs:j * bs + m])
                if m < bs:
                    pin[k][m:].zero_()
                return pin[k]

            from concurrent.futures import ThreadPoolExecutor
            with ThreadPoolExecutor(max_workers=1) as pool:  # staging memcpy of batch j+1 overlaps the launches of batch j
                nxt = pool.submit(fill, 0)
                for j in range(nb):
                    buf = nxt.result()
                    pin_free[j % 2] = eng.prefetch_batch(buf)
                    if j + 1 < nb:
                        nxt = pool.submit(fill, j + 1)
                    eng.take_prefetched()
                    res[j * bs:(j + 1) * bs].copy_(eng.infer(), non_blocking=True)
        torch.cuda.synchronize()
        out[:] = res.numpy()[:n]
        return out

    def evaluate(self, X, Y, batch_size=32, verbose=0):
        yp = self.predict(X, batch_size=batch_size)
        return custom_loss(np.asarray(Y, np.float32), yp) + self._l2_value()

    def _l2_value(self):
        if not self.use_l2:
            return 0.0
        w = self._weights_dict()
        return float(sum(arch.L2_COEF * np.sum(w[k].astype(np.float64) ** 2) for k in self.losses))

    # ---- training -----------------------------------------------------------------------------
    def fit(self, X, Y, batch_size=32, epochs=1, shuffle=True, verbose=1, validation_data=None, callbacks=None,
            initial_epoch=0):
        torch = _torch()
        if self.optimizer is None:
            raise RuntimeError("You must compile a model before training/testing. Use `model.compile(optimizer, loss)`.")
        # Device-resident input path: X (and optionally Y) given as CUDA tensors stay in HBM for the whole fit;
        # batches are gathered on the device (no host staging, no H2D copy) and callbacks.AugmentOnTheFly
        # rewrites X there once per epoch. The host path below is the reference's numpy interface.
        on_device = torch.is_tensor(X) and X.is_cuda
        if on_device:
            X = X.float().contiguous() if X.dtype != torch.float32 or not X.is_contiguous() else X
            Y = (Y if torch.is_tensor(Y) else torch.from_numpy(np.asarray(Y, dtype=np.float32))).to(X.device).float().contiguous()
        else:
            # uint8 X = raw frames (pixel values 0..255, utils.build_X(raw_u8=True)): a quarter of the host gather and
            # PCIe traffic, normalised on the device bit-exactly; anything else is the reference's normalised float32
            X = np.asarray(X) if getattr(X, "dtype", None) == np.uint8 else np.asarray(X, dtype=np.float32)
            Y = np.asarray(Y, dtype=np.float32)
        if X.shape[0] != Y.shape[0]:
            raise ValueError("Input arrays should have the same number of samples as target arrays. Found %d input samples and %d target samples." % (X.shape[0], Y.shape[0]))
        if Y.shape[1] != self.Y0size:
            raise ValueError("Error when checking target: expected FinalOutput to have shape (%d,) but got array with shape (%d,)" % (self.Y0size, Y.shape[1]))
        rank, world = multi_gpu.world() if self.parallel else (0, 1)
        local_bs = batch_size // world
        n = X.shape[0]
        steps = n // batch_size
        if steps == 0:
            raise ValueError("fit: %d samples are fewer than one batch of %d" % (n, batch_size))
        if steps * batch_size != n and verbose:
            print("fit: dropping the trailing %d samples (static batch of %d)" % (n - steps * batch_size, batch_size))
        eng = self._engine(local_bs, True)
        if world > 1 and eng.grad_hook is None:
            multi_gpu.attach_data_parallel(eng)
        self._master = eng
        callbacks = list(callbacks or [])
        hist = History()
        for cb in callbacks + [hist]:
            if hasattr(cb, "set_model"):
                cb.set_model(self)
            else:
                cb.model = self
            if hasattr(cb, "set_params"):
                cb.set_params({"batch_size": batch_size, "epochs": epochs, "steps": steps, "samples": n, "verbose": verbose})
        self.stop_training = False
        _call(callbacks, "on_train_begin", {})
        if not on_device:
            xpin = [torch.empty((local_bs,) + X.shape[1:], dtype=torch.uint8 if X.dtype == np.uint8 else torch.float32).pin_memory()
                    for _ in range(2)]
            ypin = [torch.empty((local_bs, self.Y0size), dtype=torch.float32).pin_memory() for _ in range(2)]
            xpin_np, ypin_np = [t.numpy() for t in xpin], [t.numpy() for t in ypin]
            # the batch gather (50 MB of float32 frames per step at batch 64) runs on a few host threads straight into
            # the pinned staging buffer: one copy, off the critical path of the step it overlaps
            from concurrent.futures import ThreadPoolExecutor
            nthr = max(1, min(8, (os.cpu_count() or 2) // 2, local_bs))
            pool = ThreadPoolExecutor(nthr)
        loss_acc = torch.zeros(6, device=eng.device)
        rng = np.random.RandomState(np.random.randint(0, 2 ** 31 - 1))
        captured = False
        for epoch in range(initial_epoch, epochs):
            _call(callbacks, "on_epoch_begin", epoch, {})
            t0 = time.time()
            order = rng.permutation(n) if shuffle else np.arange(n)
            loss_acc.zero_()
            def stage(b):
                """Gather batch b into pinned buffer b % 2 and start its H2D copy on the copy stream."""
                idx = order[b * batch_size:(b + 1) * batch_size]
                lo, hi = multi_gpu.batch_slice(batch_size, rank, world)
                idx = np.sort(idx[lo:hi]) if not shuffle else idx[lo:hi]
                k = b % 2
                if pin_free[k] is not None:
                    pin_free[k].synchronize()  # the H2D copy that last read this pinned buffer is done
                cuts = np.linspace(0, len(idx), nthr + 1).astype(int)
                # mode 'clip': numpy writes straight into `out` (the default 'raise' gathers into a temporary first)
                futs = [pool.submit(np.take, X, idx[a:b_], 0, xpin_np[k][a:b_], "clip") for a, b_ in zip(cuts[:-1], cuts[1:]) if b_ > a]
                np.take(Y, idx, axis=0, out=ypin_np[k], mode="clip")
                for f in futs:
                    f.result()
                pin_free[k] = eng.prefetch_batch(xpin[k], ypin[k])

            def gather_on_device(b):
                idx = order[b * batch_size:(b + 1) * batch_size]
                lo, hi = multi_gpu.batch_slice(batch_size, rank, world)
                idx_t = torch.from_numpy(np.ascontiguousarray(idx[lo:hi])).to(X.device, non_blocking=True)
                torch.index_select(X, 0, idx_t, out=eng.x0)
                torch.index_select(Y, 0, idx_t, out=eng.y_true)

            pin_free = [None, None]
            if not on_device:
                stage(0)
            for b in range(steps):
                _call(callbacks, "on_batch_begin", b, {"batch": b, "size": batch_size})
                if on_device:
                    gather_on_device(b)
                else:
                    eng.take_prefetched()
                if not on_device and b + 1 < steps:
                    stage(b + 1)  # host gather + H2D of the next batch overlap this step's kernels
                loss6 = eng.train_step(float(self.optimizer.lr))
                loss_acc += loss6
                if not captured and eng.graph is None and b == 0 and epoch == initial_epoch and os.environ.get("SPNET_B200_NO_GRAPH") is None:
                    torch.cuda.synchronize()
                    eng.capture()
                    captured = True
                _call(callbacks, "on_batch_end", b, {"batch": b, "size": batch_size})
            self._version += 1
            eng._version = self._version
            torch.cuda.synchronize()
            lv = (loss_acc / steps).cpu().numpy()
            logs = {"loss": float(lv[0]) + float(eng.l2_out[0])}
            if validation_data is not None:
                Xv, Yv = validation_data[0], validation_data[1]
                logs["val_loss"] = custom_loss(Yv, self.predict(Xv, batch_size=batch_size)) + float(eng.l2_out[0])
            if verbose:
                dt = time.time() - t0
                print("Epoch %d/%d - %ds %dms/step - " % (epoch + 1, epochs, dt, 1e3 * dt / max(n, 1)) +
                      " - ".join("%s: %.4f" % kv for kv in logs.items()))
            hist.epoch.append(epoch)
            for kk, vv in logs.items():
                hist.history.setdefault(kk, []).append(vv)
            _call(callbacks, "on_epoch_end", epoch, logs)
            if self.stop_training:
                break
        if not on_device:
            pool.shutdown(wait=False)
        _call(callbacks, "on_train_end", {})
        return hist


def _call(callbacks, hook, *args):
    for cb in callbacks:
        fn = getattr(cb, hook, None)
        if fn is not None:
            fn(*args)


# ------------------------------------------------------------------------------------------------
def str_to_class(name):
    return getattr(sys.modules[__name__], name)


def Xception(weights=None, include_top=False, input_tensor=None, input_shape=None):
    """Backbone plug-in point resolved by name from cf.basemodel (spnet/models.py:43-44,357-359)."""
    return "Xception"


def MobileNet(weights=None, include_top=False, input_tensor=None, input_shape=None):
    """keras.applications.mobilenet.MobileNet plug-in (spnet/models.py:20,349-355). The reference asks
    for weights='imagenet', which Keras 2.1.3 only provides for square 128-224 inputs; here the backbone
    is always built with the supplied / Keras-default-initialised weights."""
    return "MobileNet"


def InceptionResNetV2(weights=None, include_top=False, input_tensor=None, input_shape=None):
    """keras.applications.inception_resnet_v2.InceptionResNetV2 plug-in (spnet/models.py:18, built through
    the generic backbone branch :357-359 with weights=None)."""
    return "InceptionResNetV2"


def create_model_functional(X, Y0size=576, freeze_fac=0.75, quick_setup=False):
    """spnet/models.py:302-424. Stem -> cf.basemodel -> Flatten -> Dense(Y0size,'FinalOutput')."""
    print("Using functional API model, cf.basemodel =", cf.basemodel)
    print("X[0].shape = ", X[0].shape)
    if not hasattr(sys.modules[__name__], cf.basemodel):
        raise AttributeError("module 'spnet.models' has no attribute '%s'" % cf.basemodel)
    if cf.basemodel not in ("Xception", "MobileNet", "InceptionResNetV2"):
        raise NotImplementedError("cf.basemodel = %r: the Xception (reference default, spnet/config.py:52), MobileNet and "
                                  "InceptionResNetV2 backbones are built" % cf.basemodel)
    model = SPNetModel(X[0].shape, Y0size=Y0size, quick_setup=quick_setup, backbone=cf.basemodel)
    # base_model.layers[:int(num_layers * freeze_fac)].trainable = False (spnet/models.py:361-372), on the exact Keras
    # layer order for Xception (144 layers, paper/run_logs/log_DatasetA_*.txt:95) and MobileNet (94)
    names, freeze_layers, num_layers = arch.frozen_layer_names(cf.basemodel, freeze_fac, model.spec)
    print("Freezing ", freeze_layers, "/", num_layers, " layers of base_model")
    model.frozen_layers = set(names)
    if not quick_setup:
        tr, nt = model._count_trainable()
        print("After adding l2 regularization, model.losses =", model.losses)
        print("create_model_functional: Total params: {:,}".format(tr + nt))
        print("create_model_functional: Trainable params: {:,}".format(tr))
        print("create_model_functional: Non-trainable params: {:,}".format(nt))
    return model


def setup_model(X, Y0size=576, try_checkpoint=True, no_cp_fatal=False, weights_file="weights.hdf5", freeze_fac=0.75,
                parallel=False, quick_setup=False):
    """Main routine for setting up the model, from scratch or from a checkpoint
    (spnet/models.py:461-507). Returns (model, serial_model)."""
    print("Initializing blank model: Y0size =", Y0size)
    if cf.model_type == "simple":
        raise NotImplementedError("cf.model_type == 'simple' (NASNetMobile, 'Not recommended!' in the reference) is not built")
    model = create_model_functional(X, Y0size=Y0size, freeze_fac=freeze_fac, quick_setup=quick_setup)
    if try_checkpoint:
        if isfile(weights_file):
            print("Weights file detected. Loading from", weights_file)
            model.load_weights(weights_file)
        else:
            if no_cp_fatal:
                raise Exception("*** No weights file detected; can't do anything.  Aborting.")
            else:
                print("    No weights file detected, so starting from scratch.")
    serial_model = model
    opt = Adam(lr=0.00001)
    if parallel and (len(multi_gpu.get_available_gpus()) > 1):
        model = multi_gpu.make_parallel(model)
    print("Compiling the model")
    model.compile(loss=custom_loss, optimizer=opt)
    return model, serial_model


def unfreeze_model(model, X, Y, parallel=False):
    """New identical model with every layer trainable and the old weights (spnet/models.py:510-552)."""
    print("Unfreezing Model: make a new identical model, then copy the layer weights.")
    y0size = int(Y[0].numel()) if hasattr(Y[0], "numel") else int(Y[0].size)  # device-resident targets are tensors
    new_model = create_model_functional(X, y0size, freeze_fac=0)
    new_model.set_weights(multi_gpu.get_serial_part(model, parallel=parallel).get_weights())
    if parallel:
        new_model = multi_gpu.make_parallel(new_model)
    new_model.compile(loss=custom_loss, optimizer=Adam(lr=0.00001))
    print("  ...finished un-freezing model")
    tr, nt = new_model._count_trainable()
    tot = tr + nt
    print("post-unfreeze_model: Total params: {:,}".format(tot))
    print("post-unfreeze_model: Trainable params: {:,}".format(tr))
    print("post-unfreeze_model: Non-trainable params: {:,}".format(nt))
    return new_model


def load_model(filepath):
    """keras.models.load_model counterpart (reference call sites: predict_spnet.py:77-79, evaluate_spnet.py). Reads files
    written by SPNetModel.save (HDF5 or .npz) and Keras `model.save` HDF5 files: the weights come from /model_weights,
    the backbone from the layer names, the input size from the Keras model_config's InputLayer."""
    d, cfg = SPNetModel._read_weight_file(filepath)
    own = (cfg or {}).get("spnet_b200")
    if own is not None:
        H, W, Y0, use_l2, backbone = own["H"], own["W"], own["Y0size"], own["use_l2"], own.get("backbone") or "Xception"
        if own.get("loss_type"):
            cf.loss_type = own["loss_type"]   # the reference's load_model restores the compiled loss with the model
    else:
        backbone = "MobileNet" if "conv_pw_13/kernel" in d else ("InceptionResNetV2" if "conv_7b/kernel" in d else "Xception")
        Y0, use_l2 = int(d["FinalOutput/kernel"].shape[1]), True
        H = W = None
        try:   # Keras model_config: {"class_name": "Model", "config": {"layers": [{"class_name": "InputLayer", "config": {...}}]}}
            for layer in cfg["config"]["layers"]:
                if layer["class_name"] == "InputLayer":
                    _, H, W = layer["config"]["batch_input_shape"][:3]
                    break
        except Exception:
            pass
        if H is None:
            raise ValueError("load_model: %s carries no input size (neither an spnet_b200 config nor a Keras model_config)" % filepath)
    m = SPNetModel((int(H), int(W), 1), Y0size=int(Y0), quick_setup=not use_l2, backbone=backbone)
    missing = [k for k, _, _, _ in m.spec if k not in d]
    if missing:
        raise ValueError("load_model: %s does not hold a %s-SPNet for %dx%d input (%d tensors missing, first: %s)"
                         % (filepath, backbone, H, W, len(missing), missing[0]))
    m._load_dict(d)
    m.compile(loss=custom_loss, optimizer=Adam(lr=0.00001))
    return m
