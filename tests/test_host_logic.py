"""CPU tests: the product's host-side codec (spnet_b200/utils.py, callbacks.py) against the
reference-generated goldens, the C-ABI library (loads, exports every declared symbol), the
Keras-like surface that needs no GPU, and the data-parallel host logic on gloo (world size 2)."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(G, "ref_numpy_side.npz")), json.load(open(os.path.join(G, "ref_text.json")))


def test_library_builds_loads_and_exports_every_symbol():
    import __graft_entry__ as ge
    lib_path = ge.build()
    from spnet_b200 import _lib
    protos = _lib.parse_header()
    assert len(protos) >= 39
    dll = ctypes.CDLL(lib_path)
    for name in protos:
        assert hasattr(dll, name), name
    assert dll.spnet_version() >= 100
    # error convention: bad arguments -> negative code + message, never a crash (no GPU needed: checked before launch)
    dll.spnet_last_error.restype = ctypes.c_char_p
    rc = dll.spnet_yolo_ellipse_loss(None, None, 0, 0, 0, 0, None, None, None)
    assert rc == -1 and b"null pointer" in dll.spnet_last_error()


def test_product_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from spnet_b200 import models
    with pytest.raises(Exception):
        models.custom_loss(np.zeros((1, 576), np.float32), np.zeros((1, 576), np.float32))


def test_utils_match_reference_goldens(gold):
    a, t = gold
    from spnet import utils
    r = utils.setup_means_and_ranges([6, 6, 2, 8])
    assert tuple(r[:6]) == (40, 40, 470, 350, 71, 51)
    np.testing.assert_array_equal(r[6], a["smr_grid_defaults"])
    np.testing.assert_array_equal(utils.means, a["means"])
    np.testing.assert_array_equal(utils.ranges, a["ranges"])
    for i, rows in enumerate(t["meta_rows"]):
        parsed = utils.parse_meta_rows(rows)
        assert len(parsed) == len(t["parsed_meta"][i])
        if parsed:
            np.testing.assert_array_equal(np.array(parsed, float), np.array(t["parsed_meta"][i], float))
        np.testing.assert_array_equal(utils.true_to_pred_grid(np.array(parsed), [6, 6, 2, 8]).flatten(), a["grid_Y_raw"][i])
    Y, shape = utils.build_Y_from_rows(t["meta_rows"])
    np.testing.assert_array_equal(Y, a["grid_Y_norm"])
    np.testing.assert_array_equal(utils.denorm_Y(a["grid_Y_norm"]), a["grid_Y_denorm"])
    with pytest.raises(AssertionError):
        utils.true_to_pred_grid(np.array([[100, 140, 30, 20, 1, 0, 0, 3]] * 3, float), [6, 6, 2, 8])
    assert utils.nearest_multiple(720, 31) == 713
    assert utils.add_to_stack(utils.add_to_stack(None, 5), 5) == [5, 5]


def test_csv_writer_matches_reference_text(gold, tmp_path):
    a, t = gold
    from spnet import utils
    utils.setup_means_and_ranges([6, 6, 2, 8])
    Yp = a["csv_Yp_denorm"]
    out = tmp_path / "hawley_spnet.csv"
    utils.show_pred_ellipses(Yp, Yp, t["csv_files"], num_draw=Yp.shape[0], log_dir=str(tmp_path), out_csv=str(out),
                             show_true=False, draw_images=False)
    assert out.read_text() == t["csv_text"]
    ints, exists = utils.decode_host(Yp)
    np.testing.assert_array_equal(ints.reshape(-1, 5), a["cleanup_ints"])
    np.testing.assert_array_equal(utils._angles(Yp).reshape(-1), a["cleanup_angle"])
    for j in range(3):
        for an in range(72):
            c = utils.cleanup_antinode_vars(Yp[j, an * 8:(an + 1) * 8])
            assert (c[0], c[1], c[2], c[3], c[5]) == tuple(ints[j, an])


def test_meta_file_and_build_Y(tmp_path, gold):
    a, t = gold
    from spnet import utils
    metas, imgs = [], []
    for i, rows in enumerate(t["meta_rows"][:6]):
        p = tmp_path / ("steelpan_%07d.csv" % i)
        p.write_text("\n".join(",".join(str(v) for v in r) for r in rows))
        metas.append(str(p))
        imgs.append(str(p).replace(".csv", ".png"))
    Y, shape = utils.build_Y(6, metas, imgs)
    np.testing.assert_array_equal(Y, a["grid_Y_norm"][:6])
    assert list(shape) == [6, 6, 2, 8]


def test_build_X_normalisation(tmp_path):
    from PIL import Image
    from spnet import utils
    rng = np.random.default_rng(0)
    files = []
    for i in range(3):
        arr = rng.integers(0, 256, (384, 512), dtype=np.uint8)
        p = tmp_path / ("img%d.png" % i)
        Image.fromarray(arr).save(p)
        files.append((str(p), arr))
    X, dims = utils.build_X(3, [f for f, _ in files], force_dim=None, grayscale=True)
    assert X.shape == (3, 384, 512, 1) and X.dtype == np.float32
    for i, (_, arr) in enumerate(files):
        ref = arr.astype(np.float32) / 255.0
        ref -= 0.5
        ref *= 2.0
        np.testing.assert_array_equal(X[i, :, :, 0], ref)
    X331, _ = utils.build_X(2, [f for f, _ in files], force_dim=331, grayscale=True)
    assert X331.shape == (2, 331, 331, 1) and -1.0 <= X331.min() and X331.max() <= 1.0


def test_one_cycle_schedule_and_callback(gold):
    a, _ = gold
    from spnet import callbacks
    lrs = callbacks.get_1cycle_schedule(lr_max=4e-5, n_data_points=40000, epochs=100, batch_size=16)
    np.testing.assert_array_equal(np.array([len(lrs), lrs[0], lrs[2499], lrs[4999], lrs.max(), lrs[-1]]), a["lrs_probe"])
    np.testing.assert_array_equal(callbacks.get_1cycle_schedule(1e-3, 64, 5, 8), a["lrs_small"])

    class Opt:
        lr = 0.0

    class M:
        optimizer = Opt()
    cb = callbacks.OneCycleScheduler(lr_max=1e-3, n_data_points=64, epochs=5, batch_size=8)
    cb.set_model(M())
    seen = []
    for _ in range(40):
        cb.on_batch_begin(0)
        seen.append(cb.model.optimizer.lr)
    np.testing.assert_array_equal(np.array(seen), a["lrs_small"])
    logs = {}
    cb.on_epoch_end(0, logs)
    assert logs["lr"] == seen[-1]


def test_model_surface_without_gpu(tmp_path):
    from spnet import models
    import spnet.config as cf
    from spnet_b200 import arch
    X = np.zeros((2, 331, 331, 1), np.float32)
    model, serial = models.setup_model(X, 576, try_checkpoint=True, no_cp_fatal=False, weights_file=str(tmp_path / "none.hdf5"),
                                       freeze_fac=0.0)
    assert model is serial and model.count_params() == 50353481          # paper/run_logs/log_DatasetA_*.txt:99
    assert arch.count_params(model.spec) == (50353481, 50298935, 54546)
    assert sorted(k.split("/")[0] for k in model.losses) == sorted(
        ["conv2d_%d" % i for i in range(1, 8)] + ["block1_conv1", "block1_conv2", "FinalOutput"])   # log:98
    assert model.optimizer.lr == 0.00001 and model.loss is models.custom_loss
    assert arch.shape_walk(331, 331)["stem"] == (165, 165) and arch.shape_walk(331, 331)["out13"] == (5, 5)
    assert arch.count_params(arch.param_spec(384, 512))[0] == 77485385
    with pytest.raises(Exception, match="No weights file detected"):
        models.setup_model(X, 576, no_cp_fatal=True, weights_file=str(tmp_path / "none.hdf5"))
    with pytest.raises(ValueError):
        models.SPNetModel((331, 331, 1), Y0size=577)
    # weights round trip through the file format and get/set_weights
    small = models.SPNetModel((67, 67, 1), quick_setup=True)
    path = str(tmp_path / "w.hdf5")
    small.save_weights(path)
    other = models.SPNetModel((67, 67, 1), quick_setup=True, seed=99)
    other.load_weights(path)
    for x, y in zip(small.get_weights(), other.get_weights()):
        np.testing.assert_array_equal(x, y)
    other.set_weights(small.get_weights())
    with pytest.raises(ValueError):
        other.set_weights(small.get_weights()[:-1])
    small.save(str(tmp_path / "full.h5"))
    again = models.load_model(str(tmp_path / "full.h5"))
    np.testing.assert_array_equal(again.get_weights()[0], small.get_weights()[0])
    names = [l.name for l in small.layers]
    assert names[0] == "conv2d_1" and names[-1] == "FinalOutput" and "block8_sepconv2_bn" in names
    assert cf.vars_per_pred == 8 and cf.ind_noobj == 6


def test_fake_espi_generator_statistics():
    from spnet_b200 import fake_espi
    ref = np.load(os.path.join(G, "fake_espi_frames.npz"))["frames"]
    img, rows = fake_espi.make_frame(0)
    assert img.shape == (384, 512) and img.dtype == np.uint8 and 1 <= len(rows) <= 7
    # same recipe as the reference's drawing code: half the pixels dropped, comparable brightness
    assert abs((img == 0).mean() - (ref == 0).mean()) < 0.1
    assert abs(float(img.mean()) - float(ref.mean())) < 15
    X, Y, _ = fake_espi.make_dataset(3, base_seed=5)
    assert X.shape == (3, 384, 512, 1) and Y.shape == (3, 576) and X.min() >= -1 and X.max() <= 1
    X2, Y2, _ = fake_espi.make_dataset(3, base_seed=5)
    np.testing.assert_array_equal(X, X2)
    np.testing.assert_array_equal(Y, Y2)


DP_SCRIPT = r"""
import os, sys
sys.path.insert(0, %r)
import numpy as np, torch, torch.distributed as dist
from collections import OrderedDict
from spnet_b200 import multi_gpu
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
assert multi_gpu.world() == (rank, world)
lo, hi = multi_gpu.batch_slice(10, rank, world)      # get_slice: size = shape[0] // parts, remainder dropped
assert (lo, hi) == (rank * 5, rank * 5 + 5)
class FakeEngine:
    device = "cpu"
    lowp = False                         # fp32 engine -> fp32 communication
    def __init__(self, tail_key):
        self.offsets = OrderedDict([("FinalOutput/kernel", (0, 24, (4, 6))), ("entry", (24, 8, (8,))), ("middle", (32, 16, (16,)))])
        self.tail_param_key = tail_key
        self.grads = torch.arange(48, dtype=torch.float32) * (rank + 1)
        self.steps = []
    def optimizer_step(self, grad_scale=1.0, lo=0, hi=None, g_bf16=None):
        # the bucket's gradients must already be the sum over the ranks when its update is launched
        expect = torch.arange(lo, hi, dtype=torch.float32) * sum(r + 1 for r in range(world))
        assert torch.equal(self.grads[lo:hi], expect), (lo, hi)
        assert g_bf16 is None
        self.steps.append((lo, hi, grad_scale))
for tail_key in ("middle", None):        # with and without a tail bucket (Xception / MobileNet engines)
    eng = FakeEngine(tail_key)
    hook = multi_gpu.attach_data_parallel(eng)
    assert hook.ranges["head"] == (0, 24) and hook.ranges["tail"] == ((32, 48) if tail_key else (48, 48))
    assert hook.ranges["rest"] == ((24, 32) if tail_key else (24, 48))
    hook.step_begin(eng)
    hook.bucket_ready(eng, "head")       # on CPU the buckets are reduced in the final call
    hook.bucket_ready(eng, "tail")
    hook(eng)
    expect = torch.arange(48, dtype=torch.float32) * sum(r + 1 for r in range(world))
    assert torch.equal(eng.grads, expect), (eng.grads, expect)
    # every parameter updated exactly once, each bucket with the 1/world average
    covered = sorted((lo, hi) for lo, hi, _ in eng.steps)
    assert covered == sorted(r for r in hook.ranges.values() if r[1] > r[0]), covered
    assert all(sc == 1.0 / world for _, _, sc in eng.steps)
    assert eng.skip_default_optimizer
dist.barrier()
if rank == 0:
    print("DP_OK")
"""


def test_data_parallel_host_logic_gloo_world2(tmp_path):
    script = tmp_path / "dp.py"
    script.write_text(DP_SCRIPT % ROOT)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29533")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29533", str(script)],
                         capture_output=True, text=True, env=env, timeout=240)
    assert "DP_OK" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]


def test_stream_X_yields_build_X_in_chunks(tmp_path):
    """utils.stream_X: same values as build_X (spnet/utils.py:325-421), chunked, next chunk decoded in the
    background; ragged last chunk; both the native-size grayscale path and the LANCZOS-resize path."""
    from PIL import Image
    from spnet_b200 import utils
    rng = np.random.RandomState(4)
    files = []
    for i in range(7):
        img = rng.randint(0, 256, (48, 64), dtype=np.uint8)
        f = str(tmp_path / ("f_%02d.png" % i))
        Image.fromarray(img).save(f)
        files.append(f)
    for force_dim, gray in ((None, True), (32, True), (32, False)):
        X, _ = utils.build_X(len(files), files, force_dim=force_dim, grayscale=gray)
        got, starts = [], []
        for lo, Xc in utils.stream_X(files, 3, force_dim=force_dim, grayscale=gray):
            starts.append(lo)
            got.append(Xc)
        assert starts == [0, 3, 6] and [g.shape[0] for g in got] == [3, 3, 1]
        np.testing.assert_array_equal(np.concatenate(got, axis=0), X)
    assert list(utils.stream_X([], 3)) == []


def test_every_exported_entry_point_is_documented():
    """INTEGRATION.md is the map from reference operations to C-ABI entry points: nothing the header exports may
    be missing from it (names may be written with {a,b} alternations)."""
    import re
    from spnet_b200._lib import parse_header
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    text = open(os.path.join(root, "INTEGRATION.md")).read()
    expanded = set(re.findall(r"spnet_\w+", text))
    for stem, alts, tail in re.findall(r"(spnet_\w*?)\{([^}]*)\}(\w*)", text):
        for a in alts.split(","):
            expanded.add(stem + a.strip() + tail)
    for stem in re.findall(r"(spnet_\w+_)\*", text):
        expanded.update(n for n in parse_header() if n.startswith(stem))
    missing = sorted(n for n in parse_header() if n not in expanded)
    assert not missing, missing


# ------------------------------------------------------------------ round 2: freeze list, checkpoints, sharded CSV merge
def test_keras_layer_order_and_freeze_cut():
    """base_model.layers[:int(144 * freeze_fac)].trainable = False (spnet/models.py:361-372) on the Keras layer order:
    144 layers for Xception-SPNet (paper/run_logs/log_DatasetA_*.txt:95), the 75 % cut ends with block 10."""
    from spnet_b200 import arch
    L = arch.xception_keras_layers()
    assert len(L) == 144 and len(set(L)) == 144 and L[0] == "input_1" and L[12] == "dropout_1"
    assert L[19:28] == ["block2_sepconv1", "block2_sepconv1_bn", "block2_sepconv2_act", "block2_sepconv2", "block2_sepconv2_bn",
                        "conv2d_4", "block2_pool", "batch_normalization_4", "add_2"]
    spec = arch.param_spec(331, 331)
    with_weights = set(k.split("/")[0] for k, _, _, _ in spec)
    assert with_weights - {"FinalOutput"} <= set(L)
    names, nf, nt = arch.frozen_layer_names("Xception", 0.75, spec)
    assert (nf, nt) == (108, 144) and names[-1] == "block10_sepconv3_bn" and "block11_sepconv1" not in names
    assert arch.frozen_layer_names("Xception", 0.0, spec)[0] == []
    assert set(arch.frozen_layer_names("Xception", 1.0, spec)[0]) == with_weights - {"FinalOutput"}
    assert len(arch.mobilenet_keras_layers()) == 94
    import spnet.config as cf
    from spnet import models
    cf.basemodel = "Xception"
    m = models.create_model_functional(np.zeros((1, 331, 331, 1), np.float32), 576, freeze_fac=0.75)
    tr, ntr = m._count_trainable()
    assert tr + ntr == 50353481 and tr == 39508112
    m0 = models.create_model_functional(np.zeros((1, 331, 331, 1), np.float32), 576, freeze_fac=0.0)
    assert m0._count_trainable() == (50298935, 54546)   # log_DatasetA_*.txt:100-101


@pytest.mark.parametrize("backbone,hw", [("Xception", (96, 128)), ("MobileNet", (96, 128)), ("InceptionResNetV2", (200, 260))])
def test_full_model_save_and_load_model_round_trip(tmp_path, backbone, hw):
    """spnet.model / full_model.h5 (ParallelCheckpointCallback, train_spnet.py:149): load_model rebuilds the backbone
    that was saved, with its weights and the loss type it was compiled with."""
    import spnet.config as cf
    from spnet import models
    cf.basemodel, old_loss = backbone, cf.loss_type
    try:
        cf.loss_type = "hybrid"
        m = models.create_model_functional(np.zeros((1,) + hw + (1,), np.float32), 576, freeze_fac=0.0, quick_setup=True)
        path = str(tmp_path / "spnet.model")
        m.save(path)
        cf.loss_type = "same"
        m2 = models.load_model(path)
        assert m2.backbone == backbone and cf.loss_type == "hybrid" and (m2.H, m2.W) == hw
        for a, b in zip(m.get_weights(), m2.get_weights()):
            np.testing.assert_array_equal(a, b)
        wrong = models.SPNetModel((hw[0] * 2, hw[1], 1), backbone=backbone, quick_setup=True)
        with pytest.raises(ValueError):
            wrong.set_weights(m.get_weights())
    finally:
        cf.basemodel, cf.loss_type = "Xception", old_loss


def test_checkpoint_callback_saves_like_the_reference(tmp_path):
    """spnet/callbacks.py:35-41: save when save_every == 1, or after the 5th, 10th, ... epoch for save_every = 5; paths
    are dir + '/' + filepath and dir + '/spnet.model'."""
    from spnet import callbacks

    class M:
        saved = []

        def save_weights(self, p):
            self.saved.append(("w", p))

        def save(self, p):
            self.saved.append(("m", p))

    m = M()
    ck = callbacks.ParallelCheckpointCallback(m, filepath="weights.hdf5", save_every=5, dir=str(tmp_path / "logs"))
    ck.model = None
    hits = []
    for epoch in range(12):
        n0 = len(m.saved)
        ck.on_epoch_end(epoch)
        if len(m.saved) > n0:
            hits.append(epoch)
    assert hits == [4, 9]
    assert m.saved[0] == ("w", str(tmp_path / "logs") + "/weights.hdf5") and m.saved[1] == ("m", str(tmp_path / "logs") + "/spnet.model")
    m.saved.clear()
    ck1 = callbacks.ParallelCheckpointCallback(m, save_every=1, dir=str(tmp_path))
    ck1.model = None
    for epoch in range(3):
        ck1.on_epoch_end(epoch)
    assert len(m.saved) == 6
    # device-augmentation epoch keys: no two (epoch, frame) pairs of neighbouring epochs share a key
    G = 0x9E3779B97F4A7C15
    keys = set()
    for e in range(20):
        sd = callbacks._epoch_seed(1234, e) & (2 ** 63 - 1)
        for f in range(50):
            keys.add((sd + G * (f + 1)) & 0xFFFFFFFFFFFFFFFF)
    assert len(keys) == 20 * 50


def test_sharded_csv_parts_merge_in_rank_order(tmp_path, monkeypatch):
    import predict_spnet
    out = str(tmp_path / "hawley_spnet.csv")
    monkeypatch.setenv("MASTER_PORT", "12345")
    for r, text in ((2, "c\n"), (1, "b1\nb2\n"), (0, "a\n")):
        with open(out + ".part%d" % r, "w") as f:
            f.write(text)
    predict_spnet.merge_csv_parts(out, 2, 3)
    predict_spnet.merge_csv_parts(out, 1, 3)
    assert not os.path.exists(out)
    predict_spnet.merge_csv_parts(out, 0, 3)
    assert open(out).read() == "a\nb1\nb2\nc\n"
    assert os.listdir(str(tmp_path)) == ["hawley_spnet.csv"]


def test_stored_oracle_is_the_plain_oracle_without_rounding():
    """oracle/xception_torch.py Oracle*Stored(storage='fp32') restates the engine's storage points without rounding: it
    must compute what the plain oracle computes (inference mode: to fp32 rounding)."""
    import torch
    from oracle import xception_torch as xt
    from spnet_b200.selfcheck import make_case
    for name, plain, stored, (H, W) in (("Xception", xt.OracleSPNet, xt.OracleSPNetStored, (96, 128)),
                                        ("MobileNet", xt.OracleMobileNetSPNet, xt.OracleMobileNetSPNetStored, (96, 128))):
        w, x, yt = make_case(H, W, 2, seed=3, backbone=name)
        with torch.no_grad():
            ya = plain(w, H, W).forward(x, training=False)
            yb = stored(w, H, W, storage="fp32").forward(x, training=False)
            yc = stored(w, H, W, storage="bf16").forward(x, training=False)
        assert float((ya - yb).abs().max() / ya.abs().max()) < 2e-6
        assert 1e-4 < float((ya - yc).norm() / ya.norm()) < 2e-2   # bf16 storage is visible, and small in inference mode


# ------------------------------------------------------------------ Keras HDF5 checkpoints (spnet_b200/hdf5_min.py)
def test_hdf5_reader_on_a_file_written_by_libhdf5():
    """The reader against a GENUINE HDF5 file (MATLAB v7.3 = libhdf5; a copy of scipy's test file
    scipy/io/matlab/tests/data/testhdf5_7.4_GLNX86.mat, BSD-licensed: 512-byte user block, superblock 0, symbol-table
    group, B-tree + local heap, version-1 object header, attribute, dataset)."""
    from spnet_b200 import hdf5_min
    r = hdf5_min.Reader(os.path.join(G, "testhdf5_7.4_GLNX86.mat"))
    assert r.base == 512 and list(r.links(r.root)) == ["testdouble"]
    a = r.resolve("testdouble")
    assert r.attrs(a) == {"MATLAB_class": b"double"}
    np.testing.assert_allclose(r.dataset(a).ravel(), np.arange(0, 2 * np.pi + 1e-9, np.pi / 4), rtol=0, atol=1e-15)


@pytest.mark.parametrize("backbone,hw", [("Xception", (96, 128)), ("InceptionResNetV2", (200, 260))])
def test_keras_hdf5_weight_files_round_trip(tmp_path, backbone, hw):
    """weights.hdf5 / full_model.h5 in the Keras layout (layer_names / weight_names attributes, datasets at
    /<layer>/<layer>/<weight>:0, /model_weights for full models): written and read back bit for bit; a 450-group root
    (InceptionResNetV2) exercises the multi-level B-tree."""
    import spnet.config as cf
    from spnet import models
    from spnet_b200 import hdf5_min
    cf.basemodel = backbone
    try:
        m = models.create_model_functional(np.zeros((1,) + hw + (1,), np.float32), 576, freeze_fac=0.0, quick_setup=True)
        wpath, fpath = str(tmp_path / "weights.hdf5"), str(tmp_path / "full_model.h5")
        m.save_weights(wpath)
        m.save(fpath)
        assert open(wpath, "rb").read(8) == b"\x89HDF\r\n\x1a\n"
        d, attrs = hdf5_min.read_keras_weights(wpath)
        assert attrs["keras_version"] == b"2.1.3" and attrs["backend"] == b"tensorflow"
        r = hdf5_min.Reader(wpath)
        names = [n.decode() for n in r.attrs(r.root)["layer_names"]]
        assert "FinalOutput" in names and len(names) == len(set(names)) and set(r.links(r.root)) == set(names)
        if backbone == "Xception":
            assert names[:3] == ["input_1", "conv2d_1", "average_pooling2d_1"] and len(names) == 146
            assert [w.decode() for w in r.attrs(r.resolve("block5_sepconv1"))["weight_names"]] == [
                "block5_sepconv1/depthwise_kernel:0", "block5_sepconv1/pointwise_kernel:0"]
            assert r.dataset(r.resolve("block5_sepconv1/block5_sepconv1/pointwise_kernel:0")).shape == (1, 1, 728, 728)
        w0 = m.get_weights()
        m2 = models.create_model_functional(np.zeros((1,) + hw + (1,), np.float32), 576, freeze_fac=0.0, quick_setup=True)
        m2._load_dict({k: np.zeros_like(v) for k, v in m._weights_dict().items()})
        m2.load_weights(wpath)
        for a, b in zip(w0, m2.get_weights()):
            np.testing.assert_array_equal(a, b)
        m3 = models.load_model(fpath)
        assert m3.backbone == backbone and (m3.H, m3.W) == hw
        for a, b in zip(w0, m3.get_weights()):
            np.testing.assert_array_equal(a, b)
        # the .npz container (any other file name) still works, and a file of the wrong size is refused
        m.save_weights(str(tmp_path / "weights.npz"))
        m2.load_weights(str(tmp_path / "weights.npz"))
        other = models.SPNetModel((hw[0] * 2, hw[1], 1), backbone=backbone, quick_setup=True)
        with pytest.raises(ValueError):
            other.load_weights(wpath)
    finally:
        cf.basemodel = "Xception"


def test_csv_rows_text_equals_the_reference_row_format_on_awkward_values():
    """csv_rows formats from Python lists (%r / %d); the reference formats numpy float32 scalars with "{}".format
    (spnet/utils.py:122-126). Same text for integral values, tiny / huge magnitudes, negatives and empty images."""
    import spnet.config as cf
    from spnet_b200 import utils
    utils.setup_means_and_ranges([6, 6, 2, 8])
    rng = np.random.default_rng(3)
    n, v = 7, cf.vars_per_pred
    Yp = (rng.standard_normal((n, 576)) * 60 + 120).astype(np.float32)
    Yp[:, cf.ind_noobj::v] = 0.0                        # every predictor "exists" ...
    Yp[2, cf.ind_noobj::v] = 1.0                        # ... except in image 2 (the "0,0,name,0,0,0,0" row)
    Yp[0, cf.ind_rings::v] = np.float32(3.0)            # integral float -> "3.0"
    Yp[1, cf.ind_rings::v] = np.float32(1e-5)           # -> "9.999999747378752e-06"
    Yp[3, cf.ind_rings::v] = np.float32(-0.1)
    Yp[4, cf.ind_rings::v] = np.float32(1.5e9)
    ints, exists = utils.decode_host(Yp)
    names = ["some/dir/frame_%03d.png" % i for i in range(n)]
    got = utils.csv_rows(Yp, ints, exists, names)
    ang, rings = utils._angles(Yp), Yp[:, cf.ind_rings::v]
    want = []
    for j in range(n):
        base, idx = os.path.basename(names[j]), np.nonzero(exists[j])[0]
        if idx.size == 0:
            want.append("0,0," + base + ",0,0,0,0\n")
            continue
        want.append("".join("{},{},{},{},{},{},{}".format(int(ints[j, an, 0]), int(ints[j, an, 1]), base, rings[j, an],
                                                          int(ints[j, an, 2]), int(ints[j, an, 3]), ang[j, an]) + "\n" for an in idx))
    assert got == want
    assert want[2] == "0,0,frame_002.png,0,0,0,0\n" and ",3.0," in want[0]
