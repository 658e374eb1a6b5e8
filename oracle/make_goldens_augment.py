"""ORACLE tooling — run ONCE in the authoring container (needs /root/reference and cv2):
    python oracle/make_goldens_augment.py
Runs the reference's own AugmentOnTheFly.on_epoch_begin (spnet/callbacks.py:272-341) on seeded frames with
np.random.seed(123) and stores input and output as tests/golden/ref_augment.npz: the host path of
spnet_b200.callbacks.AugmentOnTheFly consumes numpy's stream in the same order and must reproduce it bit for bit."""
import os
import random
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_shim  # noqa: E402

ref_shim.install()
sys.argv = ["make_goldens_augment"]
from spnet import callbacks  # noqa: E402


def main():
    rng = np.random.RandomState(5)
    X0 = (rng.rand(10, 96, 128, 1).astype(np.float32) * 2 - 1)
    Y0 = rng.rand(10, 8).astype(np.float32)
    X, Y = X0.copy(), Y0.copy()
    cb = callbacks.AugmentOnTheFly(X, Y, aug_every=1)
    np.random.seed(123)
    random.seed(123)
    cb.on_epoch_begin(0)
    first = X.copy()
    cb.on_epoch_begin(1)  # second epoch continues the stream from the pristine copy
    # each epoch as the pixels it changed, NaN elsewhere: the unchanged pixels are X0's and compress poorly
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "ref_augment.npz"), X0=X0, Y0=Y0,
                        epoch0_changed=np.where(first != X0, first, np.float32(np.nan)),
                        epoch1_changed=np.where(X != X0, X, np.float32(np.nan)), Y_after=Y)
    print("changed:", [(first[i] != X0[i]).mean().round(3) for i in range(10)])


if __name__ == "__main__":
    main()
