"""The C restatement of OpenCV's MOG2 (oracle/mog2_oracle.c) against live cv2.createBackgroundSubtractorMOG2(detectShadows=False):
every foreground mask and getBackgroundImage() after every frame are equal, over the designed scenes and learning-rate
schedules of tests/mog2_helpers.py.  This pins the arithmetic the device kernels (csrc/mog2_kernels.cu) are held to.  No GPU."""
import numpy as np
import pytest

from tests import mog2_helpers as mh

cv2 = pytest.importorskip("cv2")


def run_both(frames, lrs, history):
    from oracle.mog2_oracle import Mog2Oracle

    cvm = cv2.createBackgroundSubtractorMOG2(history=history, detectShadows=False)
    orc = Mog2Oracle(frames.shape[1:], history=history)
    for t, (f, lr) in enumerate(zip(frames, lrs)):
        a = cvm.apply(f, None, lr)
        b = orc.apply(f, lr)
        assert np.array_equal(a, b), "mask of frame {} (lr {}): {} pixels differ".format(t, lr, int((a != b).sum()))
        bg = cvm.getBackgroundImage()
        assert np.array_equal(bg, orc.background()), "background after frame {}".format(t)
    return orc


@pytest.mark.parametrize("name", mh.SCENES)
@pytest.mark.parametrize("history", [1000, 4])
def test_oracle_equals_cv2_on_designed_scenes(name, history):
    frames = mh.scene(name, (61, 97), 60, seed=3)
    orc = run_both(frames, mh.scene_rates(name, len(frames)), history)
    for branch in mh.BRANCHES[name]:
        assert orc.stat(branch) > 0, (name, branch, orc.stats.tolist())


@pytest.mark.parametrize("sched", mh.SCHEDULES)
def test_oracle_equals_cv2_on_learning_rate_schedules(sched):
    frames = mh.scene("mixed", (64, 64), 60, seed=5)
    run_both(frames, mh.schedule(sched, len(frames)), history=1000)
    run_both(frames, mh.schedule(sched, len(frames)), history=3)


def test_oracle_equals_cv2_640x480():
    frames = mh.scene("walk", (480, 640), 40, seed=7)
    run_both(frames, mh.schedule("recording", len(frames)), history=1000)


def test_prune_constant_is_float_product():
    """prune = (float)(-lr * (double)0.05f): at lr = 1/66 it differs from (float)(-lr * 0.05), which is why the constant is
    computed so (and a mask pixel of cv2 depends on it)."""
    from oracle.mog2_oracle import rates

    lr = 1.0 / 66
    _, prune = rates(lr, 2, 1000)
    assert prune == np.float32(-lr * np.float64(np.float32(0.05)))
    assert prune != np.float32(-lr * 0.05)
