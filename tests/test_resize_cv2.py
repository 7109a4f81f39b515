"""Hold the numpy restatement of cv2.resize (oracle/preprocess_oracle.py: resize_linear, resize_nearest) to the
installed OpenCV bit for bit, with no tolerance, on a designed grid of geometry classes and source data
(tests/resize_grid.py).  The device resize kernels are held to the same grid in tests/test_resize_gpu.py, so a
difference between the restatement and cv2 cannot hide behind a difference the device shares."""
import numpy as np
import pytest

from oracle import preprocess_oracle as po
from tests import resize_grid as rg

cv2 = pytest.importorskip("cv2")


@pytest.mark.parametrize("kind", rg.DATA)
@pytest.mark.parametrize("geometry", list(rg.GEOMETRIES))
@pytest.mark.parametrize("interpolation", ["linear", "nearest"])
def test_restatement_matches_cv2(interpolation, geometry, kind):
    flag, ours = {"linear": (cv2.INTER_LINEAR, po.resize_linear), "nearest": (cv2.INTER_NEAREST, po.resize_nearest)}[interpolation]
    bad = []
    n = 0
    for sw, sh, dw, dh, src in rg.cases(geometry, kind):
        ref = cv2.resize(src, dsize=(dw, dh), interpolation=flag)
        n += 1
        if not rg.same_bits(ours(src, dw, dh), ref):
            bad.append((sw, sh, dw, dh))
    assert n > 0
    assert not bad, "{} of {} geometries differ from cv2.resize, e.g. (sw, sh, dw, dh) {}".format(len(bad), n, bad[:5])


def test_grid_reaches_each_class():
    """Each class holds what its name says, so a class cannot silently lose its geometries."""
    g = rg.GEOMETRIES
    assert all((sw, sh) == (dw, dh) for sw, sh, dw, dh in g["identity"])
    assert all((sw == dw) != (sh == dh) for sw, sh, dw, dh in g["one_side_unchanged"])
    assert all(sw == 1 or sh == 1 for sw, sh, dw, dh in g["thin"])
    assert (1, 1, 64, 64) in g["thin"]
    thin = g["thin"]
    assert any(sw == 1 and dh > sh for sw, sh, dw, dh in thin) and any(sw == 1 and 1 < dh < sh for sw, sh, dw, dh in thin)
    assert any(sh == 1 and dw > sw for sw, sh, dw, dh in thin) and any(sh == 1 and 1 < dw < sw for sw, sh, dw, dh in thin)
    sizes = {max(dw, dh) for sw, sh, dw, dh in g["aspect_preserving"]}
    assert set(rg.FRAME_SIZES) <= sizes
    assert {sw // dw for sw, sh, dw, dh in g["integer_scale"] if sw > dw} == {2, 3, 4}
    assert any(dw > sw and dw % sw == 0 for sw, sh, dw, dh in g["integer_scale"])
    # every landing geometry has a destination index whose exact source coordinate is an integer, on a side > 1
    for sw, sh, dw, dh in g["integer_landing"]:
        assert any(sn > 1 and any(((2 * d + 1) * sn - dn) % (2 * dn) == 0 for d in range(dn))
                   for sn, dn in ((sw, dw), (sh, dh)))


def test_fma32_rounds_once():
    """The oracle's fused multiply-add is one rounding of the exact value, where the plain fp64 sum rounds twice."""
    x = np.float32(2.0 ** -12 * (1 + 2.0 ** -23))
    y = np.float32(2.0 ** -12 * (1 - 2.0 ** -23))  # x * y = 2^-24 - 2^-70
    z = np.float32(1 + 2.0 ** -23)
    # exact x * y + z = 1 + 2^-23 + 2^-24 - 2^-70: just below the midpoint of 1 + 2^-23 and 1 + 2^-22, so it rounds down;
    # the fp64 sum lands on the midpoint itself and then rounds to the even 1 + 2^-22
    assert np.float32(x.astype(np.float64) * y + z) == np.float32(1 + 2.0 ** -22)
    assert po.fma32(x, y, z) == np.float32(1 + 2.0 ** -23)
    assert po.fma32(-x, y, -z) == np.float32(-(1 + 2.0 ** -23))
