"""GPU parity of the single-image ml_tools.imageprocessing helpers (normalize, resize_and_pad, resize_cv,
detect_objects) through the C ABI, against the C / numpy oracles (which are pinned to cv2 / the reference)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def test_detect_objects_matches_oracle_lepton_and_ir_sizes():
    from classifier_pipeline_b200.ml_tools import imageprocessing as ip
    from oracle import oracle as orc

    rng = np.random.default_rng(11)
    for (H, W), thr in (((120, 160), 40.0), ((120, 160), 12.7), ((480, 640), 60.0), ((37, 53), 30.0), ((2, 2), 1.0)):
        for trial in range(3):
            img = rng.integers(0, 40, size=(H, W)).astype(np.float32)
            for _ in range(int(rng.integers(0, 12))):
                y, x = int(rng.integers(0, H)), int(rng.integers(0, W))
                h, w = int(rng.integers(1, max(2, H // 6))), int(rng.integers(1, max(2, W // 6)))
                img[y : y + h, x : x + w] += rng.integers(50, 200)
            img = np.clip(img, 0, 255)
            n, labels, stats, cents = ip.detect_objects(img, threshold=thr, kernel=(5, 5))
            on, olabels, ocomp = orc.detect_objects(np.uint8(img), thr, max_comp=8192)
            assert n == on + 1
            assert labels.dtype == np.int32 and np.array_equal(labels, olabels)
            ostats, ocents = orc.stats_centroids_from_comp(ocomp)
            assert np.array_equal(stats[1:], ostats)
            assert np.array_equal(cents[1:], ocents)
            bg = labels == 0
            if bg.any():
                ys, xs = np.nonzero(bg)
                assert list(stats[0]) == [xs.min(), ys.min(), xs.max() - xs.min() + 1, ys.max() - ys.min() + 1, bg.sum()]


def test_detect_objects_options():
    """The default (15, 15) kernel and Otsu are built (fixtures: tests/test_ir_gpu.py); kernel sizes whose fixed-point taps
    are not built are refused instead of approximated."""
    from classifier_pipeline_b200.ml_tools import imageprocessing as ip

    n, labels, stats, cents = ip.detect_objects(np.zeros((8, 8)))
    assert n == 1 and labels.shape == (8, 8) and not labels.any()
    n, _, _, _ = ip.detect_objects(np.zeros((8, 8)), otsus=True, kernel=(5, 5))
    assert n == 1
    with pytest.raises(NotImplementedError):
        ip.detect_objects(np.zeros((8, 8)), kernel=(9, 9))
    with pytest.raises(NotImplementedError):
        ip.detect_objects(np.zeros((8, 8)), kernel=(5, 7))


def test_normalize_matches_numpy_semantics():
    from classifier_pipeline_b200.ml_tools import imageprocessing as ip
    from oracle import preprocess_oracle as po

    rng = np.random.default_rng(2)
    f32 = rng.normal(0, 50, size=(31, 17)).astype(np.float32)
    out, (ok, mx, mn) = ip.normalize(f32, new_max=255)
    ref, _ = po.normalize(f32, new_max=255)
    assert ok and out.dtype == np.float32 and mx == f32.max() and mn == f32.min()
    np.testing.assert_allclose(out, ref, rtol=1e-6, atol=1e-5)
    u16 = rng.integers(2800, 3300, size=(120, 160)).astype(np.uint16)
    out, (ok, mx, mn) = ip.normalize(u16, new_max=255)
    ref, _ = po.normalize(u16, new_max=255)
    assert out.dtype == ref.dtype
    np.testing.assert_allclose(out, ref, rtol=1e-6, atol=1e-5)
    f64 = rng.integers(-200, 900, size=(20, 30)).astype(np.float64)  # get_delta_frame: float64 in, float64 arithmetic
    out, _ = ip.normalize(f64, new_max=255)
    ref, _ = po.normalize(f64, new_max=255)
    assert out.dtype == np.float64 and np.array_equal(out, ref)
    out, (ok, _, _) = ip.normalize(np.zeros((4, 4), np.float32))
    assert not ok and not out.any()
    out, (ok, _, _) = ip.normalize(np.full((4, 4), 7, np.float32))
    assert ok and np.array_equal(out, np.ones((4, 4), np.float32))
    out, (ok, _, _) = ip.normalize(np.zeros((0, 4)))
    assert not ok and out.shape == (0, 4)
    out, _ = ip.normalize(f32, min=-10.0, max=300.0, new_max=255)
    ref, _ = po.normalize(f32, -10.0, 300.0, new_max=255)
    np.testing.assert_allclose(out, ref, rtol=1e-6, atol=1e-5)


def test_resize_helpers_match_oracle():
    from classifier_pipeline_b200.ml_tools import imageprocessing as ip
    from classifier_pipeline_b200.ml_tools.rectangle import Rectangle
    from oracle import preprocess_oracle as po

    rng = np.random.default_rng(9)
    crop = Rectangle(1, 1, 158, 118)
    for _ in range(40):
        w, h = int(rng.integers(1, 70)), int(rng.integers(1, 60))
        x, y = int(rng.integers(1, 159 - w + 1)), int(rng.integers(1, 119 - h + 1))
        src = rng.integers(0, 4000, size=(h, w)).astype(np.float32)
        region = Rectangle(x, y, w, h)
        got = ip.resize_and_pad(src, (32, 32), region, crop, keep_edge=True)
        ref = po.resize_and_pad(src, (32, 32), (x, y, w, h), (1, 1, 158, 118), keep_edge=True)
        assert np.array_equal(got, ref)
        got = ip.resize_and_pad(src, (32, 32), region, crop, keep_edge=True, pad=0, interpolation=ip.INTER_NEAREST)
        ref = po.resize_and_pad(src, (32, 32), (x, y, w, h), (1, 1, 158, 118), keep_edge=True, pad=0, interpolation=po.INTER_NEAREST)
        assert np.array_equal(got, ref)
        dw, dh = int(rng.integers(1, 40)), int(rng.integers(1, 40))
        assert np.array_equal(ip.resize_cv(src, (dw, dh)), po.resize_linear(src, dw, dh))


def test_preprocess_frame_single_matches_oracle():
    """ml_tools.preprocess.preprocess_frame on one Frame == one tile of the batched oracle."""
    from classifier_pipeline_b200.ml_tools.frame import Frame
    from classifier_pipeline_b200.ml_tools.preprocess import preprocess_frame, preprocess_movement
    from classifier_pipeline_b200.ml_tools.rectangle import Rectangle
    from classifier_pipeline_b200.synthetic import make_clip
    from classifier_pipeline_b200.track.region import Region
    from oracle import preprocess_oracle as po

    pix, _ = make_clip(2, frames=30)
    filtered = (pix.astype(np.int64) - pix[0].astype(np.int64)).astype(np.float32)
    crop = Rectangle(1, 1, 158, 118)
    regions = np.array([[t, 20 + t, 30, 24, 18, 0] for t in range(5, 30)], np.int32)
    lo, hi = po.track_limits(filtered, regions)
    seg = [np.arange(5, 30)]
    oracle = po.preprocess_track(pix, filtered, regions, (1, 1, 158, 118), seg)[0]
    clip_zero = True
    for t in range(5, 30):
        sub = np.float32(pix[t][30:48, 20 + t : 44 + t]) - np.median(pix[t])
        if np.median(sub) <= 0:
            clip_zero = False
    frames = []
    for i, t in enumerate(range(5, 30)):
        fr = Frame(pix[t], filtered[t], t)
        out = preprocess_frame(fr, (32, 32), Region(20 + t, 30, 24, 18), None, crop, calculate_filtered=False,
                               filtered_norm_limits=(lo, hi), median=np.median(pix[t]), clip_thermals_at_zero=clip_zero)
        r, c = divmod(i, 5)
        assert np.array_equal(out.thermal, oracle[r * 32 : (r + 1) * 32, c * 32 : (c + 1) * 32, 0])
        assert np.array_equal(out.filtered, oracle[r * 32 : (r + 1) * 32, c * 32 : (c + 1) * 32, 1])
        frames.append(out)
    tiled = preprocess_movement(frames, 5, 32, ["thermal", "filtered"])
    assert np.array_equal(tiled, oracle)


def test_nlm_denoise_matches_oracle_and_reference_fixture():
    """cv2.fastNlMeansDenoising on the device, bit for bit: against the C oracle (pinned to cv2) on random and
    structured images of several sizes, and against the reference's own denoised frames where the fixture has them."""
    from classifier_pipeline_b200.ml_tools import imageprocessing as ip
    from oracle import oracle as orc

    rng = np.random.default_rng(21)
    # (330 columns: three column tiles of the quad kernel, 70 rows: three row tiles; tiny images: reflection wraps more than once)
    for H, W in ((120, 160), (70, 330), (37, 53), (16, 16), (5, 7)):
        img = rng.integers(0, 60, size=(H, W)).astype(np.uint8)
        img[H // 3 : H // 3 + max(2, H // 5), W // 4 : W // 4 + max(2, W // 4)] += 150
        assert np.array_equal(ip.fast_nl_means_denoising(img), orc.nlm_denoise(img))
    batch = rng.integers(0, 255, size=(3, 60, 80)).astype(np.uint8)
    got = ip.fast_nl_means_denoising(batch)
    for i in range(3):
        assert np.array_equal(got[i], orc.nlm_denoise(batch[i]))
