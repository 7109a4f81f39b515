"""The device resize, bit for bit: resize_pad_kernel through ml_tools.imageprocessing (resize_cv, resize_and_pad) against
live cv2.resize on the designed grid of tests/resize_grid.py, and segment_tiles_kernel (BatchPreprocessor) against the
numpy oracle, whose resize is held to cv2 bit for bit in tests/test_resize_cv2.py, on thin regions and real-valued
filtered frames at every even frame_size.  No tolerance anywhere: -0.0 and 0.0 count as different."""
import numpy as np
import pytest

from oracle import preprocess_oracle as po
from tests import resize_grid as rg

pytestmark = pytest.mark.gpu

cv2 = pytest.importorskip("cv2")


@pytest.mark.parametrize("geometry", list(rg.GEOMETRIES))
@pytest.mark.parametrize("interpolation", ["linear", "nearest"])
def test_resize_cv_matches_cv2(interpolation, geometry):
    from classifier_pipeline_b200.ml_tools import imageprocessing as ip

    ours, flag = {"linear": (ip.INTER_LINEAR, cv2.INTER_LINEAR), "nearest": (ip.INTER_NEAREST, cv2.INTER_NEAREST)}[interpolation]
    bad = []
    for kind in rg.DATA:
        for sw, sh, dw, dh, src in rg.cases(geometry, kind):
            if not rg.same_bits(ip.resize_cv(src, (dw, dh), interpolation=ours), cv2.resize(src, (dw, dh), interpolation=flag)):
                bad.append((kind, sw, sh, dw, dh))
    assert not bad, "{} cases differ from cv2.resize, e.g. (data, sw, sh, dw, dh) {}".format(len(bad), bad[:5])


def _cv2_resize_and_pad(frame, dim, region, crop, keep_edge, pad, interpolation):
    """resize_and_pad (imageprocessing.py:11-70) composed from the oracle's size and offsets and cv2.resize itself."""
    h, w = frame.shape
    fw, fh = po.resized_size(w, h, dim)
    out = np.full(dim, frame.min() if pad is None else pad, dtype=np.float32)
    ox, oy = po.paste_offsets(fw, fh, dim, region, crop, keep_edge)
    out[oy : oy + fh, ox : ox + fw] = cv2.resize(frame, (fw, fh), interpolation=interpolation)
    return out


CROP = (1, 1, 158, 118)


def _regions(rng):
    """(x, y, w, h) inside CROP: thin, 1x1, larger than the tile, and touching each side of the crop and two corners."""
    out = [(50, 50, 1, 1), (60, 20, 1, 37), (5, 70, 41, 1), (1, 1, 1, 1), (158, 118, 1, 1), (1, 30, 1, 90), (20, 118, 100, 1),
           (1, 40, 9, 13), (150, 40, 9, 13), (60, 1, 13, 9), (60, 110, 13, 9), (1, 1, 158, 118), (140, 100, 19, 19), (70, 40, 5, 16)]
    for _ in range(16):
        w, h = int(rng.integers(1, 100)), int(rng.integers(1, 100))
        out.append((int(rng.integers(1, 159 - w + 1)), int(rng.integers(1, 119 - h + 1)), w, h))
    return out


@pytest.mark.parametrize("kind", ["u16", "real", "signed_zero"])
@pytest.mark.parametrize("size", [8, 24, 32, 48, 64])
def test_resize_and_pad_matches_cv2(size, kind):
    from classifier_pipeline_b200.ml_tools import imageprocessing as ip
    from classifier_pipeline_b200.ml_tools.rectangle import Rectangle

    rng = np.random.default_rng(size)
    crop = Rectangle(*CROP)
    dim = (size, size)
    regions = _regions(rng)
    n = 0
    for i, (x, y, w, h) in enumerate(regions):
        src = rg.make_source(kind, h, w, seed=(size, i))
        for keep_edge in (True, False):
            for pad in (None, -7.25):
                for ours, flag in ((ip.INTER_LINEAR, cv2.INTER_LINEAR), (ip.INTER_NEAREST, cv2.INTER_NEAREST)):
                    got = ip.resize_and_pad(src, dim, Rectangle(x, y, w, h), crop, keep_edge=keep_edge, pad=pad, interpolation=ours)
                    want = _cv2_resize_and_pad(src, dim, (x, y, w, h), CROP, keep_edge, pad, flag)
                    assert rg.same_bits(got, want), ((x, y, w, h), keep_edge, pad, ours)
                    oracle = po.resize_and_pad(src, dim, (x, y, w, h), CROP, keep_edge=keep_edge, pad=pad,
                                               interpolation=po.INTER_LINEAR if flag == cv2.INTER_LINEAR else po.INTER_NEAREST)
                    assert rg.same_bits(oracle, want), ((x, y, w, h), keep_edge, pad, ours)
                    n += 1
    assert n == 2 * 2 * 2 * len(regions)


# ---------------------------------------------------------------- the tile kernel
W, H = 160, 120
N_FRAMES = 24


@pytest.fixture(scope="module")
def frames():
    """Thermal (uint16) frames and real-valued filtered (fp32) frames of the same clip, as host and device arrays."""
    import torch

    from classifier_pipeline_b200 import engine
    from classifier_pipeline_b200.synthetic import make_clip

    thermal, _ = make_clip(5, frames=N_FRAMES)
    rng = np.random.default_rng(21)
    filtered = ((thermal.astype(np.int64) - thermal[0].astype(np.int64)) + rng.standard_normal(thermal.shape) * 3.7).astype(np.float32)
    eng = engine.get_engine(None, W, H, 1)
    d_t = torch.from_numpy(thermal.view(np.int16)).cuda().view(torch.uint16)
    return eng, thermal, filtered, d_t, torch.from_numpy(filtered).cuda()


def _tile_boxes(fs):
    """Thin regions (1 x k and k x 1, growing and shrinking into the tile, and 1 x 1), a region exactly the tile's size
    (the copy), and 2-D regions larger and smaller than the tile, two of them touching the crop's sides."""
    ks = sorted({2, 3, max(fs // 2, 2), fs + 1, 2 * fs + 1, 100})
    boxes = [(50, 50, 1, 1), (1, 1, 1, 1), (158, 118, 1, 1)]
    boxes += [(40, 10, 1, k) for k in ks if k <= 100] + [(10, 60, k, 1) for k in ks]
    boxes += [(1, 20, 1, 17), (30, 118, 23, 1)]
    boxes += [(30, 30, fs, min(fs, 100)), (20, 10, min(2 * fs + 9, 130), min(fs + 7, 100)), (70, 40, 5, 16), (1, 50, 9, 13), (60, 110, 13, 9)]
    return boxes


@pytest.mark.parametrize("fs", list(range(2, 65, 2)))
def test_tiles_match_oracle_exactly(frames, fs):
    from classifier_pipeline_b200.batch import BatchPreprocessor

    eng, thermal, filtered, d_t, d_f = frames
    rng = np.random.default_rng(fs)
    tracks = []
    for x, y, w, h in _tile_boxes(fs):
        fr = np.sort(rng.choice(N_FRAMES, 9, replace=False))
        regions = np.array([[f, x, y, w, h, 0] for f in fr], np.int64)
        tracks.append((regions, [fr[:9], fr[:4]]))
    for diff_norm in (True, False):
        bp = BatchPreprocessor(eng, frame_size=fs, frames_per_row=3, diff_norm=diff_norm)
        for crop in ((1, 1, W - 2, H - 2), None):
            got = bp.run(d_t, d_f, tracks, crop, seed=3)["segments"].cpu().numpy()
            at = 0
            for regions, segs in tracks:
                want = po.preprocess_track(thermal, filtered, regions, crop, segs, dim=(fs, fs), frames_per_row=3, seed=3,
                                           diff_norm=diff_norm)
                assert rg.same_bits(got[at : at + len(segs)], want), (tuple(regions[0, 1:5]), diff_norm, crop)
                at += len(segs)
            assert at == len(got)
