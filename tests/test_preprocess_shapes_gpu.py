"""The classifier-input tiling at non-default HyperParams against the numpy oracle: every frame_size the tile kernel takes
(powers of two and not, up to its limit of 64) with 3, 4 and 5 frames per row, regions that exercise each branch of the
resize and the paste, flat crops that take each branch of normalize, short segments with the seeded padding, and the
Interpreter entry points with square_width 4, 6 and frame_size 96."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

W, H = 160, 120
CROP = (1, 1, W - 2, H - 2)
N_FRAMES = 40
FLAT_FRAMES = 4
FLAT_BOX = (30, 30, 12, 12)
FLAT_THERMAL, FLAT_FILTERED = 3000, 37.0


def _frames():
    """Synthetic thermal (uint16) / filtered (float32) frames; the last FLAT_FRAMES hold a constant crop at FLAT_BOX whose
    thermal value is the frame median and whose filtered value is FLAT_FILTERED."""
    from classifier_pipeline_b200.synthetic import make_clip

    pix, _ = make_clip(3, frames=N_FRAMES)
    rng = np.random.default_rng(8)
    flat = np.full((FLAT_FRAMES, H, W), FLAT_THERMAL, np.uint16)
    x, y, w, h = FLAT_BOX
    outside = np.ones((H, W), bool)
    outside[y : y + h, x : x + w] = False
    n_out = int(outside.sum())
    for i in range(FLAT_FRAMES):
        # as many pixels below FLAT_THERMAL as above it, so the frame median is FLAT_THERMAL
        vals = np.concatenate([np.full(n_out // 2, FLAT_THERMAL - 100 - i), np.full(n_out - n_out // 2, FLAT_THERMAL + 100 + i)])
        flat[i][outside] = rng.permutation(vals)
    thermal = np.concatenate([pix, flat])
    filtered = (thermal.astype(np.int64) - pix[0].astype(np.int64)).astype(np.float32)
    filtered[N_FRAMES:, y : y + h, x : x + w] = FLAT_FILTERED
    return thermal, filtered


def _boxes(fs):
    """(x, y, w, h) regions for frame_size fs."""
    boxes = [
        (1, 1, W - 2, H - 2),                         # the whole crop: larger than the tile, touching every side
        (20, 10, min(2 * fs + 9, 130), min(fs + 7, 100)),  # larger than the tile in both dimensions, inside
        (30, 40, fs, fs),                             # exactly the tile
        (50, 50, 1, 1), (60, 20, 1, 37), (5, 70, 41, 1), (1, 1, 1, 1), (158, 118, 1, 1),  # the taps of a 1-D resize
        (70, 40, 5, 16),                              # 5x16: a resized side of k + 0.5 at frame_size 8 and 24
        (20, 60, 2 * fs, 7),                          # height 7 * fs / (2 fs) = 3.5: rounds half to even
        (1, 50, 9, 13), (150, 50, 9, 13), (60, 1, 13, 9), (60, 110, 13, 9),  # touching the left, right, top, bottom
    ]
    if 2 * fs <= H - 2:
        boxes.append((100, 1, 9, 2 * fs))            # width 9 / 2 = 4.5
    return boxes


def _tracks(fs, sw, rng):
    """[(regions, segments)]: one track per box over random frames, segments both shorter and longer than square_width **
    2 and than the frames_per_row * 5 padded samples; plus the flat track."""
    lengths = sorted({1, 2, sw * sw - 1, sw * sw, sw * 5 - 1, sw * 5, 30})
    tracks = []
    for k, (x, y, w, h) in enumerate(_boxes(fs)):
        frames = np.sort(rng.choice(N_FRAMES, 34, replace=False))
        blank = (rng.random(len(frames)) < 0.1) & (np.arange(len(frames)) > 0)
        regions = np.array([[f, x, y, w, h, int(b)] for f, b in zip(frames, blank)], np.int64)
        usable = regions[regions[:, 5] == 0, 0]
        segs = [usable[: lengths[(k + j) % len(lengths)]] for j in (0, 3)]
        tracks.append((regions, segs))
    flat = np.array([[N_FRAMES + i, *FLAT_BOX, 0] for i in range(FLAT_FRAMES)], np.int64)
    tracks.append((flat, [flat[:, 0], flat[:2, 0]]))
    return tracks


@pytest.fixture(scope="module")
def dev():
    import torch

    from classifier_pipeline_b200 import engine

    thermal, filtered = _frames()
    eng = engine.get_engine(None, W, H, 1)
    d_t = torch.from_numpy(thermal.view(np.int16)).cuda().view(torch.uint16)
    d_f = torch.from_numpy(filtered).cuda()
    return eng, thermal, filtered, d_t, d_f


@pytest.mark.parametrize("sw", [3, 4, 5])
@pytest.mark.parametrize("fs", [8, 24, 32, 48, 64])
def test_tiling_matches_oracle(dev, fs, sw):
    from classifier_pipeline_b200.batch import BatchPreprocessor
    from oracle import preprocess_oracle as po

    eng, thermal, filtered, d_t, d_f = dev
    assert np.median(thermal[N_FRAMES]) == FLAT_THERMAL
    tracks = _tracks(fs, sw, np.random.default_rng(fs * 10 + sw))
    for diff_norm in (True, False):
        bp = BatchPreprocessor(eng, frame_size=fs, frames_per_row=sw, diff_norm=diff_norm)
        for crop in (CROP, None):
            res = bp.run(d_t, d_f, tracks, crop, seed=77)
            got = res["segments"].cpu().numpy()
            at = 0
            for regions, segs in tracks:
                want = po.preprocess_track(thermal, filtered, regions, crop, segs, dim=(fs, fs), frames_per_row=sw, seed=77,
                                           diff_norm=diff_norm)
                np.testing.assert_array_equal(got[at : at + len(segs)], want)
                at += len(segs)
            assert got.shape == bp.output_shape(at) == (at, sw * fs, sw * fs, 2)
            # the flat track: thermal all zero after the median (mx == mn == 0), filtered constant (data / max)
            flat = got[at - len(tracks[-1][1]) : at]
            assert not flat[..., 0].any() and np.array_equal(flat[..., 1], np.ones_like(flat[..., 1]))
            if diff_norm:
                norms = bp.tracks_numpy(res["tracks"])[-1]
                assert norms["filtered_min"] == norms["filtered_max"] == FLAT_FILTERED and norms["clip_at_zero"] == 0


def test_inc3_at_a_non_default_size(dev):
    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.batch import BatchPreprocessor
    from oracle import preprocess_oracle as po

    eng, thermal, filtered, d_t, d_f = dev
    fs, sw = 24, 4
    tracks = _tracks(fs, sw, np.random.default_rng(3))
    bp = BatchPreprocessor(eng, frame_size=fs, frames_per_row=sw, preprocess_fn=native.PREPROCESS_INC3)
    got = bp.run(d_t, d_f, tracks, CROP, seed=5)["segments"].cpu().numpy()
    at = 0
    for regions, segs in tracks:
        want = po.preprocess_track(thermal, filtered, regions, CROP, segs, dim=(fs, fs), frames_per_row=sw, seed=5, preprocess_fn="inc3")
        np.testing.assert_array_equal(got[at : at + len(segs)], want)
        at += len(segs)
    assert at == len(got)


# ---------------------------------------------------------------- Interpreter
def _oracle_inputs(clip, track):
    """(thermal, filtered) indexed by frame number and the track's region rows, for the oracle."""
    from classifier_pipeline_b200.ml_tools.interpreter import Interpreter

    numbers = [int(r.frame_number) for r in track.bounds_history]
    n = max(numbers) + 1
    thermal = np.zeros((n, clip.res_y, clip.res_x), np.uint16)
    filtered = np.zeros((n, clip.res_y, clip.res_x), np.float32)
    index = {}
    for f in set(numbers):
        fr = clip.get_frame(f)
        if fr is not None:
            thermal[f], filtered[f], index[f] = fr.thermal, fr.filtered, f
    return thermal, filtered, Interpreter._region_rows(track, index)


def test_interpreter_square_width_4_frame_size_48_matches_oracle():
    from classifier_pipeline_b200.ml_tools.interpreter import HyperParams, Interpreter
    from oracle import preprocess_oracle as po
    from tests.test_classify_inputs_gpu import _parse

    ref = _parse(["synth1_raw"], False, False)[0]
    dev = _parse(["synth1_raw"], True, False)[0]
    assert ref.tracks and [t.get_id() for t in ref.tracks] == [t.get_id() for t in dev.tracks]
    interp = Interpreter(HyperParams(square_width=4, frame_size=48), seed=1234)
    c = ref.crop_rectangle
    crop = (c.x, c.y, c.width, c.height)
    np.random.seed(11)
    got_clips = interp.preprocess_clips([dev])[0]
    np.random.seed(11)
    n_checked = 0
    for track, (_, got_clips_data, _) in zip(ref.tracks, got_clips):
        segments = list(interp.frames_for_prediction(ref, track))
        _, got, _ = interp.preprocess_segments(ref, track, segments)
        thermal, filtered, regions = _oracle_inputs(ref, track)
        want = po.preprocess_track(thermal, filtered, regions, crop, [s.frame_indices for s in segments], dim=(48, 48), frames_per_row=4,
                                   seed=1234)
        assert got.shape == got_clips_data.shape == (len(segments), 192, 192, 2)
        np.testing.assert_array_equal(got, want)
        np.testing.assert_array_equal(got_clips_data, want)
        n_checked += len(segments)
    assert n_checked


def test_interpreter_rejects_square_width_6_and_frame_size_96():
    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.ml_tools.interpreter import HyperParams, Interpreter
    from tests.test_classify_inputs_gpu import _parse

    dev = _parse(["synth1_raw"], True, False)[0]
    track = max(dev.tracks, key=lambda t: len(t.bounds_history))  # (a track with segments: without one nothing launches)
    six = Interpreter(HyperParams(square_width=6), seed=1234)
    with pytest.raises(ValueError, match="square_width"):
        six.preprocess(dev, track)
    with pytest.raises(ValueError, match="square_width"):
        six.preprocess_clips([dev])
    big = Interpreter(HyperParams(frame_size=96), seed=1234)
    with pytest.raises(native.NativeError, match="64"):
        big.preprocess(dev, track)
    with pytest.raises(native.NativeError, match="64"):
        big.preprocess_clips([dev])
