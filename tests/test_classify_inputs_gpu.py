"""Classifier inputs straight from an extraction's device buffers: the cpt_preprocess_* entry points given the extraction's
filtered rows, frame medians and frame records against the same entry points on repacked frames, and
ClipTrackExtractor.parse_clips(keep_on_device=True) + Interpreter.preprocess_clips against parse_clips + per-clip
Interpreter.preprocess."""
import json
import os

import numpy as np
import pytest

from tests import helpers
from tests.tracking_helpers import MemReader

pytestmark = pytest.mark.gpu

W, H = 160, 120
CLIP_NAMES = ["possum", "hedgehog", "synth0_raw", "synth1_raw", "synth2_raw", "synth3_raw"]


# ---------------------------------------------------------------- kernel level
def _layout(rng):
    """Random uint16 frames laid out as an extraction's input: per clip an init frame, 0-2 leading background frames,
    then the tracked frames; the filtered rows are the tracked frames back to back.  Returns (thermal, filtered, row_map,
    clip (thermal_row0, n_frames) list)."""
    counts = [7, 1, 12, 5, 9]
    rows, clips, out = [], [], 0
    for n in counts:
        lead = 1 + int(rng.integers(0, 3))
        start = sum(len(r) for r in rows) + lead
        base = int(rng.integers(2000, 9000))
        block = rng.integers(base, base + 1500, size=(lead + n, H, W)).astype(np.uint16)
        rows.append(block)
        clips.append((start, n))
        out += n
    thermal = np.concatenate(rows)
    # a few frames with a wide value range (median.cuh's radix path)
    for r in rng.choice(len(thermal), 4, replace=False):
        thermal[r] = rng.integers(0, 65535, size=(H, W)).astype(np.uint16)
    row_map = np.full(len(thermal), -1, np.int64)
    o = 0
    for start, n in clips:
        row_map[start : start + n] = np.arange(o, o + n)
        o += n
    filtered = rng.integers(-300, 700, size=(out, H, W)).astype(np.float32)
    return thermal, filtered, row_map, clips


def _random_region(rng):
    kind = rng.integers(0, 5)
    if kind == 0:
        return int(rng.integers(0, W)), int(rng.integers(0, H)), 1, 1
    if kind == 1:
        return 0, 0, W, H
    if kind == 2:  # touching an edge
        w, h = int(rng.integers(1, 60)), int(rng.integers(1, 50))
        return (W - w if rng.random() < 0.5 else 0), int(rng.integers(0, H - h + 1)), w, h
    w, h = int(rng.integers(1, 50)), int(rng.integers(1, 40))
    return int(rng.integers(0, W - w + 1)), int(rng.integers(0, H - h + 1)), w, h


def _tracks(rng, clips):
    """Per track (regions [thermal row, x, y, w, h, blank], segments of thermal rows)."""
    tracks = []
    for start, n in clips:
        for _ in range(int(rng.integers(1, 4))):
            regs = []
            for t in range(n):
                x, y, w, h = _random_region(rng)
                regs.append([start + t, x, y, w, h, int(n > 1 and rng.random() < 0.1)])
            regs = np.asarray(regs, np.int64)
            usable = regs[regs[:, 5] == 0, 0]
            segs = [np.sort(rng.choice(usable, size=int(rng.integers(1, len(usable) + 1)), replace=False))
                    for _ in range(int(rng.integers(1, 4)))] if len(usable) else []
            tracks.append((regs, segs))
    return tracks


@pytest.fixture(scope="module")
def layout():
    import torch

    from classifier_pipeline_b200 import engine, native

    rng = np.random.default_rng(2024)
    thermal, filtered, row_map, clips = _layout(rng)
    tracks = _tracks(rng, clips)
    eng = engine.get_engine(None, W, H, 1)
    eng.ctx.use_torch_stream()
    d_thermal = torch.from_numpy(thermal.view(np.int16)).cuda().view(torch.uint16)
    d_filtered = torch.from_numpy(filtered).cuda()
    d_med = torch.empty(len(thermal), dtype=torch.float32, device="cuda")
    eng.ctx.frame_medians(d_thermal, len(thermal), d_med)
    # the frame records an extraction with CPT_CLIP_FRAME_STATS writes, per filtered row
    info = np.zeros(len(filtered), native.INFO_DTYPE)
    tracked = row_map >= 0
    info["thermal_min"][row_map[tracked]] = thermal[tracked].reshape(tracked.sum(), -1).min(1)
    info["thermal_max"][row_map[tracked]] = thermal[tracked].reshape(tracked.sum(), -1).max(1)
    d_info = torch.from_numpy(info.view(np.uint8)).cuda()
    # the repacked copy the existing entry points take: thermal row of every tracked frame moved to its filtered row
    packed = np.empty((len(filtered), H, W), np.uint16)
    packed[row_map[tracked]] = thermal[tracked]
    d_packed = torch.from_numpy(packed.view(np.int16)).cuda().view(torch.uint16)
    return dict(eng=eng, tracks=tracks, row_map=row_map, d_thermal=d_thermal, d_filtered=d_filtered, d_med=d_med, d_info=d_info,
                d_packed=d_packed)


@pytest.mark.parametrize("variant", ["default", "inc3", "per_tile", "thermal_diff_norm", "tdn_per_tile", "rows_only"])
def test_ex_entry_points_equal_the_existing_ones_on_repacked_frames(layout, variant):
    import torch

    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.batch import BatchPreprocessor

    L = layout
    kw = dict(preprocess_fn=native.PREPROCESS_INC3 if variant == "inc3" else 0, diff_norm=variant not in ("per_tile", "tdn_per_tile"),
              thermal_diff_norm=variant in ("thermal_diff_norm", "tdn_per_tile"))
    bp = BatchPreprocessor(L["eng"], **kw)
    lim, smp, seg, _ = bp.build_tables(L["tracks"], seed=5)
    crop = (1, 1, W - 2, H - 2)
    stats = {} if variant == "rows_only" else dict(frame_medians=L["d_med"], frame_info=L["d_info"])
    new = bp.run_tables(L["d_thermal"], L["d_filtered"], lim, smp, seg, len(L["tracks"]), crop, row_map=L["row_map"], **stats)
    lim_old, smp_old = lim.copy(), smp.copy()
    lim_old["frame"] = L["row_map"][lim["frame"]]
    smp_old["frame"] = L["row_map"][smp["frame"]]
    assert (lim_old["frame"] >= 0).all() and (smp_old["frame"] >= 0).all()
    old = bp.run_tables(L["d_packed"], L["d_filtered"], lim_old, smp_old, seg, len(L["tracks"]), crop)
    torch.cuda.synchronize()
    assert np.array_equal(new["segments"].cpu().numpy(), old["segments"].cpu().numpy())
    assert np.array_equal(new["tracks"].cpu().numpy(), old["tracks"].cpu().numpy())
    s_new = new["samples"].cpu().numpy().view(native.SAMPLE_DTYPE)
    s_old = old["samples"].cpu().numpy().view(native.SAMPLE_DTYPE)
    assert np.array_equal(s_new["median"], s_old["median"])
    # cpt_frame_medians == the medians cpt_preprocess_medians writes, bit for bit
    assert np.array_equal(L["d_med"].cpu().numpy()[smp["frame"]].view(np.uint32), s_old["median"].view(np.uint32))
    assert len(seg) >= 5
    t = BatchPreprocessor.tracks_numpy(new["tracks"])
    assert (t["clip_at_zero"] == 0).any()
    if kw["thermal_diff_norm"]:
        assert (t["has_thermal_limits"] == 1).all()


# ---------------------------------------------------------------- API level
def _synth_pix():
    from classifier_pipeline_b200.synthetic import make_clip

    return {n: make_clip(*helpers.SYNTH[n]) for n in CLIP_NAMES if n in helpers.SYNTH}


def _path(name):
    return os.path.join(helpers.GOLDEN, "clips", name + ".cptv") if name in ("possum", "hedgehog") else name


def _parse(names, keep_on_device, device_decode, denoise=False, **kw):
    from classifier_pipeline_b200.config import Config
    from classifier_pipeline_b200.cptv import CptvReader
    from classifier_pipeline_b200.track.clip import Clip
    from classifier_pipeline_b200.track.cliptrackextractor import ClipTrackExtractor

    config = Config.get_defaults()
    config.tracking["thermal"].denoise = denoise
    ext = ClipTrackExtractor(config.tracking, False, cache_to_disk=False, **kw)
    if not device_decode:
        pix = _synth_pix()
        ext.reader_factory = lambda path: MemReader(*pix[path]) if path in pix else CptvReader(path)
    clips = [Clip(config.tracking["thermal"], _path(n)) for n in names]
    ext.parse_clips(clips, keep_on_device=keep_on_device)
    return clips


INTERPRETERS = {
    "default": lambda I, HP, inc3: I(HP(), seed=1234),
    "thermal_diff_norm": lambda I, HP, inc3: I(HP(thermal_diff_norm=True), seed=1234),
    "no_diff_norm": lambda I, HP, inc3: I(HP(diff_norm=False), seed=1234),
    "tdn_no_diff_norm": lambda I, HP, inc3: I(HP(thermal_diff_norm=True, diff_norm=False), seed=1234),
    "three_channels": lambda I, HP, inc3: I(HP(channels=["thermal", "filtered", "filtered"]), seed=1234),
    "inc3": lambda I, HP, inc3: I(HP(), preprocess_fn=inc3, seed=1234),
    "host_fn": lambda I, HP, inc3: I(HP(), preprocess_fn=lambda x: x * np.float32(0.5) + np.float32(3.0), seed=1234),
}


def _interpreters():
    from classifier_pipeline_b200.ml_tools.interpreter import HyperParams, Interpreter, inc3_preprocess

    return {k: f(Interpreter, HyperParams, inc3_preprocess) for k, f in INTERPRETERS.items()}


def _assert_same(got, want):
    assert len(got) == len(want)
    for (f1, d1, m1), (f2, d2, m2) in zip(got, want):
        assert len(f1) == len(f2) and all(np.array_equal(a, b) for a, b in zip(f1, f2))
        assert d1.dtype == d2.dtype and np.array_equal(d1, d2)
        assert list(m1) == list(m2)


def _compare(dev_clips, ref_clips, interps, args=None):
    args = args or {}
    n_segments = 0
    for name, interp in interps.items():
        # (the masked segment selection shuffles with the global generator, as the reference does)
        np.random.seed(11)
        got = interp.preprocess_clips(dev_clips, **args)
        assert len(got) == len(ref_clips)
        np.random.seed(11)
        want_all = [[interp.preprocess(ref, t, **args) for t in ref.tracks] for ref in ref_clips]
        for g, want in zip(got, want_all):
            _assert_same(g, want)
            n_segments += sum(len(d) for _, d, _ in want)
        if name in ("default", "thermal_diff_norm", "tdn_no_diff_norm"):
            for dc, rc in zip(dev_clips, ref_clips):
                for td, tr in zip(dc.tracks, rc.tracks):
                    a, b = interp.get_limits(dc, td), interp.get_limits(rc, tr)
                    assert repr(a) == repr(b)
    assert n_segments > 0


@pytest.mark.parametrize("layout_kind", ["host_assembled", "device_decoded"])
@pytest.mark.parametrize("keep_frames", [True, False])
def test_preprocess_clips_equals_per_clip_preprocess(layout_kind, keep_frames):
    device_decode = layout_kind == "device_decoded"
    names = ["possum", "hedgehog"] if device_decode else CLIP_NAMES
    ref = _parse(names, False, device_decode)
    dev = _parse(names, True, device_decode, keep_frames=keep_frames)
    for d, r in zip(dev, ref):
        assert [t.get_id() for t in d.tracks] == [t.get_id() for t in r.tracks]
        assert d.device_frames is not None and d.device_frames.live
        if not keep_frames:
            assert len(d.frame_buffer.frames) == 0
            assert d.frame_buffer.current_frame.filtered is None and d.frame_buffer.current_frame.mask is None
    assert sum(len(c.tracks) for c in ref) >= 3
    _compare(dev, ref, _interpreters())
    # preprocess_tracks / preprocess_segments on a clip with a handle use the device rows as well
    interp = _interpreters()["default"]
    for d, r in zip(dev, ref):
        for td, tr in zip(d.tracks, r.tracks):
            segs = list(interp.frames_for_prediction(r, tr))
            _assert_same(interp.preprocess_tracks(d, [(td, segs)]), interp.preprocess_tracks(r, [(tr, segs)]))


def test_device_decoded_clip_with_leading_background_frames():
    """possum.cptv starts with background frames: the thermal rows of the device-decoded input are shifted against the
    filtered rows, and the handle says so."""
    dev = _parse(["possum"], True, True)
    h = dev[0].device_frames
    assert h.thermal_row0 > 0 and h.filtered_row0 == 0
    assert h.batch.row_map[h.thermal_row0] == 0 and (h.batch.row_map[: h.thermal_row0] == -1).all()


def test_preprocess_clips_matches_the_reference_fixtures():
    """pre_possum.npz / pre_possum_opts.npz (what the unmodified reference produced) through preprocess_clips."""
    from classifier_pipeline_b200.ml_tools.interpreter import HyperParams, Interpreter
    from tests.test_preprocess_oracle import ATOL, OPTION_SETS, RTOL

    clip = _parse(["possum"], True, True, keep_frames=False)[0]
    tracks = list(clip.tracks) + [t for _, t in clip.filtered_tracks if len(t) >= 8]
    for tag in ["default"] + list(OPTION_SETS):
        pre = np.load(os.path.join(helpers.GOLDEN, "pre_possum.npz" if tag == "default" else "pre_possum_opts.npz"))
        meta = json.loads(str(pre["meta"]))
        interp = Interpreter(HyperParams({} if tag == "default" else OPTION_SETS[tag]), seed=1234)
        assert meta["tracks"]
        for entry in meta["tracks"]:
            ti = entry["index"]
            track = tracks[ti]
            assert track.get_id() == entry["id"]
            seg_frames = [pre["t{}_seg{}".format(ti, s)] for s in range(entry["segments"])]
            clip.tracks = [track]
            [[(_, data, _)]] = interp.preprocess_clips([clip], segment_frames=seg_frames)
            expected = pre["t{}_out".format(ti) if tag == "default" else "t{}_out_{}".format(ti, tag)]
            np.testing.assert_allclose(data, expected, rtol=RTOL, atol=ATOL)


def test_preprocess_clips_with_denoise():
    from classifier_pipeline_b200 import native

    if not native.HAS_NLM:
        pytest.skip("no NLM kernel in this build")
    names = ["possum", "synth1_raw"]
    ref = _parse(names, False, False, denoise=True)
    dev = _parse(names, True, False, denoise=True, keep_frames=False)
    interps = _interpreters()
    _compare(dev, ref, {k: interps[k] for k in ("default", "thermal_diff_norm")})


def test_released_handle_raises_and_mixed_lists_work():
    names = ["synth0_raw", "synth2_raw", "synth3_raw"]
    ref = _parse(names, False, False)
    dev = _parse(names, True, False)
    plain = _parse(["synth1_raw"], False, False)
    interp = _interpreters()["default"]
    mixed = [dev[0], plain[0], dev[1], dev[2]]
    np.random.seed(3)
    got = interp.preprocess_clips(mixed)
    np.random.seed(3)
    want = [[interp.preprocess(c, t) for t in c.tracks] for c in [ref[0], plain[0], ref[1], ref[2]]]
    for g, w in zip(got, want):
        _assert_same(g, w)
    track = next(t for t in dev[1].tracks)
    dev[1].device_frames.release()
    with pytest.raises(Exception, match="released"):
        interp.preprocess(dev[1], track)
    with pytest.raises(Exception, match="released"):
        interp.preprocess_clips([dev[0], dev[1]])
    # the other clips of the batch still hold the buffers
    np.random.seed(4)
    got = interp.preprocess_clips([dev[2]])[0]
    np.random.seed(4)
    _assert_same(got, [interp.preprocess(ref[2], t) for t in ref[2].tracks])


def test_max_frames_hides_evicted_frames_like_the_frame_buffer():
    """With max_frames the frame buffer keeps the last max_frames frames: the handle exposes the same frames, a segment
    over kept frames gives the same tiles and a segment naming an evicted frame raises the same exception."""
    from types import SimpleNamespace

    names = ["synth0_raw", "synth1_raw"]
    ref = _parse(names, False, False, max_frames=60)
    dev = _parse(names, True, False, max_frames=60)
    interp = _interpreters()["default"]
    kept_checked = evicted_checked = 0
    for d, r in zip(dev, ref):
        h = d.device_frames
        assert h.n_frames > 60 and h.first_kept == h.n_frames - 60
        assert r.get_frame(h.first_kept - 1) is None and r.get_frame(h.first_kept) is not None
        for td, tr in zip(d.tracks, r.tracks):
            numbers = [int(b.frame_number) for b in tr.bounds_history if not b.blank and b.width > 0 and b.height > 0]
            kept = [n for n in numbers if n >= h.first_kept][:25]
            evicted = [n for n in numbers if n < h.first_kept]
            if kept:
                seg = [SimpleNamespace(frame_indices=np.asarray(kept), mass=1)]
                _assert_same([interp.preprocess_segments(d, td, seg)], [interp.preprocess_segments(r, tr, seg)])
                kept_checked += 1
            if evicted:
                seg = [SimpleNamespace(frame_indices=np.asarray(evicted[-1:] + kept[:3]), mass=1)]
                for clip, track in ((r, tr), (d, td)):
                    with pytest.raises(Exception, match="can't get frame {}".format(evicted[-1])):
                        interp.preprocess_segments(clip, track, seg)
                evicted_checked += 1
    assert kept_checked and evicted_checked
