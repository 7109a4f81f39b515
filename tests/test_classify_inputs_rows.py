"""Row bookkeeping of classifier inputs made from an extraction's device buffers (no GPU needed): frame numbers map to the
right thermal, filtered and median rows in both input layouts, and the flat tables of a multi-clip batch are the per-clip
tables with the rows shifted."""
from types import SimpleNamespace

import numpy as np
import pytest

from classifier_pipeline_b200.batch import BatchPreprocessor, ClipDeviceFrames, linear_clips, tracked_row_map
from classifier_pipeline_b200.ml_tools.interpreter import Interpreter


def _host_layout(counts):
    """The records ClipTrackExtractor._run_batch builds for host-assembled frames: [init][tracked frames] per clip."""
    clips = linear_clips(counts, 0, 0)
    pos = 0
    for i, n in enumerate(counts):
        clips["init_offset"][i] = pos
        clips["frame_offset"][i] = pos + 1
        pos += 1 + n
    return clips, pos


def _device_layout(file_frames, skips):
    """The records for device-decoded CPTV: every frame of the file is an input row, the first one initialises the
    background and ``skip`` leading background frames are not tracked."""
    counts = [f - s for f, s in zip(file_frames, skips)]
    first = np.concatenate([[0], np.cumsum(file_frames)[:-1]])
    clips = linear_clips(counts, 0, 0)
    clips["init_offset"] = first
    clips["frame_offset"] = first + np.asarray(skips)
    return clips, int(sum(file_frames))


def _handles(clips):
    return [ClipDeviceFrames(None, c["frame_offset"], c["out_offset"], c["n_frames"]) for c in clips]


def test_rows_of_host_assembled_layout():
    counts = [3, 5, 2]
    clips, n_input = _host_layout(counts)
    row_map = tracked_row_map(clips, n_input)
    # input rows: init 0, frames 1-3 | init 4, frames 5-9 | init 10, frames 11-12; output rows 0-2 | 3-7 | 8-9
    assert row_map.tolist() == [-1, 0, 1, 2, -1, 3, 4, 5, 6, 7, -1, 8, 9]
    h = _handles(clips)
    assert [(x.thermal_row0, x.median_row0, x.filtered_row0, x.n_frames) for x in h] == [(1, 1, 0, 3), (5, 5, 3, 5), (11, 11, 8, 2)]
    for x in h:
        for n in range(x.n_frames):
            assert row_map[x.thermal_row0 + n] == x.filtered_row0 + n


def test_rows_of_device_decoded_layout_with_leading_background_frames():
    # three files of 6, 4 and 5 frames; the first and last start with 2 and 1 background frames
    clips, n_input = _device_layout([6, 4, 5], [2, 0, 1])
    row_map = tracked_row_map(clips, n_input)
    assert row_map.tolist() == [-1, -1, 0, 1, 2, 3, 4, 5, 6, 7, -1, 8, 9, 10, 11]
    h = _handles(clips)
    assert [(x.thermal_row0, x.median_row0, x.filtered_row0, x.n_frames) for x in h] == [(2, 2, 0, 4), (6, 6, 4, 4), (11, 11, 8, 4)]
    # without leading background frames the init frame is tracked frame 0
    clips, n_input = _device_layout([3, 2], [0, 0])
    assert tracked_row_map(clips, n_input).tolist() == [0, 1, 2, 3, 4]


def _track(tid, regions):
    bounds = [SimpleNamespace(frame_number=n, x=x, y=y, width=w, height=h, blank=b) for n, x, y, w, h, b in regions]
    return SimpleNamespace(bounds_history=bounds, get_id=lambda: tid)


def _clip(cid, row0, n_frames, tracks, first_kept=0):
    clip = SimpleNamespace(tracks=tracks, get_id=lambda: cid)
    clip.device_frames = ClipDeviceFrames(None, row0, 0, n_frames, first_kept=first_kept)
    return clip


def _random_clip(rng, cid, row0, n_frames):
    tracks, jobs = [], []
    for t in range(int(rng.integers(1, 4))):
        start = int(rng.integers(0, n_frames - 8))
        length = int(rng.integers(6, n_frames - start + 1))
        regions = []
        for n in range(start, start + length):
            w, h = int(rng.integers(1, 30)), int(rng.integers(1, 30))
            regions.append((n, int(rng.integers(0, 160 - w + 1)), int(rng.integers(0, 120 - h + 1)), w, h, bool(rng.random() < 0.15)))
        track = _track(t + 1, regions)
        usable = [r[0] for r in regions if not r[5]]
        segs = [SimpleNamespace(frame_indices=np.sort(rng.choice(usable, size=min(len(usable), int(rng.integers(1, 30))), replace=False)))
                for _ in range(int(rng.integers(0, 4)))]
        tracks.append(track)
        jobs.append((track, segs))
    return _clip(cid, row0, n_frames, tracks), jobs


def test_flat_tables_of_a_batch_are_the_per_clip_tables_shifted():
    rng = np.random.default_rng(7)
    interp = Interpreter(seed=3)
    bp = BatchPreprocessor(SimpleNamespace(torch=None, device=None, width=160, height=120))
    row0s = [1, 60, 101, 190]
    clip_jobs = [_random_clip(rng, i, r0, 40) for i, r0 in enumerate(row0s)]

    def tables_of(cj, shift):
        tables = []
        for clip, jobs in cj:
            h = clip.device_frames
            if not shift:
                h = ClipDeviceFrames(None, 0, 0, h.n_frames, h.first_kept)
            tables.extend(interp._tables(clip, jobs, interp._device_index(h, jobs)))
        return tables

    lim, smp, seg, seg_track = bp.build_tables(tables_of(clip_jobs, True), seed=3)
    # per clip, in the clip's own frame numbering
    at_t = at_s = at_l = 0
    smp_base = 0
    for clip, jobs in clip_jobs:
        l1, s1, g1, k1 = bp.build_tables(tables_of([(clip, jobs)], False), seed=3)
        shift = clip.device_frames.thermal_row0
        lsl = lim[at_l : at_l + len(l1)]
        assert np.array_equal(lsl["frame"], l1["frame"] + shift)
        for f in ("x", "y", "width", "height"):
            assert np.array_equal(lsl[f], l1[f]) and np.array_equal(smp[at_s : at_s + len(s1)][f], s1[f])
        assert np.array_equal(lsl["track"], l1["track"] + at_t)
        assert np.array_equal(smp[at_s : at_s + len(s1)]["frame"], s1["frame"] + shift)
        assert np.array_equal(smp[at_s : at_s + len(s1)]["track"], s1["track"] + at_t)
        assert np.array_equal(seg[smp_base : smp_base + len(g1)], g1 + at_s)
        assert np.array_equal(seg_track[smp_base : smp_base + len(k1)], k1 + at_t)
        at_t += len(jobs)
        at_s += len(s1)
        at_l += len(l1)
        smp_base += len(g1)
    assert (at_l, at_s, smp_base) == (len(lim), len(smp), len(seg))


def test_segment_frame_outside_the_clip_raises_like_the_upload_path():
    interp = Interpreter(seed=3)
    track = _track(1, [(n, 10, 10, 5, 5, False) for n in range(8)])
    clip = _clip(1, 4, 6, [track])  # frames 6 and 7 were never tracked in this clip
    seg = SimpleNamespace(frame_indices=np.arange(2, 8))
    index = interp._device_index(clip.device_frames, [(track, [seg])])
    assert index == {n: 4 + n for n in range(6)}
    with pytest.raises(Exception, match="can't get frame 6"):
        interp._tables(clip, [(track, [seg])], index)


def test_released_handle_raises():
    clip = _clip(1, 0, 4, [])
    clip.device_frames.batch = object()
    assert Interpreter._device_batch(clip) is clip.device_frames.batch
    clip.device_frames.release()
    assert not clip.device_frames.live
    with pytest.raises(Exception, match="released"):
        Interpreter._device_batch(clip)
    assert Interpreter._device_batch(SimpleNamespace(device_frames=None)) is None


def test_uint16_frame_numbers_map_past_65535_rows():
    """Tracks loaded from metadata carry np.uint16 frame numbers: the thermal row must not wrap at 65 536 (a batch of
    73 clips x 900 frames already has more input rows)."""
    import warnings

    interp = Interpreter(seed=3)
    frames = [7990, 8000, 8001]
    track = _track(1, [(np.uint16(n), 10, 10, 5, 5, False) for n in frames])
    clip = _clip(1, 60000, 9000, [track])
    seg = SimpleNamespace(frame_indices=np.asarray(frames, np.uint16))
    with warnings.catch_warnings():
        warnings.simplefilter("error")  # (numpy reports uint16 overflow only as a RuntimeWarning)
        index = interp._device_index(clip.device_frames, [(track, [seg])])
        assert index == {n: 60000 + n for n in frames}
        [(regions, seg_rows)] = interp._tables(clip, [(track, [seg])], index)
    assert regions[:, 0].tolist() == [67990, 68000, 68001]
    assert seg_rows[0].tolist() == [67990, 68000, 68001]
    clip = _clip(1, 70000, 9000, [track])  # (a row0 above 65 535 used to raise OverflowError)
    assert interp._device_index(clip.device_frames, [(track, [])]) == {n: 70000 + n for n in frames}


def test_frames_evicted_by_max_frames_are_missing_like_the_upload_path():
    """A frame buffer with max_frames keeps the last max_frames frames; the handle's first_kept hides the earlier ones."""
    interp = Interpreter(seed=3)
    track = _track(1, [(n, 10, 10, 5, 5, False) for n in range(10)])
    clip = _clip(1, 4, 10, [track], first_kept=6)  # 10 tracked frames, max_frames 4
    index = interp._device_index(clip.device_frames, [(track, [])])
    assert index == {n: 4 + n for n in range(6, 10)}
    [(regions, _)] = interp._tables(clip, [(track, [])], index)
    # evicted frames become rows without a frame, as _region_rows makes them for frames clip.get_frame cannot supply
    assert regions[:6, 0].tolist() == [-1] * 6 and regions[:6, 5].tolist() == [1] * 6
    assert regions[6:, 0].tolist() == [10, 11, 12, 13]
    with pytest.raises(Exception, match="can't get frame 5"):
        interp._tables(clip, [(track, [SimpleNamespace(frame_indices=np.arange(5, 10))])], index)
