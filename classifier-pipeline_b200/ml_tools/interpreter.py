"""The preprocessing half of ``ml_tools.interpreter.Interpreter`` on the B200
(ml_tools/interpreter.py:103-474 of the reference): frame selection, ``get_limits`` and
``preprocess_segments`` -- everything up to the tensor handed to ``predict``.  Model loading and
inference (TFLite / Keras / OpenVINO) are outside this path: subclass and implement ``predict``.

``preprocess_segments`` uploads the frames the track needs once, then runs the three preprocessing
launches (track limits, medians + clip test, fused crop/resize/normalise/tile); ``preprocess_tracks``
does the same for every track of a clip in one go, and ``BatchPreprocessor`` (``..batch``) is the
device-resident form used after a batched extraction.

A clip parsed with ``parse_clips(..., keep_on_device=True)`` carries ``clip.device_frames``: its frames are then read from
the extraction's device buffers instead of being uploaded, the frame medians (and, for ``thermal_diff_norm``, the frame
extrema) the extraction computed are reused, and ``preprocess_clips`` makes the classifier inputs of every track of many
clips in one set of launches.
"""
import logging

import numpy as np

from .. import engine as _engine
from ..batch import BatchPreprocessor
from .segments import SegmentType


class HyperParams(dict):
    """The preprocessing-relevant defaults of ml_tools/hyperparams.py:9-170."""

    @property
    def channels(self):
        return self.get("channels", ["thermal", "filtered"])

    @property
    def frame_size(self):
        return self.get("frame_size", 32)

    @property
    def square_width(self):
        return self.get("square_width", 5 if self.use_segments else 1)

    @property
    def use_segments(self):
        return self.get("use_segments", True)

    @property
    def diff_norm(self):
        return self.get("diff_norm", True)

    @property
    def thermal_diff_norm(self):
        return self.get("thermal_diff_norm", False)

    @property
    def mvm(self):
        return self.get("mvm", False)

    @property
    def segment_types(self):
        types = self.get("segment_types", [SegmentType.ALL_RANDOM_MASKED])
        return [SegmentType[t] if isinstance(t, str) else (SegmentType(t) if isinstance(t, int) else t) for t in types]


def inc3_preprocess(x):
    """interpreter.py:563-566 (inceptionv3 / wr-resnet input scaling)."""
    x /= 127.5
    x -= 1.0
    return x


class Interpreter:
    def __init__(self, params=None, preprocess_fn=None, seed=None, device=None):
        self.params = params if params is not None else HyperParams()
        self.preprocess_fn = preprocess_fn
        self.seed = seed
        self.device = device
        self.labels = []
        # preprocess_movement stacks one tiled image per entry of params.channels (preprocess.py:169-189): any list over
        # thermal / filtered (repeats included, e.g. thermal, filtered, filtered) is a selection from the pair the device
        # kernel emits; the flow and mask channels are outside this path
        names = [c if isinstance(c, str) else getattr(c, "name", str(c)) for c in self.params.channels]
        unknown = [c for c in names if c not in ("thermal", "filtered")]
        if unknown or not names:
            raise NotImplementedError("channels {}: the device tiling kernel emits thermal and filtered".format(unknown or names))
        self._channel_index = [0 if c == "thermal" else 1 for c in names]
        if self.params.mvm:
            raise NotImplementedError("the movement-feature input (mvm) is outside this path")

    def predict(self, frames):
        raise NotImplementedError("model inference is outside the extraction / preprocessing path")

    # ------------------------------------------------------------------ selection
    def frames_for_prediction(self, clip, track, **args):
        """interpreter.py:178-257 for segment models."""
        frames_per_classify = args.get("frames_per_classify", 25)
        if frames_per_classify <= 1:
            raise NotImplementedError("single-frame models: the reference's own dispatch does not run here (interpreter.py:126-129 calls "
                                      "preprocess_frames without its samples argument); only segment models are built")
        predict_from_last = args.get("predict_from_last", None)
        segment_frames = args.get("segment_frames", None)
        dont_filter = args.get("dont_filter", False)
        if predict_from_last is not None and segment_frames is None:
            kept = clip.frames_kept()
            available = min(len(track.bounds_history), kept) if kept is not None else len(track.bounds_history)
            predict_from_last = min(predict_from_last, available)
            if available > predict_from_last:
                target, valid, predict_from_last = predict_from_last, 0, 0
                for i, r in enumerate(reversed(track.bounds_history[-available:])):
                    if r.blank:
                        continue
                    valid += 1
                    predict_from_last = i + 1
                    if valid >= target:
                        break
        return track.get_segments(self.params.square_width ** 2, ffc_frames=[] if dont_filter else clip.ffc_frames, repeats=1,
                                  segment_frames=segment_frames, segment_types=self.params.segment_types,
                                  from_last=predict_from_last, max_segments=args.get("num_predictions"),
                                  dont_filter=dont_filter, min_segments=args.get("min_segments"), seed=self.seed)

    # ------------------------------------------------------------------ device plumbing
    def _engine_for(self, clip):
        return _engine.get_engine(self.device, clip.res_x, clip.res_y, clip.config.edge_pixels)

    def _upload(self, eng, clip, frame_numbers):
        """The named frames' thermal (uint16) and filtered (float32) images -> device, plus number -> index."""
        import torch

        index = {}
        thermal = np.empty((len(frame_numbers), clip.res_y, clip.res_x), np.uint16)
        filtered = np.empty((len(frame_numbers), clip.res_y, clip.res_x), np.float32)
        for i, n in enumerate(frame_numbers):
            f = clip.get_frame(n)
            if f is None:
                raise Exception("Clasifying clip {} can't get frame {}".format(clip.get_id(), n))
            thermal[i] = f.thermal
            filtered[i] = f.filtered
            index[n] = i
        d_t = torch.from_numpy(thermal.view(np.int16)).to(eng.device).view(torch.uint16)
        d_f = torch.from_numpy(filtered).to(eng.device)
        return d_t, d_f, index

    @staticmethod
    def _region_rows(track, index):
        rows = []
        for r in track.bounds_history:
            i = index.get(r.frame_number, -1)
            rows.append([i, r.x, r.y, r.width, r.height, int(bool(r.blank) or i < 0)])
        return np.asarray(rows, dtype=np.int64).reshape(-1, 6)

    def get_limits(self, clip, track):
        """(thermal_norm_limits, filtered_norm_limits) (interpreter.py:315-363)."""
        res = self._run(clip, [(track, [])])
        n = BatchPreprocessor.tracks_numpy(res["tracks"])[0]
        thermal_limits = filtered_limits = None
        if self.params.thermal_diff_norm:
            found = int(n["has_thermal_limits"]) == 1
            thermal_limits = (np.float32(n["thermal_min"]) if found else None, np.float32(n["thermal_max"]) if found else None)
        if self.params.diff_norm:
            lo = np.float32(n["filtered_min"]) if n["has_limits"] else None
            filtered_limits = (lo, np.float32(n["filtered_max"]) if n["has_limits"] else 0)
        return thermal_limits, filtered_limits

    @staticmethod
    def _needed(jobs):
        needed = []
        for track, _ in jobs:
            needed.extend(int(r.frame_number) for r in track.bounds_history if not r.blank and r.width > 0 and r.height > 0)
        return sorted(set(needed))  # (Python ints: frame numbers of tracks loaded from metadata are np.uint16)

    def _tables(self, clip, jobs, index):
        """Per track (region rows, segment frames) with frame numbers mapped through ``index`` to device rows."""
        tables = []
        for track, segments in jobs:
            seg_frames = []
            for s in segments:
                missing = [int(n) for n in s.frame_indices if int(n) not in index]
                if missing:
                    raise Exception("Clasifying clip {} track {} can't get frame {}".format(clip.get_id(), track.get_id(), missing[0]))
                seg_frames.append(np.array([index[int(n)] for n in s.frame_indices], dtype=np.int64))
            tables.append((self._region_rows(track, index), seg_frames))
        return tables

    @staticmethod
    def _device_batch(clip):
        """The live ``DeviceBatch`` of a clip parsed with keep_on_device, None for any other clip."""
        h = getattr(clip, "device_frames", None)
        if h is None:
            return None
        if not h.live:
            raise Exception("Clasifying clip {}: its device frames were released".format(clip.get_id()))
        return h.batch

    def _run(self, clip, jobs):
        batch = self._device_batch(clip)
        if batch is not None:
            return self._run_device(batch, clip.crop_rectangle, [(clip, jobs)])
        eng = self._engine_for(clip)
        needed = [n for n in self._needed(jobs) if clip.get_frame(n) is not None]
        d_t, d_f, index = self._upload(eng, clip, needed)
        return self._launch(eng, d_t, d_f, self._tables(clip, jobs, index), clip.crop_rectangle)

    def _device_index(self, handle, jobs):
        """frame number -> thermal row of the frames the jobs' regions name that the clip's handle holds."""
        return {n: int(handle.thermal_row0) + n for n in self._needed(jobs) if handle.first_kept <= n < handle.n_frames}

    def _run_device(self, batch, crop, clip_jobs):
        """The tracks of several clips of one keep_on_device batch in one set of launches on the batch's own buffers: frame
        number n of a clip is thermal row ``thermal_row0 + n``; ``row_map`` takes each thermal row to its filtered row."""
        tables = []
        for clip, jobs in clip_jobs:
            tables.extend(self._tables(clip, jobs, self._device_index(clip.device_frames, jobs)))
        return self._launch(batch.engine, batch.thermal, batch.filtered, tables, crop, row_map=batch.row_map,
                            frame_medians=batch.medians, frame_info=batch.info)

    def _launch(self, eng, d_t, d_f, tables, crop, **device_stats):
        fn = 0
        if self.preprocess_fn is not None:
            from . import preprocess as _pp

            # the x / 127.5 - 1 scaling is built into the tiling kernel; any other callable is applied to each segment's array
            # on the host afterwards, as preprocess_movement does (preprocess.py:200-201)
            if self.preprocess_fn in (inc3_preprocess, _pp.preprocess_fn):
                fn = 1
        bp = BatchPreprocessor(eng, frame_size=self.params.frame_size, frames_per_row=self.params.square_width, preprocess_fn=fn,
                               diff_norm=self.params.diff_norm, thermal_diff_norm=self.params.thermal_diff_norm)
        return bp.run(d_t, d_f, tables, (crop.x, crop.y, crop.width, crop.height), seed=self.seed, **device_stats)

    def _fn_on_device(self):
        from . import preprocess as _pp

        return self.preprocess_fn in (inc3_preprocess, _pp.preprocess_fn)

    # ------------------------------------------------------------------ the path proper
    def preprocess_segments(self, clip, track, segments, predict_from_last=None):
        """-> (frame_indices per segment, float32 (n, H, W, C), masses) (interpreter.py:365-474)."""
        out = self.preprocess_tracks(clip, [(track, segments)])
        return out[0]

    def preprocess_tracks(self, clip, jobs):
        """``preprocess_segments`` for several (track, segments) pairs of one clip in one set of launches."""
        jobs = [(t, list(s)) for t, s in jobs]
        return self._collect(self._run(clip, jobs), jobs)

    def _collect(self, res, jobs):
        """Launch results -> per job (frame_indices per segment, data, masses), on the host."""
        d_seg = res["segments"]
        if self._channel_index != [0, 1]:
            import torch

            d_seg = d_seg.index_select(-1, torch.tensor(self._channel_index, device=d_seg.device))
        data = d_seg.cpu().numpy()
        if self.preprocess_fn is not None and not self._fn_on_device():
            data = np.float32([self.preprocess_fn(seg) for seg in data]) if len(data) else data
        out, at = [], 0
        for track, segments in jobs:
            n = len(segments)
            out.append(([s.frame_indices for s in segments], data[at : at + n], [s.mass for s in segments]))
            at += n
        return out

    def preprocess(self, clip, track, **args):
        segments = self.frames_for_prediction(clip, track, **args)
        return self.preprocess_segments(clip, track, segments, args.get("predict_from_last"))

    def preprocess_clips(self, clips, **args):
        """``preprocess`` for every track of every clip: per clip, per track in ``clip.tracks``, ``(frame_indices, data,
        masses)``.  The clips parsed in one ``parse_clips(..., keep_on_device=True)`` batch (with the same crop rectangle) go
        through one set of launches on the extraction's buffers; a clip without ``device_frames`` takes the per-clip path.
        Segments are selected in clip and track order first, so the random draws are those of ``preprocess`` called in a loop."""
        clip_jobs = []
        for clip in clips:
            self._device_batch(clip)  # (a released handle fails before anything runs)
            clip_jobs.append([(t, list(self.frames_for_prediction(clip, t, **args))) for t in clip.tracks])
        out = [None] * len(clips)
        groups = {}
        for i, clip in enumerate(clips):
            batch = self._device_batch(clip)
            if batch is None:
                out[i] = [self.preprocess_segments(clip, t, segments) for t, segments in clip_jobs[i]]
                continue
            c = clip.crop_rectangle
            groups.setdefault((id(batch), c.x, c.y, c.width, c.height), (batch, c, []))[2].append(i)
        for batch, crop, members in groups.values():
            res = self._collect(self._run_device(batch, crop, [(clips[i], clip_jobs[i]) for i in members]),
                                [j for i in members for j in clip_jobs[i]])
            at = 0
            for i in members:
                out[i] = res[at : at + len(clip_jobs[i])]
                at += len(clip_jobs[i])
        return out
