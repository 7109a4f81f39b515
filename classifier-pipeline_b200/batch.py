"""Batched clip extraction driver: many independent clips per launch, one persistent CTA per
clip (``csrc/extract_kernel.cu``).  This is the engine behind ``ClipTrackExtractor.parse_clip``
and the clip-sharded multi-GPU path; it only moves buffers and builds descriptors.
"""
import numpy as np

from . import native


def linear_clips(n_frames, background_thresh, weight_table, flags=native.CLIP_UPDATE_BACKGROUND, init_offsets=None):
    """Descriptors for clips packed back to back: clip i occupies frames [sum(n[:i]), sum(n[:i+1])).

    ``init_offsets`` (absolute frame indices) default to each clip's own first frame
    (track/cliptrackextractor.py:129-139 initialises the background from the first frame read).
    Scalars broadcast over clips.
    """
    n_frames = np.asarray(n_frames, dtype=np.int64).reshape(-1)
    n = len(n_frames)
    clips = np.zeros(n, dtype=native.CLIP_DTYPE)
    starts = np.concatenate([[0], np.cumsum(n_frames)[:-1]]) if n else np.zeros(0, np.int64)
    clips["frame_offset"] = starts
    clips["init_offset"] = starts if init_offsets is None else np.asarray(init_offsets, dtype=np.int64)
    clips["out_offset"] = starts
    clips["n_frames"] = n_frames
    clips["background_thresh"] = background_thresh
    clips["weight_table"] = weight_table
    clips["flags"] = flags
    return clips


def _total_frames(clips):
    """Frames the per-frame outputs of a batch of CLIP_DTYPE records hold: max over clips of ``out_offset + n_frames``."""
    return int((clips["out_offset"] + clips["n_frames"]).max()) if len(clips) else 0


def _pinned_out(out, name, shape, dtype):
    """``out[name]``, replaced by a new pinned host array unless it already has this shape and dtype."""
    a = out.get(name)
    if a is None or a.shape != tuple(shape) or a.dtype != np.dtype(dtype):
        a = native.pinned_empty(shape, dtype)
        out[name] = a
    return a


class BatchExtractor:
    """Owns a native context and the output buffers of one device."""

    def __init__(self, device=0, width=160, height=120, edge_pixels=1, max_regions=16):
        import torch

        if not torch.cuda.is_available():
            raise native.NativeError("CUDA device required: the extraction path has no CPU fallback")
        self.torch = torch
        self.device = torch.device("cuda", device)
        self.ctx = native.Context(device, width, height, edge_pixels, max_regions)
        self.width, self.height, self.max_regions = width, height, max_regions

    # ------------------------------------------------------------------ device-resident path
    def extract_device(self, d_frames, clips, keep_filtered=True, keep_labels=True, keep_state=False, d_state=None,
                       out=None, use_torch_stream=True):
        """Run the kernel on frames already in HBM.

        d_frames: torch.uint16 CUDA tensor, any shape whose trailing dims are (H, W).
        clips: numpy CLIP_DTYPE array (host) or a CUDA uint8 tensor holding the same records.
        Returns dict(regions, info, filtered, labels, state) of CUDA tensors (raw bytes for the
        two record arrays; view them with ``regions_numpy`` / ``info_numpy``).
        """
        torch = self.torch
        if use_torch_stream:
            self.ctx.use_torch_stream()
        if isinstance(clips, np.ndarray):
            n_clips = len(clips)
            total = _total_frames(clips)
            d_clips = torch.from_numpy(clips.view(np.uint8).reshape(-1).copy()).to(self.device)
        else:
            raise TypeError("clips must be a numpy CLIP_DTYPE array")
        npx = self.width * self.height
        if out is None:
            out = {}
        def buf(name, shape, dtype):
            t = out.get(name)
            if t is None or tuple(t.shape) != tuple(shape) or t.dtype != dtype:
                t = torch.empty(shape, dtype=dtype, device=self.device)
                out[name] = t
            return t
        regions = buf("regions", (max(total, 1), self.max_regions, native.REGION_DTYPE.itemsize), torch.uint8)
        info = buf("info", (max(total, 1), native.INFO_DTYPE.itemsize), torch.uint8)
        filtered = buf("filtered", (max(total, 1), self.height, self.width), torch.float32) if keep_filtered else None
        labels = buf("labels", (max(total, 1), self.height, self.width), torch.uint8) if keep_labels else None
        if d_state is None and keep_state:
            d_state = torch.zeros((max(n_clips, 1), self.ctx.state_bytes), dtype=torch.uint8, device=self.device)
        denoise = bool(n_clips) and bool((clips["flags"] & native.CLIP_DENOISE).any())
        if denoise and not keep_filtered:
            raise native.NativeError("denoise needs keep_filtered=True (the variance pass reads the filtered images)")
        no_resume = not (bool(n_clips) and bool((clips["flags"] & native.CLIP_RESUME).any()))
        self.ctx.extract_batch(d_frames, d_clips, n_clips, regions, info, filtered, labels, d_state, total_frames=total,
                               denoise=denoise, no_resume=no_resume)
        out.update(regions=regions, info=info, filtered=filtered, labels=labels, state=d_state, total_frames=total,
                   d_clips=d_clips)
        return out

    @staticmethod
    def regions_numpy(regions_tensor):
        a = regions_tensor.cpu().numpy()
        return a.reshape(-1).view(native.REGION_DTYPE).reshape(a.shape[0], a.shape[1])

    @staticmethod
    def info_numpy(info_tensor):
        a = info_tensor.cpu().numpy()
        return a.reshape(-1).view(native.INFO_DTYPE)

    # ------------------------------------------------------------------ host-buffer path (e2e)
    def extract_host(self, h_frames, clips, keep_filtered=False, keep_labels=False, chunk_clips=0, out=None):
        """Host uint16 frames in, host records out: H2D / kernel / D2H pipelined inside the library."""
        h_frames = np.ascontiguousarray(h_frames, dtype=np.uint16)
        total = _total_frames(clips)
        out = out if out is not None else {}
        regions = _pinned_out(out, "regions", (max(total, 1), self.max_regions), native.REGION_DTYPE)
        info = _pinned_out(out, "info", (max(total, 1),), native.INFO_DTYPE)
        filtered = _pinned_out(out, "filtered", (max(total, 1), self.height, self.width), np.float32) if keep_filtered else None
        labels = _pinned_out(out, "labels", (max(total, 1), self.height, self.width), np.uint8) if keep_labels else None
        clips = np.ascontiguousarray(clips)
        self.ctx.extract_batch_host(h_frames, clips, total, regions, info, filtered, labels, chunk_clips)
        out["total_frames"] = total
        return out


    def extract_host_packed(self, h_stream, table, clip_first, clips, chunk_clips=0, out=None):
        """Packed clips in, host records out: the inflated CPTV frame payloads (``h_stream`` uint8, ideally pinned; one
        ``native.CPTV_FRAME_DTYPE`` row per frame in ``table``; clip i = rows ``clip_first[i]:clip_first[i + 1]``) are
        staged to the device, decoded there and extracted.  ``clips`` address frames by table row."""
        h_stream = np.ascontiguousarray(h_stream, dtype=np.uint8)
        table = np.ascontiguousarray(table, dtype=native.CPTV_FRAME_DTYPE)
        clip_first = np.ascontiguousarray(clip_first, dtype=np.int64)
        clips = np.ascontiguousarray(clips)
        if len(clip_first) != len(clips) + 1:
            raise ValueError("clip_first must hold len(clips) + 1 rows")
        total = _total_frames(clips)
        out = out if out is not None else {}
        regions = _pinned_out(out, "regions", (max(total, 1), self.max_regions), native.REGION_DTYPE)
        info = _pinned_out(out, "info", (max(total, 1),), native.INFO_DTYPE)
        self.ctx.extract_batch_cptv_host(h_stream, table, clip_first, clips, total, regions, info, chunk_clips)
        out["total_frames"] = total
        return out


def pad_segment_samples(n_frames, tiles, seed=None):
    """Indices into a segment's frame list for its ``tiles`` cells: ``preprocess_movement`` repeats
    randomly chosen frames (seeded generator) when the segment is short, then sorts
    (ml_tools/preprocess.py:160-168)."""
    samples = list(np.arange(n_frames))
    if n_frames < tiles:
        rng = np.random.default_rng(seed)
        samples.extend(rng.choice(samples, tiles - n_frames))
        samples.sort()
    return np.asarray(samples[:tiles], dtype=np.int64)


class BatchPreprocessor:
    """``Interpreter.preprocess_segments`` (ml_tools/interpreter.py:365-474) for many tracks in three
    launches (csrc/preprocess_kernels.cu): track-wide filtered limits, per-frame medians + the
    clip-at-zero test, then one CTA per (segment, tile) that crops, resizes, normalises and writes the
    tile into the segment image.  Frames stay in HBM (the extraction's thermal input and filtered output)."""

    def __init__(self, extractor, frame_size=32, frames_per_row=5, preprocess_fn=0, diff_norm=True, thermal_diff_norm=False):
        # preprocess_movement pads every segment to frames_per_row * 5 samples (preprocess.py:161) and square_clip lays out the
        # first frames_per_row ** 2 of them, frames_per_row to a row (imageprocessing.py:85-104); past 5 per row a padded
        # segment has fewer samples than cells and the reference's square_clip fails with an IndexError
        if not 1 <= int(frames_per_row) <= 5:
            raise ValueError("frames_per_row (HyperParams.square_width) must be in [1, 5], got {}".format(frames_per_row))
        self.ex = extractor
        self.torch = extractor.torch
        self.device = extractor.device
        self.frame_size = frame_size
        self.frames_per_row = int(frames_per_row)
        self.tiles = self.frames_per_row * 5  # samples drawn and padded per segment: the columns of the segment table
        self.preprocess_fn = preprocess_fn
        # HyperParams.diff_norm / thermal_diff_norm (interpreter.py:315-363,405-408): track-wide limits for the filtered / the
        # thermal channel; with diff_norm off both channels are normalised per tile
        self.diff_norm = bool(diff_norm)
        self.thermal_diff_norm = bool(thermal_diff_norm)

    def build_tables(self, tracks, seed=None):
        """tracks: list of (regions, segments); regions int array (n, >=6) rows [frame, x, y, w, h, blank] with
        ``frame`` an index into the device frame buffers, segments a list of frame arrays (same index space).
        Returns (limit_regions SAMPLE_DTYPE, samples SAMPLE_DTYPE, segment_samples int32 (n_seg, tiles), seg_track).

        Flattens the per-track lists and hands them to ``build_tables_flat`` (one concatenation, one sort, one unique for
        all tracks together)."""
        n_tracks = len(tracks)
        if n_tracks == 0:
            z = np.zeros(0, native.SAMPLE_DTYPE)
            return z, z.copy(), np.zeros((0, self.tiles), np.int32), np.zeros(0, np.int32)
        reg_list = [np.asarray(r) for r, _ in tracks]
        for r in reg_list:
            if r.ndim != 2 or r.shape[1] < 6:
                raise ValueError("regions must be (n, >=6) rows [frame, x, y, w, h, blank]")
        reg_n = np.fromiter((len(r) for r in reg_list), np.int64, n_tracks)
        R = np.concatenate([r[:, :6] for r in reg_list]).astype(np.int64) if reg_n.sum() else np.zeros((0, 6), np.int64)
        r_track = np.repeat(np.arange(n_tracks, dtype=np.int64), reg_n)
        seg_arrays, seg_track = [], []
        for ti, (_, segments) in enumerate(tracks):
            for sgm in segments or ():
                a = np.asarray(sgm, dtype=np.int64).reshape(-1)
                if len(a):
                    seg_arrays.append(a)
                    seg_track.append(ti)
        seg_len = np.fromiter((len(a) for a in seg_arrays), np.int64, len(seg_arrays))
        seg_frames = np.concatenate(seg_arrays) if seg_arrays else np.zeros(0, np.int64)
        return self.build_tables_flat(R, r_track, seg_frames, seg_len, np.asarray(seg_track, np.int64), seed=seed)

    def build_tables_flat(self, regions, region_track, seg_frames, seg_len, seg_track, seed=None):
        """The same tables from flat arrays: ``regions`` (N, 6) rows [frame, x, y, w, h, blank] of all tracks with their
        track index in ``region_track``; the segments' frames back to back in ``seg_frames`` (``seg_len`` frames each,
        segment i belongs to track ``seg_track[i]``).  Pure array code: tens of milliseconds for 10 000 tracks."""
        W, H = self.ex.width, self.ex.height
        R = np.asarray(regions, dtype=np.int64).reshape(-1, 6)
        r_track = np.asarray(region_track, dtype=np.int64)
        seg_frames = np.asarray(seg_frames, dtype=np.int64)
        seg_len = np.asarray(seg_len, dtype=np.int64)
        seg_track = np.asarray(seg_track, dtype=np.int64)

        def outside(rows):
            return (rows[:, 1] < 0) | (rows[:, 2] < 0) | (rows[:, 1] + rows[:, 3] > W) | (rows[:, 2] + rows[:, 4] > H)

        # ---- get_limits: every non-blank region with an area
        ok = (R[:, 5] == 0) & (R[:, 3] > 0) & (R[:, 4] > 0) & (R[:, 0] >= 0)
        bad = ok & outside(R)
        if bad.any():
            raise ValueError("track {}: a region lies outside the {}x{} frame".format(int(r_track[np.argmax(bad)]), W, H))
        lim = np.zeros(int(ok.sum()), native.SAMPLE_DTYPE)
        Rk = R[ok]
        lim["frame"], lim["x"], lim["y"], lim["width"], lim["height"], lim["track"] = Rk[:, 0], Rk[:, 1], Rk[:, 2], Rk[:, 3], Rk[:, 4], r_track[ok]
        if len(seg_len) == 0:
            return lim, np.zeros(0, native.SAMPLE_DTYPE), np.zeros((0, self.tiles), np.int32), np.zeros(0, np.int32)
        if (seg_len <= 0).any():
            raise ValueError("empty segment")
        if (seg_frames < 0).any():
            raise ValueError("segment frames must be non-negative")
        # ---- the unique (track, frame) pairs of the segments, in (track, frame) order
        # (rows without a frame -- blank regions, frames the caller could not supply -- get the key big - 1, one past every real frame)
        big = int(max(seg_frames.max(), R[:, 0].max() if len(R) else 0)) + 2
        key = np.repeat(seg_track, seg_len) * big + seg_frames
        uniq, inverse = np.unique(key, return_inverse=True)
        # the region of each unique frame: the first row of the track with that frame number (unique_regions keeps the first)
        rkey = r_track * big + np.where(R[:, 0] >= 0, R[:, 0], big - 1)
        order = np.argsort(rkey, kind="stable")
        pos = np.searchsorted(rkey[order], uniq)
        hit = pos < len(order)
        hit[hit] &= rkey[order[pos[hit]]] == uniq[hit]
        if not hit.all():
            raise ValueError("track {}: a segment names a frame the track has no region for".format(int(uniq[np.argmin(hit)] // big)))
        rows = R[order[pos]]
        u_track = uniq // big
        empty = (rows[:, 3] <= 0) | (rows[:, 4] <= 0)
        if empty.any():
            raise ValueError("track {}: a segment frame has an empty region".format(int(u_track[np.argmax(empty)])))
        if outside(rows).any():
            raise ValueError("track {}: a region lies outside the {}x{} frame".format(int(u_track[np.argmax(outside(rows))]), W, H))
        smp = np.zeros(len(uniq), native.SAMPLE_DTYPE)
        smp["frame"], smp["x"], smp["y"], smp["width"], smp["height"], smp["track"] = rows[:, 0], rows[:, 1], rows[:, 2], rows[:, 3], rows[:, 4], u_track
        # ---- the tiles of every segment: its frames in order, padded like preprocess_movement when it is short
        seg = np.empty((len(seg_len), self.tiles), np.int32)
        starts = np.concatenate([[0], np.cumsum(seg_len)[:-1]])
        full = seg_len >= self.tiles
        if full.any():
            seg[full] = inverse[starts[full][:, None] + np.arange(self.tiles)[None, :]]
        for i in np.nonzero(~full)[0]:
            idx = inverse[starts[i] : starts[i] + seg_len[i]]
            seg[i] = idx[pad_segment_samples(int(seg_len[i]), self.tiles, seed)]
        return lim, smp, seg, seg_track.astype(np.int32)

    def output_shape(self, n_segments):
        """Shape of the segment images: the first ``frames_per_row ** 2`` samples of each segment, ``frames_per_row`` to a row,
        both channels."""
        side = self.frames_per_row * self.frame_size
        return (int(n_segments), side, side, 2)

    def run_tables(self, d_thermal, d_filtered, limit_regions, samples, segment_samples, n_tracks, crop_rectangle, out=None,
                   row_map=None, frame_medians=None, frame_info=None):
        """Launch on prepared tables (host numpy or CUDA uint8/int32 tensors).  Returns the CUDA float32
        tensor ``output_shape(n_segments)`` plus the device tables.

        On an extraction's own buffers (``DeviceBatch``): ``row_map`` (host int64, one entry per thermal row) gives the filtered
        row of every thermal row the tables name; ``frame_medians`` (CUDA float32 per thermal row, ``cpt_frame_medians``) and
        ``frame_info`` (the extraction's CUDA INFO_DTYPE records, with CLIP_FRAME_STATS) are reused instead of re-reading the
        frames.  The tables must then be host arrays."""
        torch = self.torch
        ctx = self.ex.ctx
        ctx.use_torch_stream()

        def dev(a):
            if isinstance(a, np.ndarray):
                return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).to(self.device)
            return a

        n_lim = len(limit_regions) if isinstance(limit_regions, np.ndarray) else limit_regions.numel() // native.SAMPLE_DTYPE.itemsize
        n_smp = len(samples) if isinstance(samples, np.ndarray) else samples.numel() // native.SAMPLE_DTYPE.itemsize
        n_seg = segment_samples.shape[0]
        d_lim, d_smp = dev(limit_regions), dev(samples)
        # only the first frames_per_row ** 2 columns are tiles of the image (at the default 5: all 25)
        launched = self.frames_per_row ** 2
        if isinstance(segment_samples, np.ndarray):
            d_seg = torch.from_numpy(np.ascontiguousarray(segment_samples[:, :launched], dtype=np.int32)).to(self.device)
        else:
            d_seg = segment_samples[:, :launched].contiguous()
        d_tracks = torch.empty((max(n_tracks, 1), native.TRACK_NORM_DTYPE.itemsize), dtype=torch.uint8, device=self.device)
        shape = self.output_shape(n_seg)
        d_out = None if out is None else out.get("segments")
        if d_out is None or tuple(d_out.shape) != shape:
            d_out = torch.empty(shape, dtype=torch.float32, device=self.device)
            if out is not None:
                out["segments"] = d_out
        d_lim_rows = d_smp_rows = None
        if row_map is not None:
            row_map = np.asarray(row_map, dtype=np.int64)
            d_lim_rows = torch.from_numpy(row_map[limit_regions["frame"]]).to(self.device)
            d_smp_rows = torch.from_numpy(row_map[samples["frame"]]).to(self.device)
        # (always resets the rows)
        ctx.preprocess_limits_ex(d_filtered, d_lim_rows, d_lim, n_lim if self.diff_norm else 0, d_tracks, n_tracks)
        if self.thermal_diff_norm:
            ctx.preprocess_thermal_limits_ex(d_thermal, d_lim_rows, d_lim, n_lim, d_tracks, n_tracks, frame_medians, frame_info)
        ctx.preprocess_medians_ex(d_thermal, frame_medians, d_smp, n_smp, d_tracks)
        fn = int(self.preprocess_fn) | (0 if self.diff_norm else native.PREPROCESS_PER_TILE)
        ctx.preprocess_segments_ex(d_thermal, d_filtered, d_smp_rows, d_smp, d_tracks, d_seg, n_seg, launched, self.frames_per_row,
                                   self.frame_size, crop_rectangle, fn, d_out)
        return dict(segments=d_out, tracks=d_tracks, samples=d_smp)

    def run(self, d_thermal, d_filtered, tracks, crop_rectangle, seed=None, out=None, row_map=None, frame_medians=None, frame_info=None):
        lim, smp, seg, seg_track = self.build_tables(tracks, seed=seed)
        res = self.run_tables(d_thermal, d_filtered, lim, smp, seg, len(tracks), crop_rectangle, out=out, row_map=row_map,
                              frame_medians=frame_medians, frame_info=frame_info)
        res["segment_track"] = seg_track
        return res

    @staticmethod
    def tracks_numpy(t):
        a = t.cpu().numpy()
        return a.reshape(-1).view(native.TRACK_NORM_DTYPE)


def tracked_row_map(clips, n_input):
    """thermal row -> filtered row of every tracked frame of the CLIP_DTYPE records ``clips`` (frame t of clip i is thermal
    row ``frame_offset + t`` and filtered row ``out_offset + t``); -1 for the other rows of the ``n_input``-row input (init
    frames, leading background frames)."""
    row_map = np.full(int(n_input), -1, np.int64)
    for c in np.asarray(clips, dtype=native.CLIP_DTYPE).reshape(-1):
        f0, o0, n = int(c["frame_offset"]), int(c["out_offset"]), int(c["n_frames"])
        row_map[f0 : f0 + n] = np.arange(o0, o0 + n)
    return row_map


class DeviceBatch:
    """The device buffers one ``ClipTrackExtractor.parse_clips(keep_on_device=True)`` launch leaves behind, shared by the
    ``ClipDeviceFrames`` handles of its clips: the thermal input (uint16, one row per frame read, init and leading
    background frames included), the filtered output (float32, one row per tracked frame), the frame medians (float32 per
    thermal row) and the frame records (INFO_DTYPE bytes per filtered row).  ``row_map[thermal row]`` is the filtered row of
    a tracked frame and -1 for every other row.  The memory is freed when the last handle is released."""

    def __init__(self, engine, thermal, filtered, medians, info, row_map):
        self.engine = engine
        self.thermal, self.filtered, self.medians, self.info = thermal, filtered, medians, info
        self.row_map = np.asarray(row_map, dtype=np.int64)


class ClipDeviceFrames:
    """One clip's frames inside a ``DeviceBatch``: frame number ``n`` (``Clip.current_frame``) is thermal row
    ``thermal_row0 + n``, median row ``median_row0 + n`` and filtered row ``filtered_row0 + n`` for ``first_kept <= n <
    n_frames`` (``first_kept`` > 0 only when the clip's frame buffer keeps the last ``max_frames`` frames)."""

    def __init__(self, batch, thermal_row0, filtered_row0, n_frames, first_kept=0):
        self.batch = batch
        self.thermal_row0 = int(thermal_row0)
        self.median_row0 = int(thermal_row0)
        self.filtered_row0 = int(filtered_row0)
        self.n_frames = int(n_frames)
        self.first_kept = int(first_kept)

    @property
    def live(self):
        return self.batch is not None

    def release(self):
        """Drop this clip's reference to the batch buffers (freed once every clip of the batch has released them)."""
        self.batch = None
