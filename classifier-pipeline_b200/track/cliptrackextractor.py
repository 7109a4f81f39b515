"""``ClipTrackExtractor``: thermal-clip track extraction on the B200 (track/cliptrackextractor.py:35-247).

Same constructor, attributes and methods as the reference class.  The per-pixel work of one frame
(background subtraction, normalisation, blur / threshold / close, connected components, delta-frame
variance, the weighted background update and the frame statistics) runs in the persistent
extraction kernel behind ``libcptrack.so``; this class decodes the clip, launches the kernel once
per clip (``parse_clip``) or once per frame (``process_frame`` / ``start_tracking``, streaming), and
feeds the region lists it gets back to the host-side matcher inherited from ``ClipTracker``.

``parse_clips`` is the batched entry point the reference does not have: many clips in one launch
(one persistent CTA per clip), which is how a B200 is kept busy.
"""
import logging
import time
from datetime import datetime

import numpy as np

from .. import engine as _engine
from .. import native
from ..batch import ClipDeviceFrames, DeviceBatch, linear_clips, tracked_row_map
from ..cptv import CptvReader
from ..piclassifier.cptvmotiondetector import is_affected_by_ffc
from ..piclassifier.motiondetector import WeightedBackground
from .clip import Clip
from .cliptracker import ClipTracker

RING_FRAMES = 64  # streaming ring: the kernel reads frame t-45 for the sliding mean


class ClipTrackExtractor(ClipTracker):
    PREVIEW = "preview"
    VERSION = 11
    TYPE = "thermal"
    # how clips are opened; tests and in-memory pipelines may substitute any object with
    # get_header() / next_frame() (the interface of cptv_rs_python_bindings.CptvReader)
    reader_factory = staticmethod(lambda path: CptvReader(str(path)))

    @property
    def tracker_version(self):
        return self.version

    @property
    def type(self):
        return ClipTrackExtractor.TYPE

    def __init__(self, config, use_opt_flow, cache_to_disk=False, keep_frames=True, calc_stats=True,
                 high_quality_optical_flow=False, verbose=False, do_tracking=True, update_background=True,
                 calculate_filtered=False, calculate_thumbnail_info=False, from_pi=False, max_frames=None, device=None):
        super().__init__(config, cache_to_disk, keep_frames=keep_frames, calc_stats=calc_stats, verbose=verbose,
                         do_tracking=do_tracking, calculate_thumbnail_info=calculate_thumbnail_info, max_frames=max_frames)
        self.version = f"PI-{ClipTrackExtractor.VERSION}" if from_pi else ClipTrackExtractor.VERSION
        if use_opt_flow:
            raise NotImplementedError("optical flow is not part of the B200 extraction path")
        if getattr(self.config, "denoise", False) and not native.HAS_NLM:
            raise native.NativeError(
                "TrackingConfig.denoise=True needs the non-local-means kernel, which this build of libcptrack.so "
                "does not have; set config.tracking['thermal'].denoise = False (the Pi configuration)")
        self.use_opt_flow = use_opt_flow
        self.high_quality_optical_flow = high_quality_optical_flow
        self.background_alg = None
        self.update_background = update_background
        self.calculate_filtered = calculate_filtered
        self.weighting_percent = 1
        self.device = device
        self.device_decode = True  # decode CPTV files on the device when this package's reader opens them
        self._stream = None  # streaming session (process_frame)

    @property
    def tracking_time(self):
        return self._tracking_time

    # ------------------------------------------------------------------ clip set-up
    def init_clip(self, clip):
        """Header, crop rectangle, thresholds; the first frame initialises both backgrounds
        (cliptrackextractor.py:98-139)."""
        clip.set_frame_buffer(self.high_quality_optical_flow, self.cache_to_disk, self.use_opt_flow, self.keep_frames,
                              self.max_frames)
        clip.type = self.type
        reader = self.reader_factory(clip.source_file)
        header = reader.get_header()
        clip.set_res(header.x_resolution, header.y_resolution)
        if clip.from_metadata:
            for track in clip.tracks:
                track.crop_regions()
        clip.set_model(header.model if header.model else None)
        start = datetime.fromtimestamp(header.timestamp / 1000000).astimezone(Clip.local_tz)
        clip.set_video_stats(start)
        frame = reader.next_frame()
        clip.update_background(frame.pix)
        clip._background_calculated()
        self.background_alg = self._new_background(clip)
        self.background_alg.process_frame(frame.pix)
        self._stream = None
        return reader

    def _weight_add(self, clip):
        return (1 if clip.camera_model == "lepton3.5" else 0.1) / self.weighting_percent

    def _new_background(self, clip):
        return WeightedBackground(clip.crop_rectangle.x, clip.crop_rectangle, clip.res_x, clip.res_y, self._weight_add(clip),
                                  device=self.device)

    # ------------------------------------------------------------------ whole clips
    def parse_clip(self, clip, process_background=False, *, keep_on_device=False):
        """Loads a cptv file and extracts its tracks.  Returns True.  ``keep_on_device``: as in ``parse_clips``."""
        self._tracking_time = None
        start = time.time()
        self.parse_clips([clip], process_background=process_background, keep_on_device=keep_on_device)
        self._tracking_time = time.time() - start
        return True

    def parse_clips(self, clips, process_background=False, *, keep_on_device=False):
        """Batched ``parse_clip``: decode every clip, ONE kernel launch for all of them, then the
        host-side matcher per clip.  Track ids restart at 1 for every clip, as they do when the
        reference processes the clips one after another.

        ``keep_on_device=True`` keeps the batch's frames in device memory for ``Interpreter.preprocess_clips``: the thermal
        input, the filtered output (also with ``keep_frames=False``), the frame medians (also with ``calc_stats=False``) and
        the frame records.  Each clip gets ``clip.device_frames``, a ``batch.ClipDeviceFrames`` handle; ``release()`` it when
        the clip's classifier inputs are made.  With ``keep_frames=False`` no filtered or label image is copied to the host."""
        from .track import Track

        jobs = []
        readers = []
        # CPTV files read with this package's own reader are decoded on the device (csrc/cptv_kernels.cu): the host
        # only inflates the stream and walks the section headers
        device_decode = self.device_decode and self.reader_factory is ClipTrackExtractor.reader_factory
        for clip in clips:
            reader = self.init_clip(clip)
            if clip.background is None:
                logging.error("Clip has no background have you called init_clip first")
                raise Exception("Clip has no background have you called init_clip first")
            # the reference re-opens the file (cliptrackextractor.py:160): the first frame is tracked too
            reader = self.reader_factory(clip.source_file)
            reader.get_header()
            if device_decode:
                readers.append(reader)
                jobs.append((clip, self.background_alg, None))
                continue
            frames = []
            while True:
                frame = reader.next_frame()
                if frame is None:
                    break
                if not process_background and frame.background_frame:
                    continue
                frames.append(frame)
            jobs.append((clip, self.background_alg, frames))
        device_frames = None
        if device_decode and jobs:
            jobs, device_frames = self._decode_on_device(jobs, readers, process_background)
        results = self._run_batch(jobs, device_frames, keep_on_device=keep_on_device)
        for (clip, background_alg, frames), res in zip(jobs, results):
            clip.device_frames = res.get("device_frames")
            self.background_alg = background_alg
            Track._track_id = 1
            for t, frame in enumerate(frames):
                self._consume_frame(clip, frame, res, t)
            if not clip.from_metadata and self.do_tracking:
                self.apply_track_filtering(clip)
            if self.calc_stats:
                clip.stats.completed()
        return True

    def _flags(self):
        flags = 0
        if self.update_background:
            flags |= native.CLIP_UPDATE_BACKGROUND
        if self.calc_stats:
            flags |= native.CLIP_FRAME_STATS
        if getattr(self.config, "denoise", False):
            flags |= native.CLIP_DENOISE
        return flags

    def _decode_on_device(self, jobs, readers, process_background):
        """Decode the clips' frames on the device; returns the jobs with their frame objects (pixels copied back for
        the host-side ``Clip`` objects) and ``(d_frames, init_offsets, frame_offsets)`` for the extraction launch."""
        from ..cptv import decode_clips_device

        clip0 = jobs[0][0]
        eng = _engine.get_engine(self.device, clip0.res_x, clip0.res_y, clip0.config.edge_pixels)
        d_frames, clip_first, all_frames = decode_clips_device(eng, readers)
        pix = d_frames.cpu().numpy()
        out_jobs, init_offsets, frame_offsets = [], [], []
        for i, ((clip, background_alg, _), frames) in enumerate(zip(jobs, all_frames)):
            first = clip_first[i]
            for k, f in enumerate(frames):
                f.pix = pix[first + k]
            # tracked frames must be contiguous on the device: background frames only ever lead the file
            skip = 0
            if not process_background:
                while skip < len(frames) and frames[skip].background_frame:
                    skip += 1
                if any(f.background_frame for f in frames[skip:]):
                    raise NotImplementedError("background frames after the first tracked frame")
            out_jobs.append((clip, background_alg, frames[skip:]))
            init_offsets.append(first)
            frame_offsets.append(first + skip)
        return out_jobs, (d_frames, init_offsets, frame_offsets)

    def _run_batch(self, jobs, device_frames=None, keep_on_device=False):
        """One launch over every clip of ``jobs``; per clip a dict of host arrays for its frames (and, with
        ``keep_on_device``, its ``ClipDeviceFrames`` handle)."""
        import torch

        if not jobs:
            return []
        geoms = {(c.res_x, c.res_y, c.config.edge_pixels) for c, _, _ in jobs}
        if len(geoms) != 1:
            raise ValueError("clips of one batch must share resolution and edge_pixels")
        res_x, res_y, edge = geoms.pop()
        eng = _engine.get_engine(self.device, res_x, res_y, edge)
        ctx = eng.ctx
        counts = [len(frames) for _, _, frames in jobs]
        total = sum(counts)
        keep_images = self.keep_frames or self.calculate_filtered
        # keep_on_device: the frame records carry the thermal extrema the thermal_diff_norm limits reuse
        clips = linear_clips(counts, 0, 0, flags=self._flags() | (native.CLIP_FRAME_STATS if keep_on_device else 0))
        for i, (clip, background_alg, frames) in enumerate(jobs):
            clips["background_thresh"][i] = clip.background_thresh
            clips["weight_table"][i] = ctx.weight_table(background_alg.weight_add, max_frames=max(max(counts), 1024))
        if device_frames is not None:
            # frames decoded on the device: the first frame of the file initialises the background where it lies
            d_frames, init_offsets, frame_offsets = device_frames
            clips["init_offset"] = init_offsets
            clips["frame_offset"] = frame_offsets
            n_input = int(d_frames.shape[0])
        else:
            # frame layout: [init frame of clip 0][tracked frames of clip 0][init frame of clip 1]...
            h_frames = np.empty((total + len(jobs), res_y, res_x), np.uint16)
            pos = 0
            for i, (clip, background_alg, frames) in enumerate(jobs):
                h_frames[pos] = clip.background if clip.background.dtype == np.uint16 else np.uint16(clip.background)
                clips["init_offset"][i] = pos
                clips["frame_offset"][i] = pos + 1
                for t, frame in enumerate(frames):
                    h_frames[pos + 1 + t] = frame.pix
                pos += 1 + counts[i]
            d_frames = torch.from_numpy(h_frames.view(np.int16)).to(eng.device).view(torch.uint16)
            n_input = total + len(jobs)
        denoise = bool(getattr(self.config, "denoise", False))  # the device NLM + variance passes read the filtered images
        out = eng.extract_device(d_frames, clips, keep_filtered=keep_images or denoise or keep_on_device, keep_labels=keep_images,
                                 keep_state=True, out={})
        medians = d_med = None
        if (self.calc_stats or keep_on_device) and total:
            d_med = torch.empty((n_input,), dtype=torch.float32, device=eng.device)
            ctx.frame_medians(d_frames, n_input, d_med)
            if self.calc_stats:
                medians = d_med.cpu().numpy()
        batch = None
        if keep_on_device:
            batch = DeviceBatch(eng, d_frames, out["filtered"], d_med, out["info"], tracked_row_map(clips, n_input))
        info = eng.info_numpy(out["info"])
        # (only the region slots some frame uses travel: the API engines have 255 per frame)
        used = min(int(info["n_components"][:total].max()) if total else 0, eng.max_regions)
        regions = eng.regions_numpy(out["regions"][:, : max(used, 1)].contiguous())
        if total and int(info["n_components"][:total].max()) > eng.max_regions:
            # more components than the uint8 label image can number: the first 255 (OpenCV label order) are kept
            logging.warning("%d frame(s) have more than %d components; the rest are dropped",
                            int((info["n_components"][:total] > eng.max_regions).sum()), eng.max_regions)
        filtered = out["filtered"].cpu().numpy() if keep_images else None
        labels = out["labels"].cpu().numpy() if keep_images else None
        results = []
        for i, (clip, background_alg, frames) in enumerate(jobs):
            o0, n = int(clips["out_offset"][i]), counts[i]
            f0 = int(clips["frame_offset"][i])
            # the clip's final WeightedBackground state is the kernel's state record
            background_alg.d_state.copy_(out["state"][i : i + 1])
            background_alg.invalidate()
            results.append(dict(
                regions=regions[o0 : o0 + n], info=info[o0 : o0 + n],
                filtered=None if filtered is None else filtered[o0 : o0 + n],
                labels=None if labels is None else labels[o0 : o0 + n],
                medians=None if medians is None else medians[f0 : f0 + n],
            ))
            if batch is not None:
                kept = clip.frame_buffer.max_frames if clip.frame_buffer is not None else None
                results[-1]["device_frames"] = ClipDeviceFrames(batch, f0, o0, n, first_kept=max(n - kept, 0) if kept else 0)
        return results

    def _consume_frame(self, clip, frame, res, t):
        """Host half of ``process_frame`` for frame ``t`` of a kernel result."""
        ffc_affected = is_affected_by_ffc(frame)
        clip.ffc_affected = ffc_affected
        info = res["info"][t]
        tracking = self.do_tracking or self.calculate_thumbnail_info
        filtered = res["filtered"][t] if res["filtered"] is not None else None
        mask = res["labels"][t] if (res["labels"] is not None and tracking) else None
        stats = None
        if self.calc_stats:
            npx = frame.pix.size
            stats = (res["medians"][t], int(info["thermal_max"]), int(info["thermal_min"]), int(info["thermal_sum"]) / npx,
                     float(info["abs_filtered_sum"]))
        clip.add_frame(frame.pix.copy(), filtered, mask, ffc_affected, frame_stats=stats)
        if not self.do_tracking:
            return []
        new_tracks = []
        if not clip.from_metadata:
            regions = []
            if ffc_affected:
                clip.active_tracks = set()
            else:
                n = int(info["n_components"])
                r = res["regions"][t][:n]
                area = r["area"].astype(np.float64)
                components = np.stack([r["x"], r["y"], r["width"], r["height"], r["area"]], axis=1)
                centroids = np.stack([r["sum_x"] / area, r["sum_y"] / area], axis=1)
                variances = r["pixel_variance"] if clip.current_frame > 0 or res.get("have_prev") else None
                regions = self._get_regions_of_interest(clip, components, centroids, variances)
                new_tracks = self._apply_region_matchings(clip, regions)
            clip.region_history.append(regions)
        return new_tracks

    # ------------------------------------------------------------------ streaming
    def start_tracking(self, clip, frames, track_frames=True, background_alg=None, **args):
        """Feed the preview frames of a new recording (cliptrackextractor.py:182-196)."""
        do_tracking = self.do_tracking
        self.background_alg = background_alg
        self._stream = None
        self.do_tracking = self.do_tracking and track_frames
        new_tracks = []
        for frame in frames:
            new_tracks.extend(self.process_frame(clip, frame))
        self.do_tracking = do_tracking
        return new_tracks

    def _open_stream(self, clip):
        import torch

        if self.background_alg is None or not self.background_alg.initialised:
            raise Exception("Clip has no background have you called init_clip first")
        eng = _engine.get_engine(self.device, clip.res_x, clip.res_y, clip.config.edge_pixels)
        if self.background_alg.engine is not eng:
            raise native.NativeError("background_alg lives on another device / geometry than the clip")
        self._stream = dict(
            eng=eng, t=0, out={}, background_alg=self.background_alg,
            ring=torch.zeros((RING_FRAMES, clip.res_y, clip.res_x), dtype=torch.uint16, device=eng.device),
            median=torch.empty((1,), dtype=torch.float32, device=eng.device),
        )
        return self._stream

    def process_frame(self, clip, frame, *, update_background=False):
        """Track one more frame of a clip (streaming; one kernel launch).

        As in the reference (cliptrackextractor.py:198-247) this does NOT touch the background: callers drive
        ``background_alg`` themselves (``_track_clip`` feeds it the mean of the last 45 frames, the Pi's motion detector its
        running mean).  ``update_background=True`` (keyword only, not in the reference) fuses ``_track_clip``'s update --
        ``background_alg.process_frame(mean of the last <=45 frames)`` -- into the same launch."""
        import torch

        denoise = bool(getattr(self.config, "denoise", False))
        st = self._stream
        if st is None or st["background_alg"] is not self.background_alg:
            st = self._open_stream(clip)
        eng, t = st["eng"], st["t"]
        slot = t % RING_FRAMES
        pix = np.ascontiguousarray(frame.pix, dtype=np.uint16)
        st["ring"][slot].view(torch.int16).copy_(torch.from_numpy(pix.view(np.int16)))
        # the kernel resumes from (and saves to) the background's own state record
        flags = (self._flags() | native.CLIP_RESUME) & ~native.CLIP_UPDATE_BACKGROUND
        if update_background and self.update_background:
            flags |= native.CLIP_UPDATE_BACKGROUND
        c = linear_clips([1], clip.background_thresh, self.background_alg.weight_slot, flags=flags)
        c["frame_offset"] = 0
        c["init_offset"] = 0
        c["first_frame"] = t
        c["ring_frames"] = RING_FRAMES
        c["out_offset"] = 0
        keep_images = self.keep_frames or self.calculate_filtered
        oi = 0  # output index of this frame
        if denoise:
            # TrackingConfig.denoise (cliptracker.py:116-117): the NLM, mask, component and variance passes follow the launch and
            # read the previous frame's filtered image and info at output index out_offset - 1 -- the frame goes to index 1
            # and the previous call's outputs are moved to index 0 first
            oi = 1
            c["out_offset"] = 1
            c["flags"] |= native.CLIP_DENOISE | native.CLIP_PREV_IN_OUTPUT
            prev = st["out"]
            if t > 0 and prev.get("filtered") is not None and prev["filtered"].shape[0] == 2:
                prev["filtered"][0].copy_(prev["filtered"][1])
                prev["info"][0].copy_(prev["info"][1])
        out = eng.extract_device(st["ring"], c, keep_filtered=keep_images or denoise, keep_labels=keep_images,
                                 d_state=self.background_alg.d_state, out=st["out"])
        medians = None
        if self.calc_stats:
            eng.ctx.frame_medians(st["ring"][slot], 1, st["median"])
            medians = st["median"].cpu().numpy()
        self.background_alg.invalidate()
        res = dict(
            regions=eng.regions_numpy(out["regions"])[oi:oi + 1], info=eng.info_numpy(out["info"])[oi:oi + 1],
            filtered=out["filtered"][oi:oi + 1].cpu().numpy() if keep_images else None,
            labels=out["labels"][oi:oi + 1].cpu().numpy() if keep_images else None,
            medians=medians, have_prev=t > 0,
        )
        if int(res["info"]["n_components"][0]) > eng.max_regions:
            logging.warning("frame %d has more than %d components; the rest are dropped", t, eng.max_regions)
        st["t"] = t + 1
        return self._consume_frame(clip, frame, res, 0)
