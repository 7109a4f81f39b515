"""``ClipTracker``: region filtering, track matching and end-of-clip track filtering on the host
(track/cliptracker.py:14-486).  The per-pixel work of the reference's methods of the same name
(``_get_filtered_frame``, ``get_delta_frame``, the per-region ``np.var``) runs in the extraction
kernel; what remains here consumes the compact region lists it emits.
"""
import logging
import math
from abc import ABC, abstractmethod

from ..ml_tools.rectangle import Rectangle
from .region import Region
from .track import Track


class ClipTracker(ABC):
    def __init__(self, config, cache_to_disk=False, keep_frames=True, calc_stats=True, verbose=False, do_tracking=True,
                 scale=None, calculate_thumbnail_info=False, max_frames=None):
        self.max_frames = max_frames
        config = config.get(self.type)
        self.scale = scale
        self.calculate_thumbnail_info = calculate_thumbnail_info
        self.do_tracking = do_tracking
        self.verbose = verbose
        self.config = config
        self.stats = None
        self.cache_to_disk = cache_to_disk
        self.max_tracks = config.max_tracks
        self.frame_padding = max(3, self.config.frame_padding)  # < 3 breaks small areas (cliptracker.py:39-40)
        self.keep_frames = keep_frames
        self.calc_stats = calc_stats
        self._tracking_time = None
        self.min_dimension = config.min_dimension
        self.background_alg = None

    @property
    @abstractmethod
    def type(self):
        ...

    @abstractmethod
    def parse_clip(self, clip, process_background=False):
        ...

    @property
    @abstractmethod
    def tracker_version(self):
        ...

    @abstractmethod
    def process_frame(self, clip, rawframe, ffc_affected=False):
        ...

    def print_if_verbose(self, info_string):
        if self.verbose:
            logging.info(info_string)

    # ------------------------------------------------------------------ H1: components -> regions of interest
    def _get_regions_of_interest(self, clip, component_details, centroids=None, variances=None):
        """cv2-style stats rows [left, top, width, height, area] (+ centroids, + per-component delta-frame
        variance from the device) -> filtered, padded ``Region`` list (cliptracker.py:263-365)."""
        regions = []
        strategy = self.config.cropped_regions_strategy
        if strategy not in ("all", "cautious", "none", None):
            raise ValueError(
                "Invalid mode for CROPPED_REGIONS_STRATEGY, expected ['all','cautious','none'] but found {}".format(strategy))
        border = math.ceil(clip.crop_rectangle.width * 0.03)
        for i, component in enumerate(component_details):
            left, top, width, height, area = (int(v) for v in component[:5])
            if centroids is None:
                centroid = [int(left + width / 2), int(top + height / 2)]
            else:
                centroid = centroids[i]
            region = Region(left, top, width, height, mass=area, id=i, frame_number=clip.current_frame, centroid=centroid)
            if self.scale:
                region.rescale(1 / self.scale)
            if region.width < self.min_dimension or region.height < self.min_dimension:
                continue
            if variances is not None:
                region.pixel_variance = variances[i]
            full_w, full_h = region.width, region.height
            before = (region.x, region.y, region.width, region.height)
            region.crop(clip.crop_rectangle)
            region.was_cropped = before != (region.x, region.y, region.width, region.height)
            if strategy == "cautious":
                if (full_w - region.width) / full_w > 0.25 or (full_h - region.height) / full_h > 0.25:
                    continue
            elif strategy in ("none", None):
                if region.was_cropped:
                    continue
            if self.config.filter_regions_pre_match and (
                region.pixel_variance < self.config.aoi_pixel_variance and region.mass < self.config.aoi_min_mass
            ):
                continue  # probably noise
            region.enlarge(self.frame_padding, max=clip.crop_rectangle)
            region.set_is_along_border(clip.crop_rectangle, edge=border)
            regions.append(region)
        return regions

    # ------------------------------------------------------------------ H2: matching
    def _apply_region_matchings(self, clip, regions):
        unmatched, matched_tracks = self._match_existing_tracks(clip, regions)
        new_tracks = self._create_new_tracks(clip, unmatched)
        lost = clip.active_tracks - matched_tracks - new_tracks
        clip.active_tracks = matched_tracks | new_tracks
        self._filter_inactive_tracks(clip, lost)
        return new_tracks

    def _match_existing_tracks(self, clip, regions):
        scores = []
        for track in sorted(clip.active_tracks, key=lambda t: t.get_id()):
            scores.extend(track.match(regions))
        # stable double sort: by score, ties by frames since the target was seen, then by track id
        # (the id enters as the decimal fraction ".<id>", cliptracker.py:147-151)
        scores.sort(key=lambda rec: rec[1].frames_since_target_seen + float(".{}".format(rec[1]._id)))
        scores.sort(key=lambda rec: rec[0])
        used = set()
        matched_tracks = set()
        blanked_tracks = set()
        for _, track, region in scores:
            if track in matched_tracks or track in blanked_tracks or id(region) in used:
                continue
            used.add(id(region))
            if not self.config.filter_regions_pre_match:
                if self.config.min_hist_diff is not None:
                    raise NotImplementedError("min_hist_diff (IR histogram filter) is not part of the thermal path")
                if region.pixel_variance < self.config.aoi_pixel_variance or region.mass < self.config.aoi_min_mass:
                    blanked_tracks.add(track)  # forces a blank frame instead of a match to another region
                    continue
            track.add_region(region)
            matched_tracks.add(track)
        # regions keep their label order (the reference iterates an identity-hashed set here, i.e. in
        # address order; label order makes simultaneous births deterministic)
        unmatched = [r for r in regions if id(r) not in used]
        return unmatched, matched_tracks

    def _create_new_tracks(self, clip, unmatched_regions):
        new_tracks = set()
        for region in unmatched_regions:
            # a tail tracked as a new object: skip regions mostly covered by an active track
            overlaps = [track.last_bound.overlap_area(region) for track in clip.active_tracks]
            if overlaps and max(overlaps) > region.area * 0.25:
                continue
            track = Track.from_region(clip, region, self.tracker_version, tracking_config=self.config)
            new_tracks.add(track)
            clip._add_active_track(track)
            self.print_if_verbose("Creating a new track {} with region {} mass{} area {} frame {}".format(
                track.get_id(), region, track.last_bound.mass, track.last_bound.area, region.frame_number))
        return new_tracks

    def _filter_inactive_tracks(self, clip, lost_tracks):
        for track in lost_tracks:
            track.add_blank_frame()
            if track.tracking:
                clip.active_tracks.add(track)

    # ------------------------------------------------------------------ H3: end of clip
    def apply_track_filtering(self, clip):
        filtered_tracks = self.filter_tracks(clip)
        if self.config.track_smoothing and clip.current_frame > 0:
            for track in clip.active_tracks:
                track.smooth(Rectangle(0, 0, clip.res_x, clip.res_y))
        return filtered_tracks

    def filter_tracks(self, clip):
        for track in clip.tracks:
            track.trim()
            track.set_end_s(clip.frames_per_second)
        for track in clip.tracks:
            track.calculate_stats()
        clip.tracks.sort(reverse=True, key=lambda t: t.stats.score)
        good, rejected = [], []
        for track in clip.tracks:
            (rejected if self.filter_track(clip, track) else good).append(track)
        clip.tracks = good
        if self.max_tracks is not None and self.max_tracks < len(clip.tracks):
            logging.warning(" -using only {0} tracks out of {1}".format(self.max_tracks, len(clip.tracks)))
            clip.filtered_tracks.extend([("Too many tracks", t) for t in clip.tracks[self.max_tracks :]])
            clip.tracks = clip.tracks[: self.max_tracks]
        for reason, track in clip.filtered_tracks:
            self.print_if_verbose("filtered track {} because {}".format(track.get_id(), reason))
        return rejected

    def filter_track(self, clip, track):
        """True (and a reason appended to ``clip.filtered_tracks``) when the track is noise (cliptracker.py:420-486)."""
        stats = track.stats
        reason = None
        if len(track) < self.config.min_duration_secs * clip.frames_per_second:
            reason = "Track filtered.  Too short"
        elif stats.max_offset < self.config.track_min_offset or stats.frames_moved < self.config.min_moving_frames:
            reason = "Track filtered.  Didn't move"
        elif stats.blank_percent > self.config.max_blank_percent:
            reason = "Track filtered. Too Many Blanks"
        elif stats.region_jitter > self.config.max_jitter:
            reason = "Track filtered.  Too Jittery"
        elif stats.delta_std < clip.track_min_delta:
            reason = "Track filtered.  Too static"
        elif stats.delta_std > clip.track_max_delta:
            reason = "Track filtered.  Too Dynamic"
        elif stats.average_mass < self.config.track_min_mass:
            reason = "Track filtered.  Mass too small"
        if reason is None:
            return False
        self.print_if_verbose(reason)
        clip.filtered_tracks.append((reason, track))
        return True


# ---------------------------------------------------------------------------------------------------------------
# background models of the IR tracker / motion detector (track/cliptracker.py:493-668)
# ---------------------------------------------------------------------------------------------------------------
import numpy as np  # noqa: E402


class Background(ABC):
    TRIGGER_FRAMES = 2

    def __init__(self):
        self.rescaled = None
        self.prev_triggered = False
        self.triggered = 0
        self.movement_detected = False
        self.kernel_trigger = np.ones((15, 15), "uint8")    # erosion when not recording
        self.kernel_recording = np.ones((10, 10), "uint8")  # erosion when recording
        self._frames = 0

    @abstractmethod
    def set_background(self, background, frames=1):
        ...

    @abstractmethod
    def update_background(self, thermal, filtered):
        ...

    @abstractmethod
    def compute_filtered(self, thermal, threshold):
        ...

    @property
    @abstractmethod
    def background(self):
        ...

    @property
    def frames(self):
        return self._frames

    def get_kernel(self):
        return self.kernel_recording if self.movement_detected else self.kernel_trigger


class CVBackground(Background):
    """OpenCV's MOG2 background subtractor (cliptracker.py:560-609).  Third-party arithmetic (cv2), on the host: it is used
    as-is when cv2 is importable and is not restated."""

    def __init__(self, tracking_alg="mog2"):
        super().__init__()
        if tracking_alg != "mog2":
            raise Exception(f"No algorihtm details found for {tracking_alg}")
        try:
            import cv2
        except ImportError as e:  # pragma: no cover
            raise ImportError("CVBackground wraps cv2.createBackgroundSubtractorMOG2 (third-party); install OpenCV or pass "
                              "another background model") from e
        self.use_subsense = False
        self.algorithm = cv2.createBackgroundSubtractorMOG2(history=1000, detectShadows=False)
        self._background = None

    def set_background(self, background, frames=1):
        self.update_background(background, learning_rate=1)

    def update_background(self, thermal, filtered=None, learning_rate=-1):
        self._background = self.algorithm.apply(thermal, None, learning_rate)
        self._frames += 1

    @property
    def background(self):
        return self.algorithm.getBackgroundImage()

    def compute_filtered(self, thermal, threshold=None):
        return self._background


class MOG2Background(Background):
    """``CVBackground`` on the device: cv2.createBackgroundSubtractorMOG2(history, var_threshold, detectShadows=False) bit for
    bit (csrc/mog2_kernels.cu), with the model's state in device memory.  Frames are host uint8 arrays or uint8 CUDA tensors
    of one geometry (fixed by the first frame).  ``update_backgrounds`` runs a whole clip's frames in one launch."""

    def __init__(self, history=1000, var_threshold=16, device=None):
        super().__init__()
        from .. import engine

        self.history, self.var_threshold = int(history), float(var_threshold)
        self.ctx = engine.get_engine(device).ctx
        self._model = None
        self._mask = None       # last foreground mask, [H][W] uint8 on the device
        self._mask_host = None  # its host copy, made on first request

    def _open(self, height, width):
        if self._model is None:
            from ..native import Mog2

            self._model = Mog2(self.ctx, width, height, history=self.history, var_threshold=self.var_threshold)
        elif (self._model.height, self._model.width) != (height, width):
            raise ValueError("MOG2Background holds {}x{} frames, got {}x{}".format(self._model.width, self._model.height, width, height))
        return self._model

    def _to_device(self, frames):
        import torch

        if isinstance(frames, torch.Tensor):
            if frames.dtype != torch.uint8 or not frames.is_cuda:
                raise ValueError("MOG2Background takes uint8 frames (host arrays or CUDA tensors)")
            return frames.contiguous()
        frames = np.ascontiguousarray(frames)
        if frames.dtype != np.uint8:
            raise ValueError("MOG2Background takes uint8 frames (host arrays or CUDA tensors)")
        return torch.from_numpy(frames).to("cuda:{}".format(self.ctx.device))

    def set_background(self, background, frames=1):
        self.update_background(background, learning_rate=1)

    def update_background(self, thermal, filtered=None, learning_rate=-1):
        frame = self._to_device(thermal)
        if frame.dim() != 2:
            raise ValueError("update_background takes one [H][W] frame")
        model, mask = self._steps(frame.shape[0], frame.shape[1], 1)
        self.ctx.use_torch_stream()
        model.apply(frame, [learning_rate], d_masks=mask)

    def _steps(self, height, width, n):
        """The model and a new [height][width] mask tensor for n apply() steps about to run on the device, here or in the IR
        motion detector's native calls; the steps are counted and the tensor becomes the last mask."""
        import torch

        model = self._open(height, width)
        self._mask = torch.empty((height, width), dtype=torch.uint8, device="cuda:{}".format(self.ctx.device))
        self._mask_host = None
        self._frames += n
        return model, self._mask

    def update_backgrounds(self, frames, learning_rate=-1):
        """apply() on frames [N][H][W] in one launch; learning_rate is a number or one per frame.  Returns the N masks, as
        host arrays for host input and as a CUDA tensor for device input."""
        import torch

        d = self._to_device(frames)
        if d.dim() != 3:
            raise ValueError("update_backgrounds takes frames [N][H][W]")
        n, h, w = d.shape
        model = self._open(h, w)
        self.ctx.use_torch_stream()
        masks = torch.empty((n, h, w), dtype=torch.uint8, device=d.device)
        lrs = np.full(n, float(learning_rate)) if np.isscalar(learning_rate) else learning_rate
        model.apply(d, lrs, d_masks=masks)
        self._frames += n
        if n:
            self._mask, self._mask_host = masks[n - 1], None
        return masks if isinstance(frames, torch.Tensor) else masks.cpu().numpy()

    @property
    def background(self):
        """getBackgroundImage() as a host array."""
        import torch

        if self._model is None:
            return None
        self.ctx.use_torch_stream()
        out = torch.empty((self._model.height, self._model.width), dtype=torch.uint8, device="cuda:{}".format(self.ctx.device))
        self._model.background(out)
        return out.cpu().numpy()

    @property
    def device_mask(self):
        """The last foreground mask (0 / 255) on the device, without a copy."""
        return self._mask

    def compute_filtered(self, thermal, threshold=None):
        """The last foreground mask as a host array (copied once, on first request)."""
        if self._mask is None:
            return None
        if self._mask_host is None:
            self._mask_host = self._mask.cpu().numpy()
        return self._mask_host


def get_diff_back_filtered(background, frame, back_thresh):
    """|frame - background| with everything below back_thresh zeroed, normalised to 0..255 (cliptracker.py:652-668);
    the normalisation runs on the device (ml_tools.imageprocessing.normalize)."""
    from ..ml_tools.imageprocessing import normalize

    filtered = np.float32(np.array(frame, copy=True))
    filtered = abs(filtered - background)
    filtered[filtered < back_thresh] = 0
    filtered, _ = normalize(filtered, new_max=255)
    return filtered


class DiffBackground(Background):
    """Mean of the frames seen so far, not updated where the frame differs from it (cliptracker.py:612-649)."""

    def __init__(self, background_thresh):
        super().__init__()
        self._frames = 1
        self._background = None
        self.background_thresh = background_thresh

    def set_background(self, background, frames=1):
        self._frames = frames
        self._background = np.float32(background) * self.frames

    def update_background(self, thermal, filtered=None):
        background = self.background
        filtered = get_diff_back_filtered(background, thermal, self.background_thresh)
        new_thermal = np.where(filtered > 0, background, thermal)
        self._background += new_thermal
        self._frames += 1

    def compute_filtered(self, thermal=None, threshold=None):
        return get_diff_back_filtered(self.background, thermal, self.background_thresh)

    @property
    def background(self):
        return self._background / self.frames
