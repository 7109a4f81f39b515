"""``Clip`` and ``ClipStats``: per-recording state and JSON metadata (track/clip.py:38-501)."""
import datetime
import os
import zoneinfo

import numpy as np

from ..ml_tools.rectangle import Rectangle
from .framebuffer import FrameBuffer
from .track import Track

RES_X = 160
RES_Y = 120


class Clip:
    PREVIEW = "preview"
    FRAMES_PER_SECOND = 9
    local_tz = zoneinfo.ZoneInfo("Pacific/Auckland")
    CLIP_ID = 1  # parity: process-global counters, as in the reference (clip.py:42,55-59)

    def __init__(self, trackconfig, sourcefile, background=None, calc_stats=True, model=None, type="thermal",
                 fps=FRAMES_PER_SECOND):
        self._id = Clip.CLIP_ID
        Clip.CLIP_ID += 1
        Track._track_id = 1
        self.disable_background_subtraction = False
        self.current_frame = -1
        self.ffc_affected = False
        self.crop_rectangle = None
        self.region_history = []
        self.active_tracks = set()
        self.tracks = []
        self.filtered_tracks = []
        self.from_metadata = False
        self.video_start_time = None
        self.location = None
        self.frame_buffer = None
        self.device_frames = None  # batch.ClipDeviceFrames after parse_clips(keep_on_device=True)
        self.device = None
        self._background = None
        self.background_calculated = False
        self.res_x = None
        self.res_y = None
        self.background_frames = 0
        self.config = trackconfig
        self.frames_per_second = fps
        self.station_id = None
        self.calc_stats = calc_stats
        self.source_file = sourcefile
        self.stats = ClipStats()
        self.camera_model = None
        self.threshold_config = None
        self.track_min_delta = None
        self.track_max_delta = None
        self.background_thresh = None
        self.temp_thresh = None
        self.ffc_frames = []
        self.tags = None
        self.type = type
        self.thumb_info = None
        self.rescaled = None
        self.set_model(model)
        if background is not None:
            self._background = background
            self._background_calculated()

    # ------------------------------------------------------------------ configuration
    def set_model(self, camera_model):
        self.camera_model = camera_model
        threshold = self.config.motion.threshold_for_model(camera_model)
        if threshold:
            self.threshold_config = threshold
            self.set_motion_thresholds(threshold)

    def set_motion_thresholds(self, threshold):
        self.background_thresh = threshold.background_thresh
        self.temp_thresh = threshold.temp_thresh
        self.stats.threshold = self.background_thresh
        self.track_min_delta = threshold.track_min_delta
        self.track_max_delta = threshold.track_max_delta

    def set_res(self, res_x, res_y):
        self.res_x = res_x if res_x else RES_X
        self.res_y = res_y if res_y else RES_Y
        self._set_crop_rectangle()
        for track in self.tracks:
            track.crop_rectangle = self.crop_rectangle

    def _set_crop_rectangle(self):
        edge = self.config.edge_pixels
        self.crop_rectangle = Rectangle(edge, edge, self.res_x - 2 * edge, self.res_y - 2 * edge)

    def set_frame_buffer(self, high_quality_flow, cache_to_disk, use_flow, keep_frames, max_frames=None):
        self.frame_buffer = FrameBuffer(self.source_file, high_quality_flow, cache_to_disk, use_flow, keep_frames, max_frames)

    def set_video_stats(self, video_start_time):
        self.video_start_time = video_start_time
        local = video_start_time.astimezone(Clip.local_tz)
        self.stats.date_time = local
        self.stats.is_night = local.time().hour >= 2

    # ------------------------------------------------------------------ background frame (clip-level)
    @property
    def background(self):
        return self._background

    def _background_calculated(self):
        if self.type != "IR" or self.calc_stats:
            self.stats.mean_background_value = np.average(self._background)
        self.background_calculated = True

    def on_preview(self):
        return not self.background_calculated

    def set_background(self, frame):
        self._background = frame
        self._background_calculated()

    def update_background(self, frame):
        self._background = frame if self._background is None else np.minimum(self._background, frame)
        self.background_frames += 1

    def calculate_background(self, frame_reader):
        frame = frame_reader.next_frame()
        self.update_background(frame.pix)
        self._background_calculated()

    # ------------------------------------------------------------------ frames / tracks
    def get_frame(self, frame_number):
        return self.frame_buffer.get_frame(frame_number)

    def frames_kept(self):
        return self.frame_buffer.max_frames

    def get_id(self):
        return str(self._id)

    def _add_active_track(self, track):
        self.active_tracks.add(track)
        self.tracks.append(track)

    def add_frame(self, thermal, filtered, mask=None, ffc_affected=False, frame_stats=None):
        """``frame_stats``: (median, max, min, mean, sum|filtered|) from the device (K8) instead of numpy."""
        self.current_frame += 1
        if ffc_affected:
            self.ffc_frames.append(self.current_frame)
        frame = self.frame_buffer.add_frame(thermal, filtered, mask, self.current_frame, ffc_affected)
        if self.calc_stats:
            if frame_stats is not None:
                self.stats.add_frame_stats(*frame_stats)
            else:
                self.stats.add_frame(thermal, filtered)
        return frame

    def start_and_end_in_secs(self, track):
        if track.end_s is None:
            track.end_s = (track.end_frame + 1) / self.frames_per_second
        return (track.start_s, track.end_s)

    def start_and_end_time_absolute(self, start_s=0, end_s=None):
        if not end_s:
            end_s = len(self.frame_buffer.frames) / self.frames_per_second
        return (self.video_start_time + datetime.timedelta(seconds=start_s),
                self.video_start_time + datetime.timedelta(seconds=end_s))

    # ------------------------------------------------------------------ metadata
    def load_metadata(self, metadata, tag_precedence=None):
        self._id = metadata.get("id", 0)
        device_meta = metadata.get("Device")
        self.tags = metadata.get("Tags")
        if device_meta:
            self.device = device_meta.get("devicename")
        else:
            self.device = os.path.splitext(os.path.basename(self.source_file))[0].split("-")[-1]
        self.location = metadata.get("location")
        self.station_id = metadata.get("stationId")
        self.tracks = set(self.load_tracks_meta(metadata, tag_precedence))
        self.from_metadata = True

    def load_tracks_meta(self, metadata, tag_precedence):
        tracks = []
        for track_meta in (metadata.get("Tracks", []) if "Tracks" in metadata else metadata.get("tracks", [])):
            track = Track(self.get_id())
            if track.load_track_meta(track_meta, self.frames_per_second, tag_precedence, self.config.min_tag_confidence):
                tracks.append(track)
        return tracks

    def get_metadata(self, predictions_per_model=None):
        """Key order of clip.py:436-452."""
        meta = {}
        if self.camera_model:
            meta["camera_model"] = self.camera_model
        meta["background_thresh"] = self.background_thresh
        start, end = self.start_and_end_time_absolute()
        meta["id"] = self._id
        meta["start_time"] = start.isoformat()
        meta["end_time"] = end.isoformat()
        meta["tracks"] = [track.get_metadata(predictions_per_model) for track in self.tracks]
        return meta


class ClipStats:
    """Per-frame thermal statistics (clip.py:455-492)."""

    def __init__(self):
        self.mean_background_value = 0
        self.max_temp = None
        self.min_temp = None
        self.mean_temp = None
        self.frame_stats_min = []
        self.frame_stats_max = []
        self.frame_stats_median = []
        self.frame_stats_mean = []
        self.filtered_deviation = None
        self.filtered_sum = 0
        self.temp_thresh = 0
        self.threshold = None
        self.average_delta = None
        self.is_static_background = None

    def add_frame(self, thermal, filtered=None):
        self.add_frame_stats(np.median(thermal), np.max(thermal), np.min(thermal), np.nanmean(thermal),
                             None if filtered is None else np.sum(np.abs(filtered)))

    def add_frame_stats(self, f_median, f_max, f_min, f_mean, abs_filtered_sum=None):
        self.max_temp = f_max if self.max_temp is None else max(self.max_temp, f_max)
        self.min_temp = f_min if self.min_temp is None else min(self.min_temp, f_min)
        self.frame_stats_min.append(f_min)
        self.frame_stats_max.append(f_max)
        self.frame_stats_median.append(f_median)
        self.frame_stats_mean.append(f_mean)
        if abs_filtered_sum is not None:
            self.filtered_sum += np.float64(abs_filtered_sum)

    def completed(self):
        # parity: the reference casts the float64 totals to uint16 (clip.py:489-492); out-of-range values wrap
        with np.errstate(invalid="ignore", over="ignore"):
            if self.filtered_sum is not None:
                self.filtered_deviation = np.mean(np.asarray(self.filtered_sum, dtype=np.float64).astype(np.int64).astype(np.uint16))
            self.mean_temp = np.mean(np.asarray(self.frame_stats_mean, dtype=np.float64).astype(np.int64).astype(np.uint16))
