"""ctypes binding of ``libcptrack.so`` (C ABI in ``include/cptrack.h``).

There is no CPU fallback: if the shared library is missing or a call fails, this module
raises.  Device buffers are plain ``torch`` CUDA tensors (PyTorch is only the allocator /
stream plumbing) whose ``data_ptr()`` crosses the C boundary.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CPT_LIB") or os.path.join(_HERE, "libcptrack.so")  # CPT_LIB: load another build instead (A/B of two builds in one session)

CLIP_UPDATE_BACKGROUND = 1
CLIP_RESUME = 2
CLIP_DENOISE = 4
CLIP_FRAME_STATS = 8
CLIP_SKIP_FIRST_UPDATE = 16
CLIP_PREV_IN_OUTPUT = 32
MAX_COMPONENTS = 255
MEAN_FRAMES = 45
HAS_NLM = True  # cv2.fastNlMeansDenoising on the device (batched extraction; not the frame-at-a-time streaming path)


class NativeError(RuntimeError):
    pass


class CptRegion(ctypes.Structure):
    _fields_ = [
        ("x", ctypes.c_int32), ("y", ctypes.c_int32), ("width", ctypes.c_int32), ("height", ctypes.c_int32),
        ("area", ctypes.c_int32), ("sum_x", ctypes.c_int32), ("sum_y", ctypes.c_int32), ("key", ctypes.c_int32),
        ("pixel_variance", ctypes.c_double),
    ]


class CptFrameInfo(ctypes.Structure):
    _fields_ = [
        ("background_average", ctypes.c_double), ("threshold", ctypes.c_float),
        ("norm_min", ctypes.c_int32), ("norm_max", ctypes.c_int32), ("avg_change", ctypes.c_int32),
        ("filtered_min", ctypes.c_int32), ("filtered_max", ctypes.c_int32), ("n_components", ctypes.c_int32),
        ("thermal_min", ctypes.c_int32), ("thermal_max", ctypes.c_int32), ("thermal_sum", ctypes.c_uint32),
        ("abs_filtered_sum", ctypes.c_uint32), ("thermal_median", ctypes.c_float), ("reserved", ctypes.c_int32 * 2),
    ]


class CptClip(ctypes.Structure):
    _fields_ = [
        ("frame_offset", ctypes.c_int64), ("init_offset", ctypes.c_int64), ("out_offset", ctypes.c_int64),
        ("n_frames", ctypes.c_int32), ("first_frame", ctypes.c_int32), ("ring_frames", ctypes.c_int32),
        ("background_thresh", ctypes.c_int32), ("weight_table", ctypes.c_int32), ("flags", ctypes.c_uint32),
    ]


class CptSample(ctypes.Structure):
    _fields_ = [
        ("frame", ctypes.c_int64), ("x", ctypes.c_int32), ("y", ctypes.c_int32), ("width", ctypes.c_int32),
        ("height", ctypes.c_int32), ("track", ctypes.c_int32), ("median", ctypes.c_float),
    ]


class CptTrackNorm(ctypes.Structure):
    _fields_ = [
        ("filtered_min", ctypes.c_float), ("filtered_max", ctypes.c_float), ("clip_at_zero", ctypes.c_int32),
        ("has_limits", ctypes.c_int32), ("thermal_min", ctypes.c_float), ("thermal_max", ctypes.c_float),
        ("has_thermal_limits", ctypes.c_int32), ("reserved", ctypes.c_int32),
    ]


class CptMotionResult(ctypes.Structure):
    _fields_ = [("average", ctypes.c_double), ("diff", ctypes.c_int32), ("error", ctypes.c_int32),
                ("mean_frames", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class CptMotionClipStep(ctypes.Structure):
    _fields_ = [("frame", ctypes.c_int32), ("oldest", ctypes.c_int32), ("nonffc", ctypes.c_int32), ("diff_slot_new", ctypes.c_int32),
                ("diff_slot_old", ctypes.c_int32), ("mean_first", ctypes.c_int32), ("mean_count", ctypes.c_int32),
                ("flags", ctypes.c_uint32)]


class CptMotionClip(ctypes.Structure):
    _fields_ = [("m", ctypes.c_void_p), ("d_background_state", ctypes.c_void_p), ("ring_rows", ctypes.c_void_p),
                ("init_average", ctypes.c_double), ("delta_thresh", ctypes.c_int32), ("first_step", ctypes.c_int32),
                ("n_steps", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class CptIrMotionClipStep(ctypes.Structure):
    _fields_ = [("row", ctypes.c_int64), ("slot_new", ctypes.c_int32), ("slot_oldest", ctypes.c_int32), ("detect", ctypes.c_int32),
                ("reserved", ctypes.c_int32)]


class CptIrMotionClip(ctypes.Structure):
    _fields_ = [("m", ctypes.c_void_p), ("mog2", ctypes.c_void_p), ("d_mask", ctypes.c_void_p), ("first_step", ctypes.c_int32),
                ("n_steps", ctypes.c_int32), ("movement", ctypes.c_int32), ("triggered", ctypes.c_int32)]


class CptIrMotionClipParams(ctypes.Structure):
    _fields_ = [("threshold", ctypes.c_int32), ("trigger_frames", ctypes.c_int32), ("max_triggered", ctypes.c_int32),
                ("erode_idle", ctypes.c_int32), ("erode_recording", ctypes.c_int32), ("host_frames", ctypes.c_int32)]


class CptIrMotionClipResult(ctypes.Structure):
    _fields_ = [("movement", ctypes.c_int32), ("triggered", ctypes.c_int32), ("diff_pixels", ctypes.c_int32),
                ("mask_pixels", ctypes.c_int32)]


class CptMog2Params(ctypes.Structure):
    _fields_ = [("history", ctypes.c_int), ("var_threshold", ctypes.c_double), ("background_ratio", ctypes.c_double),
                ("var_threshold_gen", ctypes.c_float), ("var_init", ctypes.c_float), ("var_min", ctypes.c_float),
                ("var_max", ctypes.c_float), ("complexity_reduction", ctypes.c_float), ("detect_shadows", ctypes.c_int)]


DETECT_CLOSE, DETECT_OPEN_GRAY, DETECT_DILATE, DETECT_OTSU, DETECT_MASK_ONLY = 1, 2, 4, 8, 16
MOTION_MEAN, MOTION_MEAN_RESTART, MOTION_BACKGROUND, MOTION_DETECT, MOTION_WARMER_ONLY, MOTION_ONE_DIFF = 1, 2, 4, 8, 16, 32


class CptOutputs(ctypes.Structure):
    _fields_ = [
        ("d_regions", ctypes.c_void_p), ("d_info", ctypes.c_void_p), ("d_filtered", ctypes.c_void_p),
        ("d_labels", ctypes.c_void_p), ("total_frames", ctypes.c_int64), ("denoise", ctypes.c_int32), ("no_resume", ctypes.c_int32),
    ]


REGION_DTYPE = np.dtype(CptRegion)
INFO_DTYPE = np.dtype(CptFrameInfo)
CLIP_DTYPE = np.dtype(CptClip)
SAMPLE_DTYPE = np.dtype(CptSample)
TRACK_NORM_DTYPE = np.dtype(CptTrackNorm)
PREPROCESS_INC3 = 1       # x / 127.5 - 1
PREPROCESS_PER_TILE = 2   # HyperParams.diff_norm off: both channels normalised by the tile's own extrema
CPTV_FRAME_DTYPE = np.dtype([("payload_offset", "<u8"), ("bit_width", "<i4"), ("reserved", "<i4")])
assert SAMPLE_DTYPE.itemsize == ctypes.sizeof(CptSample) == 32
assert TRACK_NORM_DTYPE.itemsize == ctypes.sizeof(CptTrackNorm) == 32
assert REGION_DTYPE.itemsize == ctypes.sizeof(CptRegion) == 40
assert INFO_DTYPE.itemsize == ctypes.sizeof(CptFrameInfo) == 64
assert CLIP_DTYPE.itemsize == ctypes.sizeof(CptClip) == 48
assert ctypes.sizeof(CptMotionClipStep) == 32 and ctypes.sizeof(CptMotionClip) == 48
assert ctypes.sizeof(CptIrMotionClipStep) == 24 and ctypes.sizeof(CptIrMotionClip) == 40
assert ctypes.sizeof(CptIrMotionClipParams) == 24 and ctypes.sizeof(CptIrMotionClipResult) == 16

# every symbol include/cptrack.h declares: (name, restype, argtypes)
_vp, _i, _i64, _u64, _d, _f = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_uint64, ctypes.c_double, ctypes.c_float
SYMBOLS = {
    "cpt_last_error": (ctypes.c_char_p, []),
    "cpt_device_count": (_i, []),
    "cpt_version": (_i, []),
    "cpt_ctx_create": (_vp, [_i, _i, _i, _i, _i]),
    "cpt_ctx_destroy": (None, [_vp]),
    "cpt_ctx_set_stream": (_i, [_vp, _vp]),
    "cpt_ctx_synchronize": (_i, [_vp]),
    "cpt_set_weight_table": (_i, [_vp, _i, _d, _i]),
    "cpt_build_weight_table": (_i, [_d, _i, _vp, _vp]),
    "cpt_debug_phase_cycles": (_i, [_vp, _vp, _i]),
    "cpt_debug_kernel_times_ex": (_i, [_vp, _i, _vp, _i]),
    "cpt_debug_force_single_kernel": (_i, [_vp, _i]),
    "cpt_device_alloc": (_i, [_vp, ctypes.POINTER(_vp), _u64]),
    "cpt_device_free": (_i, [_vp, _vp]),
    "cpt_host_alloc_pinned": (_i, [ctypes.POINTER(_vp), _u64]),
    "cpt_host_free_pinned": (_i, [_vp]),
    "cpt_copy_to_device": (_i, [_vp, _vp, _vp, _u64]),
    "cpt_copy_to_host": (_i, [_vp, _vp, _vp, _u64]),
    "cpt_state_bytes": (_u64, [_vp]),
    "cpt_extract_batch": (_i, [_vp, _vp, _vp, _i, ctypes.POINTER(CptOutputs), _vp]),
    "cpt_extract_batch_host": (_i, [_vp, _vp, _vp, _i, _i64, _vp, _vp, _vp, _vp, _i]),
    "cpt_background_process": (_i, [_vp, _vp, _vp, _i, _vp, _i]),
    "cpt_frame_medians": (_i, [_vp, _vp, _i64, _vp]),
    "cpt_preprocess_limits": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _i]),
    "cpt_preprocess_thermal_limits": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _i, _vp, _vp]),
    "cpt_preprocess_medians": (_i, [_vp, _vp, _vp, _vp, _i, _vp]),
    "cpt_preprocess_segments": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _i, _vp]),
    "cpt_minmax_f32": (_i, [_vp, _vp, _i64, _vp]),
    "cpt_normalize_f32": (_i, [_vp, _vp, _i64, _d, _d, _d, _i, _vp]),
    "cpt_resize_pad_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _f, _i, _vp]),
    "cpt_detect_objects": (_i, [_vp, _vp, _i, _i, _d, _i, ctypes.c_uint32, _vp, _i, _vp, _vp, _vp, _vp, ctypes.POINTER(ctypes.c_int32),
                                ctypes.POINTER(_d)]),
    "cpt_detect_objects_batch": (_i, [_vp, _vp, _i, _i, _i, _d, ctypes.c_uint32, _i, _vp, _vp, _vp, _vp]),
    "cpt_ir_merge_components": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _d, _vp, _vp]),
    "cpt_nlm_denoise_u8": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "cpt_ir_motion_open": (_vp, [_vp, _i, _i, _i]),
    "cpt_ir_motion_close": (None, [_vp]),
    "cpt_ir_motion_gray": (_i, [_vp, _vp, _i, _vp]),
    "cpt_ir_motion_detect": (_i, [_vp, _i, _i, _i, _i, _vp, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32)]),
    "cpt_ir_motion_clips": (_i, [_vp, _vp, _i, _vp, _i64, _vp, _i, ctypes.POINTER(CptIrMotionClipParams), _vp]),
    "cpt_ir_motion_step": (_i, [ctypes.POINTER(CptIrMotionClip), _vp, ctypes.POINTER(CptIrMotionClipStep), ctypes.POINTER(CptIrMotionClipParams),
                                ctypes.POINTER(CptIrMotionClipResult)]),
    "cpt_mog2_open": (_vp, [_vp, _i, _i, ctypes.POINTER(CptMog2Params)]),
    "cpt_mog2_close": (None, [_vp]),
    "cpt_mog2_apply": (_i, [_vp, _vp, _i, _i64, _vp, _vp]),
    "cpt_mog2_background": (_i, [_vp, _vp]),
    "cpt_mog2_frames": (_i, [_vp]),
    "cpt_cptv_decode": (_i, [_vp, _vp, _vp, _i, _vp, _i, _vp]),
    "cpt_extract_batch_cptv_host": (_i, [_vp, _vp, _u64, _vp, _vp, _vp, _i, _i64, _vp, _vp, _i]),
    "cpt_motion_open": (_vp, [_vp, _i, _i, _i, _i]),
    "cpt_motion_close": (None, [_vp]),
    "cpt_motion_store": (_i, [_vp, _vp, _i]),
    "cpt_motion_step": (_i, [ctypes.POINTER(CptMotionClip), _vp, ctypes.POINTER(CptMotionClipStep), _vp, _i, ctypes.POINTER(CptMotionResult)]),
    "cpt_motion_clips": (_i, [_vp, _vp, _i, _vp, _i64, _vp, _i, _vp, _i, _vp]),
    "cpt_state_read": (_i, [_vp, _vp, _i, _vp, _vp, ctypes.POINTER(_d), _vp, ctypes.POINTER(ctypes.c_int32)]),
    "cpt_state_write": (_i, [_vp, _vp, _i, _vp, _vp, _d]),
    "cpt_weight_value": (_d, [_vp, _i, _i]),
}

_lib = None


def load():
    """Load libcptrack.so; raise loudly when it is absent (no fallback path exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError(
            "libcptrack.so not found at {}: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU fallback.".format(LIB_PATH)
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise NativeError("libcptrack error {}: {}".format(rc, load().cpt_last_error().decode()))


def _ptr(t):
    """Device or host pointer of a torch tensor / numpy array / address (int) / None."""
    if t is None or isinstance(t, int):
        return t
    if isinstance(t, np.ndarray):
        return t.ctypes.data
    return t.data_ptr()


class Context:
    """One cpt_ctx: fixed geometry, one device, one stream."""

    def __init__(self, device=0, width=160, height=120, edge_pixels=1, max_regions=16):
        lib = load()
        if lib.cpt_device_count() <= 0:
            raise NativeError("no CUDA device visible: the extraction path runs on the GPU only")
        self.lib = lib
        self.device = device
        self.width, self.height, self.edge = width, height, edge_pixels
        self.max_regions = max_regions
        self._h = lib.cpt_ctx_create(device, width, height, edge_pixels, max_regions)
        if not self._h:
            raise NativeError("cpt_ctx_create failed: " + lib.cpt_last_error().decode())
        self.state_bytes = lib.cpt_state_bytes(self._h)
        self._tables = {}

    def close(self):
        if getattr(self, "_h", None):
            self.lib.cpt_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def use_torch_stream(self):
        import torch

        check(self.lib.cpt_ctx_set_stream(self._h, torch.cuda.current_stream(self.device).cuda_stream))

    def synchronize(self):
        check(self.lib.cpt_ctx_synchronize(self._h))

    def weight_table(self, weight_add, max_frames=65534):
        """Slot holding the table for ``weight_add`` (uploads it on first use)."""
        key = float(weight_add)
        if key in self._tables and self._tables[key][1] >= max_frames:
            return self._tables[key][0]
        slot = self._tables[key][0] if key in self._tables else len(self._tables)
        if slot >= 4:
            raise NativeError("at most 4 distinct weight_add values per context")
        check(self.lib.cpt_set_weight_table(self._h, slot, key, int(max_frames)))
        self._tables[key] = (slot, max_frames)
        return slot

    def weight_value(self, slot, count):
        return self.lib.cpt_weight_value(self._h, slot, int(count))

    def extract_batch(self, d_frames, d_clips, n_clips, d_regions, d_info, d_filtered=None, d_labels=None, d_state=None,
                      total_frames=0, denoise=False, no_resume=False):
        out = CptOutputs(_ptr(d_regions), _ptr(d_info), _ptr(d_filtered), _ptr(d_labels), int(total_frames), int(bool(denoise)),
                         int(bool(no_resume)))
        check(self.lib.cpt_extract_batch(self._h, _ptr(d_frames), _ptr(d_clips), int(n_clips), ctypes.byref(out), _ptr(d_state)))

    def force_single_kernel(self, enable=True):
        """Tests / diagnostics: run the single persistent kernel also where the split plan would apply."""
        check(self.lib.cpt_debug_force_single_kernel(self._h, int(bool(enable))))

    def extract_batch_host(self, h_frames, h_clips, total_frames, h_regions, h_info, h_filtered=None, h_labels=None, chunk_clips=0):
        check(
            self.lib.cpt_extract_batch_host(
                self._h, _ptr(h_frames), _ptr(h_clips), len(h_clips), int(total_frames), _ptr(h_regions), _ptr(h_info),
                _ptr(h_filtered), _ptr(h_labels), int(chunk_clips),
            )
        )

    def extract_batch_cptv_host(self, h_stream, h_table, h_clip_first, h_clips, total_frames, h_regions, h_info, chunk_clips=0):
        check(
            self.lib.cpt_extract_batch_cptv_host(
                self._h, _ptr(h_stream), int(h_stream.size), _ptr(h_table), _ptr(h_clip_first), _ptr(h_clips), len(h_clips),
                int(total_frames), _ptr(h_regions), _ptr(h_info), int(chunk_clips),
            )
        )

    def background_process(self, d_state, d_frames_i32, weight_slot, n_records=1, d_record_index=None):
        check(self.lib.cpt_background_process(self._h, _ptr(d_state), _ptr(d_record_index), int(n_records), _ptr(d_frames_i32), int(weight_slot)))

    def frame_medians(self, d_frames, n_frames, d_medians):
        check(self.lib.cpt_frame_medians(self._h, _ptr(d_frames), int(n_frames), _ptr(d_medians)))

    # d_filtered_rows: int64 filtered row per entry on an extraction's buffers (None: the entry's frame); d_frame_medians
    # float32 per thermal row and d_frame_info the extraction's INFO_DTYPE records (None: the frames are read).  Either
    # choice gives bit-identical results (include/cptrack.h)
    def preprocess_limits(self, d_filtered, d_regions, n_regions, d_tracks, n_tracks, d_filtered_rows=None):
        check(self.lib.cpt_preprocess_limits(self._h, _ptr(d_filtered), _ptr(d_filtered_rows), _ptr(d_regions), int(n_regions),
                                             _ptr(d_tracks), int(n_tracks)))

    def preprocess_thermal_limits(self, d_thermal, d_regions, n_regions, d_tracks, n_tracks, d_filtered_rows=None, d_frame_medians=None,
                                  d_frame_info=None):
        check(self.lib.cpt_preprocess_thermal_limits(self._h, _ptr(d_thermal), _ptr(d_filtered_rows), _ptr(d_regions), int(n_regions),
                                                     _ptr(d_tracks), int(n_tracks), _ptr(d_frame_medians), _ptr(d_frame_info)))

    def preprocess_medians(self, d_thermal, d_samples, n_samples, d_tracks, d_frame_medians=None):
        check(self.lib.cpt_preprocess_medians(self._h, _ptr(d_thermal), _ptr(d_frame_medians), _ptr(d_samples), int(n_samples),
                                              _ptr(d_tracks)))

    def preprocess_segments(self, d_thermal, d_filtered, d_samples, d_tracks, d_segment_samples, n_segments, tiles, per_row,
                            frame_size, crop_rectangle, preprocess_fn, d_out, d_filtered_rows=None):
        crop = None if crop_rectangle is None else (ctypes.c_int32 * 4)(*[int(v) for v in crop_rectangle])
        check(self.lib.cpt_preprocess_segments(
            self._h, _ptr(d_thermal), _ptr(d_filtered), _ptr(d_filtered_rows), _ptr(d_samples), _ptr(d_tracks), _ptr(d_segment_samples),
            int(n_segments), int(tiles), int(per_row), int(frame_size), crop, int(preprocess_fn), _ptr(d_out)))

    def minmax_f32(self, d_in, n, d_out2):
        check(self.lib.cpt_minmax_f32(self._h, _ptr(d_in), int(n), _ptr(d_out2)))

    def normalize_f32(self, d_in, n, mn, mx, new_max, use_f64, d_out):
        check(self.lib.cpt_normalize_f32(self._h, _ptr(d_in), int(n), float(mn), float(mx), float(new_max), int(use_f64), _ptr(d_out)))

    def resize_pad_f32(self, d_src, sw, sh, fw, fh, ox, oy, dw, dh, pad, interpolation, d_out):
        check(self.lib.cpt_resize_pad_f32(self._h, _ptr(d_src), int(sw), int(sh), int(fw), int(fh), int(ox), int(oy), int(dw),
                                          int(dh), float(pad), int(interpolation), _ptr(d_out)))

    def detect_objects(self, d_image, width, height, threshold, blur_ksize, steps, max_components, d_labels, d_stats, d_centroids,
                       d_or_mask=None, d_mask_out=None):
        """Returns (n_labels, threshold used)."""
        n = ctypes.c_int32()
        thr = ctypes.c_double()
        check(self.lib.cpt_detect_objects(self._h, _ptr(d_image), int(width), int(height), float(threshold), int(blur_ksize), int(steps),
                                          _ptr(d_or_mask), int(max_components), _ptr(d_labels), _ptr(d_stats), _ptr(d_centroids),
                                          _ptr(d_mask_out), ctypes.byref(n), ctypes.byref(thr)))
        return n.value, thr.value

    def detect_objects_batch(self, d_frames, n_frames, width, height, threshold, steps, max_components, d_counts, d_stats, d_centroids=None,
                             d_labels=None):
        """detect_objects_ir for n_frames frames [n][H][W] uint8 on the device (CUDA tensors or device addresses): d_counts
        int32 [n], d_stats int32 [n][max_components + 1][5], d_centroids float64 [n][max_components + 1][2] and d_labels
        int32 [n][H][W] (both may be None).  Launches on the context's stream without waiting."""
        check(self.lib.cpt_detect_objects_batch(self._h, _ptr(d_frames), int(n_frames), int(width), int(height), float(threshold), int(steps),
                                                int(max_components), _ptr(d_counts), _ptr(d_stats), _ptr(d_centroids), _ptr(d_labels)))

    def ir_merge_components(self, d_stats, d_counts, n_frames, max_components, min_mass, min_size, max_gap, d_merged, d_merged_counts):
        """merge_components for every frame of a detect_objects_batch result: d_merged int32 [n][max_components][5],
        d_merged_counts int32 [n] (-1: the frame's components overflowed).  Launches without waiting."""
        check(self.lib.cpt_ir_merge_components(self._h, _ptr(d_stats), _ptr(d_counts), int(n_frames), int(max_components), int(min_mass),
                                               int(min_size), float(max_gap), _ptr(d_merged), _ptr(d_merged_counts)))

    def motion_clips(self, h_clips, n_clips, d_frames, n_frames, h_steps, n_steps, h_mean_rows, n_mean_rows, h_results):
        """cpt_motion_clips: h_clips CptMotionClip [n_clips] (``Motion.clip_record``), h_steps CptMotionClipStep [n_steps],
        h_mean_rows int32 [n_mean_rows] and h_results CptMotionResult [n_steps] on the host; d_frames uint16 [n_frames][H][W]
        on the device."""
        check(self.lib.cpt_motion_clips(self._h, h_clips, int(n_clips), _ptr(d_frames), int(n_frames), h_steps, int(n_steps),
                                        _ptr(h_mean_rows), int(n_mean_rows), h_results))

    def ir_motion_clips(self, h_clips, n_clips, h_frames, n_frames, h_steps, n_steps, params, h_results):
        """cpt_ir_motion_clips: h_clips CptIrMotionClip [n_clips] (``IrMotion.clip_record``; movement / triggered are updated),
        h_frames uint64 [n_frames] frame addresses (host or device as ``params.host_frames`` says), h_steps
        CptIrMotionClipStep [n_steps], params CptIrMotionClipParams and h_results CptIrMotionClipResult [n_steps], all on the
        host.  Waits for the steps to finish."""
        check(self.lib.cpt_ir_motion_clips(self._h, h_clips, int(n_clips), _ptr(h_frames), int(n_frames), h_steps, int(n_steps),
                                           ctypes.byref(params), h_results))

    def nlm_denoise_u8(self, d_src, width, height, n_frames, d_dst):
        check(self.lib.cpt_nlm_denoise_u8(self._h, _ptr(d_src), int(width), int(height), int(n_frames), _ptr(d_dst)))

    def cptv_decode(self, d_stream, d_table, n_frames, d_clip_first, n_clips, d_frames):
        check(self.lib.cpt_cptv_decode(self._h, _ptr(d_stream), _ptr(d_table), int(n_frames), _ptr(d_clip_first), int(n_clips), _ptr(d_frames)))

    def state_read(self, d_state, clip_index=0, sliding_sum=False):
        bg = np.empty((self.height, self.width), np.int32)
        cnt = np.empty((self.height - 2 * self.edge, self.width - 2 * self.edge), np.uint16)
        avg = ctypes.c_double()
        seen = ctypes.c_int32()
        ssum = np.empty((self.height, self.width), np.uint32) if sliding_sum else None
        check(self.lib.cpt_state_read(self._h, _ptr(d_state), clip_index, _ptr(bg), _ptr(cnt), ctypes.byref(avg), _ptr(ssum), ctypes.byref(seen)))
        return dict(background=bg, weight_count=cnt, average=avg.value, frames_seen=seen.value, sliding_sum=ssum)

    def state_write(self, d_state, clip_index, background, weight_count, average):
        bg = np.ascontiguousarray(background, dtype=np.int32)
        cnt = None if weight_count is None else np.ascontiguousarray(weight_count, dtype=np.uint16)
        check(self.lib.cpt_state_write(self._h, _ptr(d_state), clip_index, _ptr(bg), _ptr(cnt), float(average)))


def pinned_empty(shape, dtype):
    """numpy array over cudaHostAlloc memory (freed when the array is collected)."""
    lib = load()
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    p = ctypes.c_void_p()
    check(lib.cpt_host_alloc_pinned(ctypes.byref(p), max(n, 1)))
    buf = (ctypes.c_char * max(n, 1)).from_address(p.value)

    class _Owner:
        def __init__(self, ptr):
            self.ptr = ptr

        def __del__(self):
            try:
                lib.cpt_host_free_pinned(self.ptr)
            except Exception:
                pass

    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    owner = _Owner(p.value)
    _PINNED_OWNERS[id(arr)] = owner
    import weakref

    weakref.finalize(arr, _PINNED_OWNERS.pop, id(arr), None)
    return arr


_PINNED_OWNERS = {}


class _Handle:
    """A device object of a Context: ``open(ctx, *args)`` returns its handle (NULL: NativeError), ``close`` frees it once."""

    def __init__(self, ctx, open_fn, close_fn, *args):
        self.ctx = ctx
        self._close = close_fn
        self._h = open_fn(ctx._h, *args)
        if not self._h:
            raise NativeError("{} failed: {}".format(open_fn.__name__, ctx.lib.cpt_last_error().decode()))

    @property
    def address(self):
        """Address of the native object (None once closed), for inspecting its device buffers."""
        return self._h

    def close(self):
        if getattr(self, "_h", None):
            self._close(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _IrMotionHead(ctypes.Structure):  # the leading members of struct cpt_ir_motion (csrc/ir_kernels.cu)
    _fields_ = [("ctx", _vp), ("W", _i), ("H", _i), ("ring_frames", _i), ("d_ring", _vp)]


class IrMotion(_Handle):
    """Device half of IRMotionDetector (cpt_ir_motion_*): a ring of grey frames, grey conversion and the eroded-pixel counts."""

    def __init__(self, ctx, width, height, ring_frames):
        self.width, self.height, self.ring_frames = width, height, ring_frames
        super().__init__(ctx, ctx.lib.cpt_ir_motion_open, ctx.lib.cpt_ir_motion_close, int(width), int(height), int(ring_frames))

    def gray(self, bgr, slot, copy_out=True):
        """BGR frame -> grey into ring slot ``slot``; returns the grey frame as a host array, or None with copy_out=False."""
        bgr = np.ascontiguousarray(bgr, dtype=np.uint8)
        if bgr.shape != (self.height, self.width, 3):
            raise ValueError("IR frames must be ({}, {}, 3) uint8".format(self.height, self.width))
        out = np.empty((self.height, self.width), np.uint8) if copy_out else None
        check(self.ctx.lib.cpt_ir_motion_gray(self._h, _ptr(bgr), int(slot), _ptr(out)))
        return out

    def ring_slot(self, slot):
        """Device address of the grey frame in ring slot ``slot`` ([H][W] uint8), for inspecting the ring."""
        if not 0 <= slot < self.ring_frames:
            raise NativeError("ring slot {} out of range".format(slot))
        return _IrMotionHead.from_address(self._h).d_ring + slot * self.width * self.height

    def detect(self, slot_new, slot_oldest, threshold, erode_k, mask=None):
        """(eroded difference pixels, eroded mask pixels) with the host foreground mask ``mask`` (or None)."""
        diff, cnt = ctypes.c_int32(), ctypes.c_int32()
        if mask is not None:
            mask = np.ascontiguousarray(mask, dtype=np.uint8)
        check(self.ctx.lib.cpt_ir_motion_detect(self._h, int(slot_new), int(slot_oldest), int(threshold), int(erode_k), _ptr(mask),
                                                ctypes.byref(diff), ctypes.byref(cnt)))
        return diff.value, cnt.value

    def step(self, clip, bgr, step, params):
        """One step of ``Context.ir_motion_clips`` for this detector alone (cpt_ir_motion_step): ``clip`` its CptIrMotionClip
        (``clip_record``; movement / triggered are updated), bgr a host [H][W][3] uint8 frame, ``step`` its CptIrMotionClipStep
        and ``params`` the CptIrMotionClipParams.  Waits and returns the CptIrMotionClipResult."""
        result, bgr = CptIrMotionClipResult(), np.ascontiguousarray(bgr)  # bgr: a contiguous copy lives until the call returns
        check(self.ctx.lib.cpt_ir_motion_step(ctypes.byref(clip), _ptr(bgr), ctypes.byref(step), ctypes.byref(params), ctypes.byref(result)))
        return result

    def clip_record(self, mog2, d_mask, first_step, n_steps, movement, triggered):
        """This detector's CptIrMotionClip of a ``Context.ir_motion_clips`` call or of ``step``: ``mog2`` its ``Mog2`` model, ``d_mask`` the
        [H][W] uint8 CUDA tensor that receives the foreground masks."""
        return CptIrMotionClip(self._h, mog2.address, _dptr(d_mask, self.height * self.width), int(first_step), int(n_steps),
                               int(bool(movement)), int(triggered))


def _dptr(t, min_bytes):
    """Device address of a uint8 CUDA tensor (at least min_bytes, contiguous) or a raw device address (int)."""
    if isinstance(t, int):
        return t
    if not (getattr(t, "is_cuda", False) and str(t.dtype) == "torch.uint8" and t.is_contiguous() and t.numel() >= min_bytes):
        raise ValueError("expected a contiguous uint8 CUDA tensor of at least {} bytes".format(min_bytes))
    return t.data_ptr()


class Mog2(_Handle):
    """OpenCV's BackgroundSubtractorMOG2 (detectShadows=False, one uint8 channel) on the device, bit for bit (cpt_mog2_*).
    The model's state stays in device memory; frames and masks are uint8 CUDA tensors or device addresses.  Calls launch on
    the context's stream and return without waiting."""

    def __init__(self, ctx, width, height, history=500, var_threshold=16.0, background_ratio=0.9, var_threshold_gen=9.0,
                 var_init=15.0, var_min=4.0, var_max=75.0, complexity_reduction=0.05, detect_shadows=False):
        self.width, self.height = int(width), int(height)
        self.params = CptMog2Params(int(history), float(var_threshold), float(background_ratio), float(var_threshold_gen), float(var_init),
                                    float(var_min), float(var_max), float(complexity_reduction), int(bool(detect_shadows)))
        super().__init__(ctx, ctx.lib.cpt_mog2_open, ctx.lib.cpt_mog2_close, self.width, self.height, ctypes.byref(self.params))

    @property
    def frame_bytes(self):
        return self.width * self.height

    def apply(self, d_frames, learning_rates, d_masks=None, n_frames=None, frame_stride=None):
        """apply() for consecutive frames: d_frames [n][H][W] (or [H][W]) uint8 on the device, learning_rates one cv2
        learningRate per frame (a number applies to all).  Writes n masks (0 / 255) to d_masks when given."""
        n = n_frames
        if n is None:
            if isinstance(d_frames, int):
                raise ValueError("n_frames is required with a device address")
            if tuple(d_frames.shape[-2:]) != (self.height, self.width):
                raise ValueError("MOG2 frames must be [..., {}, {}] uint8".format(self.height, self.width))
            n = 1 if d_frames.dim() == 2 else int(d_frames.shape[0])
        stride = self.frame_bytes if frame_stride is None else int(frame_stride)
        lrs = np.full(n, float(learning_rates), np.float64) if np.isscalar(learning_rates) else np.ascontiguousarray(learning_rates, np.float64)
        if lrs.shape != (n,):
            raise ValueError("one learning rate per frame")
        if n == 0:
            return
        fp = _dptr(d_frames, stride * (n - 1) + self.frame_bytes)
        mp = None if d_masks is None else _dptr(d_masks, n * self.frame_bytes)
        check(self.ctx.lib.cpt_mog2_apply(self._h, fp, int(n), int(stride), lrs.ctypes.data, mp))

    def background(self, d_out):
        """getBackgroundImage() into d_out ([H][W] uint8 on the device)."""
        check(self.ctx.lib.cpt_mog2_background(self._h, _dptr(d_out, self.frame_bytes)))

    @property
    def frames(self):
        n = self.ctx.lib.cpt_mog2_frames(self._h)
        if n < 0:
            check(n)
        return n


class Motion(_Handle):
    """Device half of CPTVMotionDetector (cpt_motion_*): the ring of frames, the running sum and the ring of delta frames.
    Ring bookkeeping (which slot is newest / oldest / oldest non-FFC) stays with the caller."""

    def __init__(self, ctx, ring_frames, mean_frames, diff_frames, weight_slot):
        super().__init__(ctx, ctx.lib.cpt_motion_open, ctx.lib.cpt_motion_close, int(ring_frames), int(mean_frames), int(diff_frames),
                         int(weight_slot))

    def store(self, h_pix, slot):
        """Host uint16 frame [H][W] into ring slot ``slot`` without processing it."""
        check(self.ctx.lib.cpt_motion_store(self._h, _ptr(h_pix), int(slot)))

    def step(self, clip, h_pix, step, mean_rows=()):
        """One process_frame (cpt_motion_step) of the detector record ``clip`` (``clip_record``): h_pix (host uint16 [H][W])
        into ring slot -1 - step[0], then the step with the cpt_motion_clip_step fields ``step`` (every frame reference a ring
        slot; the RunningMean start reads ``mean_rows``).  Waits for it and returns its CptMotionResult."""
        result = CptMotionResult()
        rows = (ctypes.c_int32 * len(mean_rows))(*mean_rows) if len(mean_rows) else None
        check(self.ctx.lib.cpt_motion_step(ctypes.byref(clip), _ptr(h_pix), ctypes.byref(CptMotionClipStep(*step)), rows, len(mean_rows),
                                           ctypes.byref(result)))
        return result

    def clip_record(self, d_background_state, ring_rows, init_average, delta_thresh, first_step, n_steps):
        """This detector's CptMotionClip of a ``Context.motion_clips`` call (ring_rows: host int32 [ring_frames]) or of ``step``."""
        return CptMotionClip(self._h, _ptr(d_background_state), _ptr(ring_rows), float(init_average), int(delta_thresh), int(first_step),
                             int(n_steps), 0)
