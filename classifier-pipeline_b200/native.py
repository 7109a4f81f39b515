"""ctypes binding of ``libcptrack.so`` (C ABI in ``include/cptrack.h``).

There is no CPU fallback: if the shared library is missing or a call fails, this module
raises.  Device buffers are plain ``torch`` CUDA tensors (PyTorch is only the allocator /
stream plumbing) whose ``data_ptr()`` crosses the C boundary.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CPT_LIB") or os.path.join(_HERE, "libcptrack.so")  # CPT_LIB: an experimental build (tools/)

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


DETECT_CLOSE, DETECT_OPEN_GRAY, DETECT_DILATE, DETECT_OTSU, DETECT_MASK_ONLY = 1, 2, 4, 8, 16
MOTION_MEAN, MOTION_MEAN_RESTART, MOTION_BACKGROUND, MOTION_DETECT, MOTION_WARMER_ONLY, MOTION_ONE_DIFF = 1, 2, 4, 8, 16, 32


class CptOutputs(ctypes.Structure):
    _fields_ = [
        ("d_regions", ctypes.c_void_p), ("d_info", ctypes.c_void_p), ("d_filtered", ctypes.c_void_p),
        ("d_labels", ctypes.c_void_p), ("total_frames", ctypes.c_int64), ("denoise", ctypes.c_int32), ("no_resume", ctypes.c_int32),
    ]


REGION_DTYPE = np.dtype(
    [("x", "<i4"), ("y", "<i4"), ("width", "<i4"), ("height", "<i4"), ("area", "<i4"), ("sum_x", "<i4"),
     ("sum_y", "<i4"), ("key", "<i4"), ("pixel_variance", "<f8")]
)
INFO_DTYPE = np.dtype(
    [("background_average", "<f8"), ("threshold", "<f4"), ("norm_min", "<i4"), ("norm_max", "<i4"),
     ("avg_change", "<i4"), ("filtered_min", "<i4"), ("filtered_max", "<i4"), ("n_components", "<i4"),
     ("thermal_min", "<i4"), ("thermal_max", "<i4"), ("thermal_sum", "<u4"), ("abs_filtered_sum", "<u4"),
     ("thermal_median", "<f4"), ("reserved", "<i4", (2,))]
)
CLIP_DTYPE = np.dtype(
    [("frame_offset", "<i8"), ("init_offset", "<i8"), ("out_offset", "<i8"), ("n_frames", "<i4"),
     ("first_frame", "<i4"), ("ring_frames", "<i4"), ("background_thresh", "<i4"), ("weight_table", "<i4"),
     ("flags", "<u4")]
)
SAMPLE_DTYPE = np.dtype(
    [("frame", "<i8"), ("x", "<i4"), ("y", "<i4"), ("width", "<i4"), ("height", "<i4"), ("track", "<i4"), ("median", "<f4")]
)
TRACK_NORM_DTYPE = np.dtype([("filtered_min", "<f4"), ("filtered_max", "<f4"), ("clip_at_zero", "<i4"), ("has_limits", "<i4"),
                             ("thermal_min", "<f4"), ("thermal_max", "<f4"), ("has_thermal_limits", "<i4"), ("reserved", "<i4")])
PREPROCESS_INC3 = 1       # x / 127.5 - 1
PREPROCESS_PER_TILE = 2   # HyperParams.diff_norm off: both channels normalised by the tile's own extrema
CPTV_FRAME_DTYPE = np.dtype([("payload_offset", "<u8"), ("bit_width", "<i4"), ("reserved", "<i4")])
assert SAMPLE_DTYPE.itemsize == ctypes.sizeof(CptSample) == 32
assert TRACK_NORM_DTYPE.itemsize == ctypes.sizeof(CptTrackNorm) == 32
assert REGION_DTYPE.itemsize == ctypes.sizeof(CptRegion) == 40
assert INFO_DTYPE.itemsize == ctypes.sizeof(CptFrameInfo) == 64
assert CLIP_DTYPE.itemsize == ctypes.sizeof(CptClip) == 48

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
    "cpt_debug_kernel_times": (_i, [_vp, _i, _vp]),
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
    "cpt_preprocess_limits": (_i, [_vp, _vp, _vp, _i, _vp, _i]),
    "cpt_preprocess_thermal_limits": (_i, [_vp, _vp, _vp, _i, _vp, _i]),
    "cpt_preprocess_medians": (_i, [_vp, _vp, _vp, _i, _vp]),
    "cpt_preprocess_segments": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _i, _vp]),
    "cpt_preprocess_limits_ex": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _i]),
    "cpt_preprocess_thermal_limits_ex": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _i, _vp, _vp]),
    "cpt_preprocess_medians_ex": (_i, [_vp, _vp, _vp, _vp, _i, _vp]),
    "cpt_preprocess_segments_ex": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _i, _vp]),
    "cpt_minmax_f32": (_i, [_vp, _vp, _i64, _vp]),
    "cpt_normalize_f32": (_i, [_vp, _vp, _i64, _d, _d, _d, _i, _vp]),
    "cpt_resize_pad_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _f, _i, _vp]),
    "cpt_detect_objects_u8": (_i, [_vp, _vp, _i, _i, _d, _i, _i, _i, _vp, _vp, _vp, ctypes.POINTER(ctypes.c_int32)]),
    "cpt_detect_objects_ex": (_i, [_vp, _vp, _i, _i, _d, _i, ctypes.c_uint32, _vp, _i, _vp, _vp, _vp, _vp, ctypes.POINTER(ctypes.c_int32),
                                   ctypes.POINTER(_d)]),
    "cpt_nlm_denoise_u8": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "cpt_ir_motion_open": (_vp, [_vp, _i, _i, _i]),
    "cpt_ir_motion_close": (None, [_vp]),
    "cpt_ir_motion_gray": (_i, [_vp, _vp, _i, _vp]),
    "cpt_ir_motion_detect": (_i, [_vp, _i, _i, _i, _i, _vp, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32)]),
    "cpt_cptv_decode": (_i, [_vp, _vp, _vp, _i, _vp, _i, _vp]),
    "cpt_extract_batch_cptv_host": (_i, [_vp, _vp, _u64, _vp, _vp, _vp, _i, _i64, _vp, _vp, _i]),
    "cpt_motion_open": (_vp, [_vp, _i, _i, _i, _i]),
    "cpt_motion_close": (None, [_vp]),
    "cpt_motion_store": (_i, [_vp, _vp, _i]),
    "cpt_motion_mean_init": (_i, [_vp, _vp, _i]),
    "cpt_motion_step": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, ctypes.c_uint32, _i, _d, ctypes.POINTER(CptMotionResult)]),
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
    """Device or host pointer of a torch tensor / numpy array / None."""
    if t is None:
        return None
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

    def preprocess_limits(self, d_filtered, d_regions, n_regions, d_tracks, n_tracks):
        check(self.lib.cpt_preprocess_limits(self._h, _ptr(d_filtered), _ptr(d_regions), int(n_regions), _ptr(d_tracks), int(n_tracks)))

    def preprocess_thermal_limits(self, d_thermal, d_regions, n_regions, d_tracks, n_tracks):
        check(self.lib.cpt_preprocess_thermal_limits(self._h, _ptr(d_thermal), _ptr(d_regions), int(n_regions), _ptr(d_tracks), int(n_tracks)))

    def preprocess_medians(self, d_thermal, d_samples, n_samples, d_tracks):
        check(self.lib.cpt_preprocess_medians(self._h, _ptr(d_thermal), _ptr(d_samples), int(n_samples), _ptr(d_tracks)))

    def preprocess_segments(self, d_thermal, d_filtered, d_samples, d_tracks, d_segment_samples, n_segments, tiles, per_row,
                            frame_size, crop_rectangle, preprocess_fn, d_out):
        crop = None if crop_rectangle is None else (ctypes.c_int32 * 4)(*[int(v) for v in crop_rectangle])
        check(self.lib.cpt_preprocess_segments(
            self._h, _ptr(d_thermal), _ptr(d_filtered), _ptr(d_samples), _ptr(d_tracks), _ptr(d_segment_samples), int(n_segments),
            int(tiles), int(per_row), int(frame_size), crop, int(preprocess_fn), _ptr(d_out)))

    # the same passes on an extraction's buffers (include/cptrack.h, cpt_preprocess_*_ex): d_filtered_rows int64 per entry
    # (None: the entry's frame), d_frame_medians float32 per thermal row, d_frame_info the extraction's INFO_DTYPE records
    def preprocess_limits_ex(self, d_filtered, d_filtered_rows, d_regions, n_regions, d_tracks, n_tracks):
        check(self.lib.cpt_preprocess_limits_ex(self._h, _ptr(d_filtered), _ptr(d_filtered_rows), _ptr(d_regions), int(n_regions),
                                                _ptr(d_tracks), int(n_tracks)))

    def preprocess_thermal_limits_ex(self, d_thermal, d_filtered_rows, d_regions, n_regions, d_tracks, n_tracks, d_frame_medians=None,
                                     d_frame_info=None):
        check(self.lib.cpt_preprocess_thermal_limits_ex(self._h, _ptr(d_thermal), _ptr(d_filtered_rows), _ptr(d_regions), int(n_regions),
                                                        _ptr(d_tracks), int(n_tracks), _ptr(d_frame_medians), _ptr(d_frame_info)))

    def preprocess_medians_ex(self, d_thermal, d_frame_medians, d_samples, n_samples, d_tracks):
        check(self.lib.cpt_preprocess_medians_ex(self._h, _ptr(d_thermal), _ptr(d_frame_medians), _ptr(d_samples), int(n_samples),
                                                 _ptr(d_tracks)))

    def preprocess_segments_ex(self, d_thermal, d_filtered, d_filtered_rows, d_samples, d_tracks, d_segment_samples, n_segments, tiles,
                               per_row, frame_size, crop_rectangle, preprocess_fn, d_out):
        crop = None if crop_rectangle is None else (ctypes.c_int32 * 4)(*[int(v) for v in crop_rectangle])
        check(self.lib.cpt_preprocess_segments_ex(
            self._h, _ptr(d_thermal), _ptr(d_filtered), _ptr(d_filtered_rows), _ptr(d_samples), _ptr(d_tracks), _ptr(d_segment_samples),
            int(n_segments), int(tiles), int(per_row), int(frame_size), crop, int(preprocess_fn), _ptr(d_out)))

    def minmax_f32(self, d_in, n, d_out2):
        check(self.lib.cpt_minmax_f32(self._h, _ptr(d_in), int(n), _ptr(d_out2)))

    def normalize_f32(self, d_in, n, mn, mx, new_max, use_f64, d_out):
        check(self.lib.cpt_normalize_f32(self._h, _ptr(d_in), int(n), float(mn), float(mx), float(new_max), int(use_f64), _ptr(d_out)))

    def resize_pad_f32(self, d_src, sw, sh, fw, fh, ox, oy, dw, dh, pad, interpolation, d_out):
        check(self.lib.cpt_resize_pad_f32(self._h, _ptr(d_src), int(sw), int(sh), int(fw), int(fh), int(ox), int(oy), int(dw),
                                          int(dh), float(pad), int(interpolation), _ptr(d_out)))

    def detect_objects_u8(self, d_image, width, height, threshold, blur_ksize, close, max_components, d_labels, d_stats, d_centroids):
        n = ctypes.c_int32()
        check(self.lib.cpt_detect_objects_u8(self._h, _ptr(d_image), int(width), int(height), float(threshold), int(blur_ksize),
                                             int(close), int(max_components), _ptr(d_labels), _ptr(d_stats), _ptr(d_centroids),
                                             ctypes.byref(n)))
        return n.value

    def detect_objects_ex(self, d_image, width, height, threshold, blur_ksize, steps, max_components, d_labels, d_stats, d_centroids,
                          d_or_mask=None, d_mask_out=None):
        """Returns (n_labels, threshold used)."""
        n = ctypes.c_int32()
        thr = ctypes.c_double()
        check(self.lib.cpt_detect_objects_ex(self._h, _ptr(d_image), int(width), int(height), float(threshold), int(blur_ksize), int(steps),
                                             _ptr(d_or_mask), int(max_components), _ptr(d_labels), _ptr(d_stats), _ptr(d_centroids),
                                             _ptr(d_mask_out), ctypes.byref(n), ctypes.byref(thr)))
        return n.value, thr.value

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


class IrMotion:
    """Device half of IRMotionDetector (cpt_ir_motion_*): a ring of grey frames, grey conversion and the eroded-pixel counts."""

    def __init__(self, ctx, width, height, ring_frames):
        self.ctx = ctx
        self.width, self.height, self.ring_frames = width, height, ring_frames
        self._h = ctx.lib.cpt_ir_motion_open(ctx._h, int(width), int(height), int(ring_frames))
        if not self._h:
            raise NativeError("cpt_ir_motion_open failed: {}".format(ctx.lib.cpt_last_error().decode()))

    def gray(self, bgr, slot):
        bgr = np.ascontiguousarray(bgr, dtype=np.uint8)
        if bgr.shape != (self.height, self.width, 3):
            raise ValueError("IR frames must be ({}, {}, 3) uint8".format(self.height, self.width))
        out = np.empty((self.height, self.width), np.uint8)
        check(self.ctx.lib.cpt_ir_motion_gray(self._h, _ptr(bgr), int(slot), _ptr(out)))
        return out

    def detect(self, slot_new, slot_oldest, threshold, erode_k, mask=None):
        diff, cnt = ctypes.c_int32(), ctypes.c_int32()
        if mask is not None:
            mask = np.ascontiguousarray(mask, dtype=np.uint8)
        check(self.ctx.lib.cpt_ir_motion_detect(self._h, int(slot_new), int(slot_oldest), int(threshold), int(erode_k), _ptr(mask),
                                                ctypes.byref(diff), ctypes.byref(cnt)))
        return diff.value, cnt.value

    def close(self):
        if self._h:
            self.ctx.lib.cpt_ir_motion_close(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
