/*
 * cptrack.h -- C ABI of libcptrack.so: B200 (sm_100a) kernels for classifier-pipeline's
 * track-extraction and classifier-input preprocessing path.
 *
 * The reference has no FFI layer of its own (it is pure Python over numpy/OpenCV wheels); the
 * entry points below are what its Python classes bind instead of those wheels.  Each one cites
 * the reference interface (path:line under the reference's src/) whose arithmetic it replaces.
 * INTEGRATION.md shows the ctypes stubs a maintainer adds on the reference side.
 *
 * Conventions: every function returns 0 on success or a negative CPT_ERR_* code and records a
 * message readable with cpt_last_error() (thread local).  A cpt_ctx is bound to one CUDA
 * device and one stream and is not thread safe; use one ctx per host thread / per GPU.
 * Pointers named d_* are device pointers (cudaMalloc / torch tensor .data_ptr()), h_* are host
 * pointers; the caller owns every buffer it passes in.  No torch types cross this boundary.
 */
#ifndef CPTRACK_H
#define CPTRACK_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CPT_OK 0
#define CPT_ERR_INVALID (-1)     /* bad argument (geometry, NULL, sizes) */
#define CPT_ERR_CUDA (-2)        /* CUDA runtime error, see cpt_last_error() */
#define CPT_ERR_UNSUPPORTED (-3) /* option not available in this build */
#define CPT_ERR_NOMEM (-4)

#define CPT_MEAN_FRAMES 45       /* track/cliptrackextractor.py:173 get_last_x(x=45) */
#define CPT_MAX_COMPONENTS 255   /* labels are written as uint8; more components => overflow flag */

/* clip flags */
#define CPT_CLIP_UPDATE_BACKGROUND 1u /* ClipTrackExtractor(update_background=True), cliptrackextractor.py:168-176 */
#define CPT_CLIP_RESUME 2u            /* continue from the state saved in d_state instead of initialising */
#define CPT_CLIP_DENOISE 4u           /* TrackingConfig.denoise: cv2.fastNlMeansDenoising, cliptracker.py:116-117 (set cpt_outputs.denoise too) */
#define CPT_CLIP_FRAME_STATS 8u       /* ClipStats.add_frame, clip.py:474-487 (min/max/median/mean, sum|filtered|) */
#define CPT_CLIP_SKIP_FIRST_UPDATE 16u /* RawDatabase.load_frames, ml_tools/rawdb.py:84-122: the frame that initialised the
                                          background is also the first kept frame and is not followed by a background update */
#define CPT_CLIP_PREV_IN_OUTPUT 32u   /* with CPT_CLIP_RESUME | CPT_CLIP_DENOISE (frame-at-a-time denoise): the caller has put the
                                          previous frame's filtered image and cpt_frame_info at output index out_offset - 1, where
                                          the passes that follow the denoise (mask, components, variance) look for them */

typedef struct cpt_ctx cpt_ctx;

/* One connected component of the closed mask == one row of
 * cv2.connectedComponentsWithStats (ml_tools/imageprocessing.py:248) plus the per-region
 * variance ClipTracker._get_regions_of_interest computes (track/cliptracker.py:316-318).
 * Regions are emitted in OpenCV label order (label = index + 1).
 * centroid = (sum_x / area, sum_y / area) in double on the host. */
typedef struct {
    int32_t x, y, width, height; /* cv2 stats: left, top, width, height */
    int32_t area;                /* cv2 stats area == Region.mass */
    int32_t sum_x, sum_y;        /* centroid numerators */
    int32_t key;                 /* first 2x2 block in raster order (label ordering key) */
    double pixel_variance;       /* np.var of the filtered delta frame over the box; 0 on frame 0 */
} cpt_region;

/* Per-frame scalars of ClipTracker._get_filtered_frame (track/cliptracker.py:93-122). */
typedef struct {
    double background_average; /* WeightedBackground.average the frame was filtered against */
    float threshold;      /* mapped_thresh handed to detect_objects (fp32) */
    int32_t norm_min;     /* min / max of G = max(thermal - background - avg_change, 0) */
    int32_t norm_max;
    int32_t avg_change;   /* int(round(mean(thermal) - background average)) */
    int32_t filtered_min; /* min / max of filtered = thermal - background (K1) */
    int32_t filtered_max;
    int32_t n_components; /* true component count (may exceed max_regions / CPT_MAX_COMPONENTS) */
    int32_t thermal_min;  /* ClipStats (only with CPT_CLIP_FRAME_STATS) */
    int32_t thermal_max;
    uint32_t thermal_sum;     /* mean = thermal_sum / (W*H) */
    uint32_t abs_filtered_sum; /* sum |filtered| */
    float thermal_median;
    int32_t reserved[2];
} cpt_frame_info;

/* One clip (or one stream step) of a batch. Frame indices are in units of W*H uint16 frames
 * from the start of d_frames.  ring_frames == 0: the clip is stored linearly; otherwise frame t
 * lives at frame_offset + ((first_frame + t) % ring_frames) (streaming ring buffers). */
typedef struct {
    int64_t frame_offset;      /* first tracked frame */
    int64_t init_offset;       /* frame WeightedBackground is initialised from (cliptrackextractor.py:129-139);
                                  ignored with CPT_CLIP_RESUME */
    int64_t out_offset;        /* index of this clip's first frame in every per-frame output */
    int32_t n_frames;
    int32_t first_frame;       /* absolute number of the first frame of this call (streaming), else 0 */
    int32_t ring_frames;
    int32_t background_thresh; /* clip.background_thresh (config/trackingmotionconfig.py:24-59) */
    int32_t weight_table;      /* slot set with cpt_set_weight_table */
    uint32_t flags;
} cpt_clip;

/* Outputs of an extraction launch; any pointer except d_info may be NULL. */
typedef struct {
    cpt_region *d_regions;   /* [total_frames][max_regions] */
    cpt_frame_info *d_info;  /* [total_frames] */
    float *d_filtered;       /* [total_frames][H][W]  K1: float32(thermal) - background */
    uint8_t *d_labels;       /* [total_frames][H][W]  K5 label image (0 = background) */
    int64_t total_frames;    /* frames the per-frame outputs hold (max over clips of out_offset + n_frames); with
                                d_filtered set it lets a second, wide launch compute the per-region variances.
                                0 = unknown: they are computed inside the extraction kernel */
    int32_t denoise;         /* 1: some clip carries CPT_CLIP_DENOISE -- the normalised images then go through
                                cv2.fastNlMeansDenoising and the mask / component passes after the recurrence
                                (needs total_frames and d_filtered; with CPT_CLIP_RESUME see CPT_CLIP_PREV_IN_OUTPUT) */
    int32_t no_resume;       /* 1: no clip of this launch carries CPT_CLIP_RESUME (d_state, if given, is only written).
                                Lets a launch with a state record take the split plan of DESIGN.md section 3.1; 0 is always safe */
} cpt_outputs;

/* Persistent per-clip state (WeightedBackground + sliding sum), one record per clip:
 * layout returned by cpt_state_bytes(); opaque to the caller except through cpt_state_*. */

const char *cpt_last_error(void);
int cpt_device_count(void);
int cpt_version(void);

/* Context: geometry is fixed per ctx.  width % 8 == 0, width <= 160, width*height <= 19200
 * (Lepton 3/3.5 is 160x120).  edge_pixels as TrackingConfig.edge_pixels (1 for thermal). */
cpt_ctx *cpt_ctx_create(int device, int width, int height, int edge_pixels, int max_regions);
void cpt_ctx_destroy(cpt_ctx *ctx);
int cpt_ctx_set_stream(cpt_ctx *ctx, void *cuda_stream); /* cudaStream_t; NULL = the legacy default stream. A new ctx launches on its own non-blocking stream */
int cpt_ctx_synchronize(cpt_ctx *ctx);

/* WeightedBackground.weight_add (motiondetector.py:182): the fp64 table w_k = fl(w_{k-1} + weight_add)
 * is built on the host and uploaded; max_frames bounds k (<= 65535). */
int cpt_set_weight_table(cpt_ctx *ctx, int slot, double weight_add, int max_frames);
/* Host-only builder of that table (no device needed; exposed for testing): thr_out[k] encodes the integer
 * form of the fp64 keep test `background < frame - w_k` (see csrc/cptrack_kernels.cuh), w_out[k] = w_k. */
int cpt_build_weight_table(double weight_add, int n, uint32_t *thr_out, double *w_out);

/* Device memory helpers so that non-torch hosts can drive the library. */
int cpt_device_alloc(cpt_ctx *ctx, void **d_ptr, uint64_t bytes);
int cpt_device_free(cpt_ctx *ctx, void *d_ptr);
int cpt_host_alloc_pinned(void **h_ptr, uint64_t bytes);
int cpt_host_free_pinned(void *h_ptr);
int cpt_copy_to_device(cpt_ctx *ctx, void *d_dst, const void *h_src, uint64_t bytes);   /* async on ctx stream */
int cpt_copy_to_host(cpt_ctx *ctx, void *h_dst, const void *d_src, uint64_t bytes);     /* async on ctx stream */

/* Diagnostics: per-phase clock64() totals summed over CTAs (all zero unless the library was built with
 * -DCPT_PHASE_TIMING); the first call allocates the counters. h_out32 (32 counters) may be NULL. */
int cpt_debug_phase_cycles(cpt_ctx *ctx, long long *h_out32, int reset);

/* Diagnostics: with enable != 0, every following cpt_extract_batch call brackets its launches with CUDA events on the
 * ctx stream.  h_ms4 (may be NULL) receives the durations of the last timed call in milliseconds after synchronising:
 * [0] the recurrence kernel (strip_sweep_kernel, or extract_clips_kernel on the single-kernel path), [1]
 * frame_scalars_kernel + the per-frame mask / component launches (0 on the single-kernel path), [2] the denoise passes,
 * [3] region_variance_kernel. */
int cpt_debug_kernel_times(cpt_ctx *ctx, int enable, float *h_ms4);
/* Same, finer: h_ms[0..n-1], n <= 5: [0] strip_sweep_kernel (the recurrence; extract_clips_kernel on the single-kernel path),
 * [1] frame_scalars_kernel, [2] the per-frame mask / component launches, [3] the denoise passes, [4] region_variance_kernel. */
int cpt_debug_kernel_times_ex(cpt_ctx *ctx, int enable, float *h_ms, int n);

/* Diagnostics / tests: with enable != 0 every extraction launch of this ctx runs the single persistent kernel, also where
 * the split plan would apply (both plans produce identical results). */
int cpt_debug_force_single_kernel(cpt_ctx *ctx, int enable);

/* Bytes of one per-clip state record for this ctx's geometry. */
uint64_t cpt_state_bytes(const cpt_ctx *ctx);

/* ClipTrackExtractor.parse_clip / process_frame for a batch of clips
 * (track/cliptrackextractor.py:141-247; K1,K2,K4,K5,K6,K7,K8 of SURVEY.md section 8a).
 * One persistent CTA per clip.  d_clips is a DEVICE array of n_clips cpt_clip records,
 * d_state (optional unless a clip has CPT_CLIP_RESUME, then required) receives each clip's
 * final state: n_clips * cpt_state_bytes(). */
int cpt_extract_batch(cpt_ctx *ctx, const uint16_t *d_frames, const cpt_clip *d_clips, int n_clips,
                      const cpt_outputs *outputs, void *d_state);

/* Same call with HOST buffers: stages frames to the device in chunks of clips on two streams
 * (copy / compute overlapped) and copies regions + info (and filtered / labels when
 * requested) back.  h_frames should be pinned (cpt_host_alloc_pinned) for full PCIe speed.  CPT_CLIP_DENOISE clips are
 * allowed (the denoise passes run per chunk); CPT_CLIP_RESUME is not. */
int cpt_extract_batch_host(cpt_ctx *ctx, const uint16_t *h_frames, const cpt_clip *h_clips, int n_clips,
                           int64_t total_frames, cpt_region *h_regions, cpt_frame_info *h_info,
                           float *h_filtered, uint8_t *h_labels, int chunk_clips);

/* WeightedBackground.process_frame(frame) (piclassifier/motiondetector.py:197-244) on n_records state
 * records: record d_record_index[i] (or i when NULL) is updated with int32 frame i of d_frames
 * ([n_records][H][W], already truncated like np.int32(frame)).  A record whose `initialised` flag is 0
 * (fresh, zero-filled memory) takes the first-call path: background = frame, average = mean (unrounded). */
int cpt_background_process(cpt_ctx *ctx, void *d_state, const int32_t *d_record_index, int n_records,
                           const int32_t *d_frames, int weight_slot);

/* np.median of each uint16 frame (ClipStats.add_frame, track/clip.py:474-487; the per-frame median of
 * Interpreter.preprocess_segments, ml_tools/interpreter.py:389).  d_medians float32 [n_frames]. */
int cpt_frame_medians(cpt_ctx *ctx, const uint16_t *d_frames, int64_t n_frames, float *d_medians);

/* ---- classifier-input preprocessing: Interpreter.preprocess_segments (ml_tools/interpreter.py:365-474) ----
 * One cpt_sample per unique (track, frame) region, one cpt_track_norm per track.  Frames are addressed by
 * their index in the uint16 thermal buffer and the float32 filtered buffer of an extraction
 * (cpt_outputs.d_filtered), both [n_frames][H][W]. */
typedef struct {
    int64_t frame;               /* frame index into d_thermal / d_filtered */
    int32_t x, y, width, height; /* Region bounds (track/region.py), inside the frame, width/height >= 1 */
    int32_t track;               /* row of the cpt_track_norm table */
    float median;                /* np.median(frame.thermal) (interpreter.py:389), written by cpt_preprocess_medians */
} cpt_sample;

typedef struct {
    float filtered_min, filtered_max; /* Interpreter.get_limits with diff_norm (interpreter.py:315-363) */
    int32_t clip_at_zero;             /* clip_thermals_at_zero (interpreter.py:391-399) */
    int32_t has_limits;               /* 0: the track had no usable region, normalise by the tile's own minimum */
    float thermal_min, thermal_max;   /* get_limits with thermal_diff_norm: extrema of frame.thermal - median over the track's frames */
    int32_t has_thermal_limits;       /* 0: thermal_diff_norm off; 1: limits above; 2: on, but the track had no usable region
                                         (per-tile extrema).  With 1 or 2 the thermal channel is not clipped at zero
                                         (preprocess.py:92-93) */
    int32_t reserved;
} cpt_track_norm;

/* get_limits: resets all n_tracks rows (min unset, max 0, clip_at_zero 1), then folds the min / max of
 * region.subimage(frame.filtered) of every entry of d_regions (all non-blank regions of each track). */
int cpt_preprocess_limits(cpt_ctx *ctx, const float *d_filtered, const cpt_sample *d_regions, int n_regions,
                          cpt_track_norm *d_tracks, int n_tracks);
/* get_limits with HyperParams.thermal_diff_norm (interpreter.py:338-345,358-359): after cpt_preprocess_limits, folds the
 * min / max of frame.thermal - np.median(frame.thermal) over the WHOLE frame of every entry of d_regions into the
 * track rows (one full-frame median per entry). */
int cpt_preprocess_thermal_limits(cpt_ctx *ctx, const uint16_t *d_thermal, const cpt_sample *d_regions, int n_regions,
                                  cpt_track_norm *d_tracks, int n_tracks);
/* Pass 1 of preprocess_segments over the unique track-frames: fills sample.median and clears the track's
 * clip_at_zero when np.median(region.subimage(thermal) - median) <= 0. */
int cpt_preprocess_medians(cpt_ctx *ctx, const uint16_t *d_thermal, cpt_sample *d_samples, int n_samples,
                           cpt_track_norm *d_tracks);
/* Pass 2 + preprocess_movement (ml_tools/preprocess.py:56-113,151-202; imageprocessing.py:11-104): every
 * segment is tiles_per_segment sample indices (d_segment_samples [n_segments][tiles_per_segment], already padded
 * and sorted as preprocess_movement does); tile i lands in row i / frames_per_row, column i % frames_per_row of
 * d_out [n_segments][rows*frame_size][frames_per_row*frame_size][2] float32 (channels thermal, filtered).
 * crop_rectangle = {x, y, width, height} of Clip.crop_rectangle (keep_edge anchoring) or NULL;
 * preprocess_fn: CPT_PREPROCESS_INC3 = x / 127.5 - 1 (interpreter.py:563-566); CPT_PREPROCESS_PER_TILE = HyperParams.diff_norm
 * off: no track-wide limits, both channels are normalised by the tile's own extrema (Frame.normalize, preprocess.py:111). */
#define CPT_PREPROCESS_INC3 1
#define CPT_PREPROCESS_PER_TILE 2
int cpt_preprocess_segments(cpt_ctx *ctx, const uint16_t *d_thermal, const float *d_filtered, const cpt_sample *d_samples,
                            const cpt_track_norm *d_tracks, const int32_t *d_segment_samples, int n_segments,
                            int tiles_per_segment, int frames_per_row, int frame_size, const int32_t *crop_rectangle,
                            int preprocess_fn, float *d_out);

/* The same passes on an extraction's own buffers (ClipTrackExtractor.parse_clips(keep_on_device=True)).  There a tracked frame
 * lives at different rows: its thermal row (sample.frame; the row of d_frames it was read from, also its row of
 * cpt_frame_medians) and its filtered row (out_offset + n, its row of d_filtered and of every other per-frame output).
 *   d_filtered_rows    one int64 per entry of d_regions / d_samples: the entry's filtered row (NULL: the same as sample.frame)
 *   d_frame_medians    float32 per thermal row as cpt_frame_medians writes them (NULL: recompute them from the frames).  Given,
 *                      the medians pass looks sample.median up and reads only the crop for the clip_thermals_at_zero test
 *   d_frame_info       the extraction's cpt_frame_info per filtered row, computed with CPT_CLIP_FRAME_STATS.  With
 *                      d_frame_medians as well, the thermal_diff_norm limits are (thermal_min - median, thermal_max - median)
 *                      folded per track without reading a frame; otherwise the frames are read as cpt_preprocess_thermal_limits does
 * Results are bit-identical to the entry points above on the same frames. */
int cpt_preprocess_limits_ex(cpt_ctx *ctx, const float *d_filtered, const int64_t *d_filtered_rows, const cpt_sample *d_regions,
                             int n_regions, cpt_track_norm *d_tracks, int n_tracks);
int cpt_preprocess_thermal_limits_ex(cpt_ctx *ctx, const uint16_t *d_thermal, const int64_t *d_filtered_rows, const cpt_sample *d_regions,
                                     int n_regions, cpt_track_norm *d_tracks, int n_tracks, const float *d_frame_medians,
                                     const cpt_frame_info *d_frame_info);
int cpt_preprocess_medians_ex(cpt_ctx *ctx, const uint16_t *d_thermal, const float *d_frame_medians, cpt_sample *d_samples, int n_samples,
                              cpt_track_norm *d_tracks);
int cpt_preprocess_segments_ex(cpt_ctx *ctx, const uint16_t *d_thermal, const float *d_filtered, const int64_t *d_filtered_rows,
                               const cpt_sample *d_samples, const cpt_track_norm *d_tracks, const int32_t *d_segment_samples,
                               int n_segments, int tiles_per_segment, int frames_per_row, int frame_size,
                               const int32_t *crop_rectangle, int preprocess_fn, float *d_out);

/* ---- ml_tools/imageprocessing.py helpers on single images (device buffers) ----
 * normalize() (imageprocessing.py:151-169): cpt_minmax_f32 writes {min, max} of d_in to d_out2; cpt_normalize_f32
 * computes new_max * (float32(data) - min) / (max - min) (max == min: zeros if max == 0, else data / max) in fp32
 * (d_out float32) or, with use_f64, in fp64 on the fp32-rounded data (d_out float64) -- numpy picks one or the
 * other from the operand types; the host mirror makes that choice. */
int cpt_minmax_f32(cpt_ctx *ctx, const float *d_in, int64_t n, float *d_out2);
int cpt_normalize_f32(cpt_ctx *ctx, const float *d_in, int64_t n, double min, double max, double new_max, int use_f64,
                      void *d_out);
/* resize_and_pad() / resize_cv() (imageprocessing.py:11-82): cv2.resize of the src_w x src_h float32 image to
 * resized_w x resized_h (interpolation 1 = INTER_LINEAR, 0 = INTER_NEAREST), pasted at (offset_x, offset_y) into an
 * out_w x out_h image filled with pad. */
int cpt_resize_pad_f32(cpt_ctx *ctx, const float *d_src, int src_w, int src_h, int resized_w, int resized_h, int offset_x,
                       int offset_y, int out_w, int out_h, float pad, int interpolation, float *d_out);

/* detect_objects() (imageprocessing.py:240-248) on one uint8 image of any size: GaussianBlur (blur_ksize 5, or 0
 * for none) -> threshold (src > floor(threshold)) -> morphologyEx CLOSE with a tuple kernel (close != 0; OpenCV turns
 * the tuple into a 2x1 element) -> connectedComponentsWithStats (8-connectivity, OpenCV label numbering).
 * d_labels int32 [H][W]; d_stats int32 [max_components + 1][5] = left, top, width, height, area; d_centroids double
 * [max_components + 1][2]; row 0 is the background.  *h_count = number of labels including the background.
 * Synchronises the ctx stream. */
int cpt_detect_objects_u8(cpt_ctx *ctx, const uint8_t *d_image, int width, int height, double threshold, int blur_ksize,
                          int close, int max_components, int32_t *d_labels, int32_t *d_stats, double *d_centroids,
                          int32_t *h_count);

/* The same pipeline with every stage the imageprocessing.py variants use, on one uint8 image of any size:
 *   detect_objects(kernel=(15,15) default, otsus)   imageprocessing.py:240-248  blur_ksize 3 / 5 / 7 / 15 (cv2.GaussianBlur 8-bit
 *                                                   fixed-point taps), CPT_DETECT_OTSU (cv2.threshold THRESH_OTSU), CPT_DETECT_CLOSE
 *   detect_objects_ir (IR 640x480 frames)           imageprocessing.py:185-199  CPT_DETECT_OPEN_GRAY (cv2.morphologyEx MORPH_OPEN
 *                                                   with a tuple kernel = 2x1 element, on the grey image), threshold, components
 *   detect_objects_both                             imageprocessing.py:202-238  blur, threshold, CPT_DETECT_DILATE, CPT_DETECT_CLOSE,
 *                                                   d_or_mask (the thresholded saliency map, any non-zero = set) OR-ed in
 * CPT_DETECT_MASK_ONLY stops after the binary stages and writes the mask (0 / 255) to d_mask_out.  h_threshold_used (may
 * be NULL) receives the threshold applied (Otsu's when CPT_DETECT_OTSU).  Synchronises the ctx stream. */
#define CPT_DETECT_CLOSE 1u
#define CPT_DETECT_OPEN_GRAY 2u
#define CPT_DETECT_DILATE 4u
#define CPT_DETECT_OTSU 8u
#define CPT_DETECT_MASK_ONLY 16u
int cpt_detect_objects_ex(cpt_ctx *ctx, const uint8_t *d_image, int width, int height, double threshold, int blur_ksize,
                          uint32_t steps, const uint8_t *d_or_mask, int max_components, int32_t *d_labels, int32_t *d_stats,
                          double *d_centroids, uint8_t *d_mask_out, int32_t *h_count, double *h_threshold_used);

/* cv2.fastNlMeansDenoising(uint8, None) (track/cliptracker.py:116-117; h = 3, 7x7 template, 21x21 search), OpenCV's
 * integer algorithm bit for bit, on n_frames images [n_frames][H][W].  The batched extractor runs the same kernel for clips
 * with CPT_CLIP_DENOISE. */
int cpt_nlm_denoise_u8(cpt_ctx *ctx, const uint8_t *d_src, int width, int height, int n_frames, uint8_t *d_dst);

/* ---- CPTV v2 frame decode (what cptv_rs_python_bindings.CptvReader.next_frame does per pixel;
 * track/cliptrackextractor.py:108-129,160-165).  The host inflates the gzip stream and walks the section headers;
 * d_stream is the inflated byte stream, one cpt_cptv_frame per frame section (in file order, clips back to back),
 * d_clip_first [n_clips + 1] the first frame index of every clip.  d_frames [n_frames][H][W] uint16. */
typedef struct {
    uint64_t payload_offset; /* byte offset of the frame payload (int32 start value, then packed deltas) */
    int32_t bit_width;       /* field 'w': bits per packed delta (1..24), MSB first, two's complement */
    int32_t reserved;
} cpt_cptv_frame;
int cpt_cptv_decode(cpt_ctx *ctx, const uint8_t *d_stream, const cpt_cptv_frame *d_table, int n_frames,
                    const int32_t *d_clip_first, int n_clips, uint16_t *d_frames);

/* cpt_extract_batch_host for clips that are still PACKED (what ClipTrackExtractor.parse_clip reads through
 * CptvReader.next_frame, track/cliptrackextractor.py:108-129,160-165): h_stream holds the inflated frame payloads, h_table
 * one row per frame of every clip (clip i = rows h_clip_first[i] .. h_clip_first[i + 1] - 1, in file order), and the
 * cpt_clip records address frames in that row space (frame_offset / init_offset = table rows; a leading background frame
 * is simply a row the clip's frame_offset skips).  The payloads (about one byte per pixel) are staged to the device in
 * chunks of clips, decoded there and extracted; regions + info come back as in cpt_extract_batch_host.  Every payload is
 * checked to lie inside the stream before anything is launched. */
int cpt_extract_batch_cptv_host(cpt_ctx *ctx, const uint8_t *h_stream, uint64_t stream_bytes, const cpt_cptv_frame *h_table,
                                const int64_t *h_clip_first, const cpt_clip *h_clips, int n_clips, int64_t total_frames,
                                cpt_region *h_regions, cpt_frame_info *h_info, int chunk_clips);

/* ---- CPTVMotionDetector (piclassifier/cptvmotiondetector.py:14-205), streaming, one launch per frame ----
 * The detector owns a ring of the last ring_frames frames (SlidingWindow of preview_secs * fps + 1 frames), the
 * uint32 running sum (RunningMean over mean_frames = 45) and, for one_diff_only == False, a ring of diff_frames
 * clamped delta frames.  Ring bookkeeping (which slot is newest / oldest / oldest non-FFC) stays on the host. */
typedef struct cpt_motion cpt_motion;
#define CPT_MOTION_MEAN 1u          /* RunningMean.add(new, oldest) (motiondetector.py:166-172) */
#define CPT_MOTION_MEAN_RESTART 2u  /* start the running sum from this frame alone */
#define CPT_MOTION_BACKGROUND 4u    /* WeightedBackground.process_frame(running_mean.mean()) (cptvmotiondetector.py:152-153) */
#define CPT_MOTION_DETECT 8u        /* detect() (cptvmotiondetector.py:74-120) */
#define CPT_MOTION_WARMER_ONLY 16u  /* config.warmer_only */
#define CPT_MOTION_ONE_DIFF 32u     /* config.one_diff_only */
typedef struct {
    double average;      /* WeightedBackground.average after this frame == temp_thresh */
    int32_t diff;        /* pixels over the delta threshold (compare with count_thresh on the host) */
    int32_t error;       /* 1: running mean left the uint16 range */
    int32_t mean_frames; /* RunningMean.running_mean_frames */
    int32_t reserved;
} cpt_motion_result;
cpt_motion *cpt_motion_open(cpt_ctx *ctx, int ring_frames, int mean_frames, int diff_frames, int weight_slot);
void cpt_motion_close(cpt_motion *m);
/* SlidingWindow.update_current_frame / add without processing: host frame -> ring slot. */
int cpt_motion_store(cpt_motion *m, const uint16_t *h_pix, int slot);
/* RunningMean(frames, window) from the listed ring slots (first processed frame after frames were only stored). */
int cpt_motion_mean_init(cpt_motion *m, const int32_t *h_slots, int n);
/* One process_frame: copies h_pix into ring slot slot_new, runs the fused step on the ctx stream, waits and
 * returns the result.  d_background_state is the WeightedBackground state record (cpt_state_bytes) the detector
 * shares with the streaming extractor; slot_oldest = SlidingWindow.oldest (-1: none); slot_nonffc / diff_slot_old =
 * the oldest non-FFC entries of the two rings (diff_slot_old -1: fewer than 3 frames processed). */
int cpt_motion_step(cpt_motion *m, const uint16_t *h_pix, void *d_background_state, int slot_new, int slot_oldest,
                    int slot_nonffc, int diff_slot_new, int diff_slot_old, uint32_t flags, int delta_thresh,
                    double init_average, cpt_motion_result *h_result);

/* ---- IRMotionDetector (piclassifier/irmotiondetector.py:55-153), streaming, 640x480 BGR frames ----
 * Per frame the reference does cv2.cvtColor(BGR2GRAY), feeds the grey frame to its background model (OpenCV's MOG2: third
 * party, stays on the host), then absdiff(oldest grey, grey) -> threshold 12 -> erode with a k x k box (15 idle / 10 while
 * recording) -> count, and the same erode + count on the background model's foreground mask.  The detector owns a ring of
 * grey frames on the device (SlidingWindow of preview_secs * fps frames).
 *   cpt_ir_motion_gray    h_bgr [H][W][3] -> grey (OpenCV's fixed point: (B*3735 + G*19235 + R*9798 + 2^14) >> 15) into ring
 *                         slot slot_new; h_gray_out (may be NULL) receives it for the host's background model
 *   cpt_ir_motion_detect  *h_diff_pixels = count(erode(|ring[slot_oldest] - ring[slot_new]| > threshold)); with h_mask (the
 *                         background model's foreground mask, [H][W], non-zero = set; may be NULL) *h_mask_pixels =
 *                         count(erode(h_mask)).  Pixels outside the image do not constrain the erosion (cv2's default). */
typedef struct cpt_ir_motion cpt_ir_motion;
cpt_ir_motion *cpt_ir_motion_open(cpt_ctx *ctx, int width, int height, int ring_frames);
void cpt_ir_motion_close(cpt_ir_motion *m);
int cpt_ir_motion_gray(cpt_ir_motion *m, const uint8_t *h_bgr, int slot_new, uint8_t *h_gray_out);
int cpt_ir_motion_detect(cpt_ir_motion *m, int slot_new, int slot_oldest, int threshold, int erode_k, const uint8_t *h_mask,
                         int32_t *h_diff_pixels, int32_t *h_mask_pixels);

/* State access for WeightedBackground.background / .background_weight / .average
 * (motiondetector.py:178-248).  h_background int32 [H][W]; h_weight_count uint16 [(H-2e)][(W-2e)]
 * (background_weight = table[count]); h_average double. Any output may be NULL. */
int cpt_state_read(cpt_ctx *ctx, const void *d_state, int clip_index, int32_t *h_background,
                   uint16_t *h_weight_count, double *h_average, uint32_t *h_sliding_sum,
                   int32_t *h_frames_seen);
int cpt_state_write(cpt_ctx *ctx, void *d_state, int clip_index, const int32_t *h_background,
                    const uint16_t *h_weight_count, double average);
/* the fp64 weight for a count (host copy of the uploaded table) */
double cpt_weight_value(const cpt_ctx *ctx, int slot, int count);

#ifdef __cplusplus
}
#endif
#endif /* CPTRACK_H */
