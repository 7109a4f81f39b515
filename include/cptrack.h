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
 * ctx stream.  h_ms (may be NULL) receives the durations of the last timed call in milliseconds after synchronising,
 * h_ms[0..n-1], n <= 5: [0] strip_sweep_kernel (the recurrence; extract_clips_kernel on the single-kernel path),
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

/* On an extraction's own buffers (ClipTrackExtractor.parse_clips(keep_on_device=True)) a tracked frame lives at two rows:
 * its thermal row (sample.frame: the row of d_frames it was read from, also its row of cpt_frame_medians) and its filtered
 * row (out_offset + n: its row of d_filtered and of every other per-frame output).  d_filtered_rows holds one int64 filtered
 * row per entry of d_regions / d_samples, d_frame_medians and d_frame_info the extraction's per-frame statistics.  Each
 * may be NULL, as each entry point below says, and every choice gives bit-identical results on the same frames. */

/* get_limits: resets all n_tracks rows (min unset, max 0, clip_at_zero 1), then folds the min / max of
 * region.subimage(frame.filtered) of every entry of d_regions (all non-blank regions of each track), read at the entry's
 * filtered row (d_filtered_rows, or NULL: sample.frame). */
int cpt_preprocess_limits(cpt_ctx *ctx, const float *d_filtered, const int64_t *d_filtered_rows, const cpt_sample *d_regions,
                          int n_regions, cpt_track_norm *d_tracks, int n_tracks);
/* get_limits with HyperParams.thermal_diff_norm (interpreter.py:338-345,358-359): after cpt_preprocess_limits, folds the
 * min / max of frame.thermal - np.median(frame.thermal) over the WHOLE frame of every entry of d_regions into the
 * track rows.  With d_frame_medians (float32 per thermal row, as cpt_frame_medians writes them) and d_frame_info (the
 * extraction's cpt_frame_info per filtered row, computed with CPT_CLIP_FRAME_STATS; d_filtered_rows, or NULL: sample.frame)
 * both given, the limits are (thermal_min - median, thermal_max - median) and no frame is read; with either NULL each
 * entry's thermal frame is read and its full-frame median computed (d_filtered_rows is then unused). */
int cpt_preprocess_thermal_limits(cpt_ctx *ctx, const uint16_t *d_thermal, const int64_t *d_filtered_rows, const cpt_sample *d_regions,
                                  int n_regions, cpt_track_norm *d_tracks, int n_tracks, const float *d_frame_medians,
                                  const cpt_frame_info *d_frame_info);
/* Pass 1 of preprocess_segments over the unique track-frames: fills sample.median and clears the track's
 * clip_at_zero when np.median(region.subimage(thermal) - median) <= 0.  d_frame_medians (float32 per thermal row, as
 * cpt_frame_medians writes them): sample.median is looked up and only the crop is read; NULL: each sample's thermal frame
 * is read and its median computed. */
int cpt_preprocess_medians(cpt_ctx *ctx, const uint16_t *d_thermal, const float *d_frame_medians, cpt_sample *d_samples, int n_samples,
                           cpt_track_norm *d_tracks);
/* Pass 2 + preprocess_movement (ml_tools/preprocess.py:56-113,151-202; imageprocessing.py:11-104): every
 * segment is tiles_per_segment sample indices (d_segment_samples [n_segments][tiles_per_segment], already padded
 * and sorted as preprocess_movement does); tile i lands in row i / frames_per_row, column i % frames_per_row of
 * d_out [n_segments][rows*frame_size][frames_per_row*frame_size][2] float32 (channels thermal, filtered).  The thermal
 * crop is read at sample.frame, the filtered crop at the sample's filtered row (d_filtered_rows, or NULL: sample.frame).
 * crop_rectangle = {x, y, width, height} of Clip.crop_rectangle (keep_edge anchoring) or NULL;
 * preprocess_fn: CPT_PREPROCESS_INC3 = x / 127.5 - 1 (interpreter.py:563-566); CPT_PREPROCESS_PER_TILE = HyperParams.diff_norm
 * off: no track-wide limits, both channels are normalised by the tile's own extrema (Frame.normalize, preprocess.py:111). */
#define CPT_PREPROCESS_INC3 1
#define CPT_PREPROCESS_PER_TILE 2
int cpt_preprocess_segments(cpt_ctx *ctx, const uint16_t *d_thermal, const float *d_filtered, const int64_t *d_filtered_rows,
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

/* detect_objects() (imageprocessing.py:240-248) and its variants on one uint8 image of any size: the grey stages, a
 * threshold (src > floor(threshold)), the binary stages, then connectedComponentsWithStats (8-connectivity, OpenCV label
 * numbering).  steps selects the stages each variant uses:
 *   detect_objects(kernel=(15,15) default, otsus)   imageprocessing.py:240-248  blur_ksize 3 / 5 / 7 / 15 (cv2.GaussianBlur 8-bit
 *                                                   fixed-point taps, 0 for none), CPT_DETECT_OTSU (cv2.threshold THRESH_OTSU),
 *                                                   CPT_DETECT_CLOSE (morphologyEx CLOSE with a tuple kernel: OpenCV turns the
 *                                                   tuple into a 2x1 element)
 *   detect_objects_ir (IR 640x480 frames)           imageprocessing.py:185-199  CPT_DETECT_OPEN_GRAY (cv2.morphologyEx MORPH_OPEN
 *                                                   with a tuple kernel = 2x1 element, on the grey image), threshold, components
 *   detect_objects_both                             imageprocessing.py:202-238  blur, threshold, CPT_DETECT_DILATE, CPT_DETECT_CLOSE,
 *                                                   d_or_mask (the thresholded saliency map, any non-zero = set) OR-ed in
 * d_labels int32 [H][W]; d_stats int32 [max_components + 1][5] = left, top, width, height, area; d_centroids double
 * [max_components + 1][2]; row 0 is the background.  *h_count = number of labels including the background.
 * CPT_DETECT_MASK_ONLY stops after the binary stages and writes the mask (0 / 255) to d_mask_out.  h_threshold_used (may
 * be NULL) receives the threshold applied (Otsu's when CPT_DETECT_OTSU).  For an image that is all foreground, the
 * background row is cv2's [-1, INT_MAX, 0, 0, 0] with a NaN centroid.  Synchronises the ctx stream. */
#define CPT_DETECT_CLOSE 1u
#define CPT_DETECT_OPEN_GRAY 2u
#define CPT_DETECT_DILATE 4u
#define CPT_DETECT_OTSU 8u
#define CPT_DETECT_MASK_ONLY 16u
int cpt_detect_objects(cpt_ctx *ctx, const uint8_t *d_image, int width, int height, double threshold, int blur_ksize,
                       uint32_t steps, const uint8_t *d_or_mask, int max_components, int32_t *d_labels, int32_t *d_stats,
                       double *d_centroids, uint8_t *d_mask_out, int32_t *h_count, double *h_threshold_used);

/* detect_objects_ir (imageprocessing.py:185-199) on n_frames uint8 frames [n_frames][H][W] of one geometry in one call, with
 * no host synchronisation: steps CPT_DETECT_OPEN_GRAY (or 0) -> threshold -> connectedComponentsWithStats per frame.
 *   d_counts     [n_frames]: cv2's label count of each frame (background included)
 *   d_stats      [n_frames][max_components + 1][5], row 0 = background; rows beyond the frame's count are not written
 *   d_centroids  [n_frames][max_components + 1][2] double, or NULL
 *   d_labels     [n_frames][H][W] int32, or NULL
 * A frame with more than max_components components reports its true count and keeps its first max_components rows in
 * label order (its label image stays complete); the call does not fail.  Other steps return CPT_ERR_UNSUPPORTED.
 * Launches go on the ctx stream. */
int cpt_detect_objects_batch(cpt_ctx *ctx, const uint8_t *d_frames, int n_frames, int width, int height, double threshold,
                             uint32_t steps, int max_components, int32_t *d_counts, int32_t *d_stats, double *d_centroids,
                             int32_t *d_labels);

/* IRTrackExtractor's rectangle merging (track/irtrackextractor.py:324-389, merge_components) for every frame of a
 * cpt_detect_objects_batch result (d_stats, d_counts, the same max_components): keep rows with area > min_mass or with
 * width and height > min_size, sort by area (descending, stable), merge pairs that overlap or lie closer than max_gap.
 * The caller derives min_mass = int(40 * scale), min_size = int(16 * scale), max_gap = 40 * scale (40, 16, 40 without a
 * scale).  d_merged [n_frames][max_components][5] (x, y, w, h, area), d_merged_counts [n_frames]: rectangles per frame,
 * -1 for a frame whose components overflowed max_components.  Launches go on the ctx stream. */
int cpt_ir_merge_components(cpt_ctx *ctx, const int32_t *d_stats, const int32_t *d_counts, int n_frames, int max_components,
                            int min_mass, int min_size, double max_gap, int32_t *d_merged, int32_t *d_merged_counts);

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

/* ---- CPTVMotionDetector (piclassifier/cptvmotiondetector.py:14-205) on the device ----
 * The detector owns a ring of the last ring_frames frames (SlidingWindow of preview_secs * fps + 1 frames), the
 * uint32 running sum (RunningMean over mean_frames = 45) and, for one_diff_only == False, a ring of diff_frames
 * clamped delta frames.  Ring bookkeeping (which slot is newest / oldest / oldest non-FFC) stays on the host, which
 * plans every frame as one cpt_motion_clip_step; cpt_motion_step runs one step and cpt_motion_clips many, with the same
 * device code and the same checks. */
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
/* One planned frame (cptvmotiondetector.py:135-205).  A frame reference r >= 0 is row r of cpt_motion_clips' d_frames;
 * r < 0 is slot -1 - r of the detector's ring as it stood before the call. */
typedef struct {
    int32_t frame;          /* the new frame (SlidingWindow.current after add) */
    int32_t oldest;         /* SlidingWindow.oldest after the add */
    int32_t nonffc;         /* SlidingWindow.oldest_nonffc; read with CPT_MOTION_DETECT only */
    int32_t diff_slot_new;  /* delta ring slots (CPT_MOTION_DETECT without CPT_MOTION_ONE_DIFF): the new delta frame and the */
    int32_t diff_slot_old;  /*   oldest non-FFC one (-1: fewer than 3 frames processed) */
    int32_t mean_first;     /* mean_count > 0: RunningMean(frames) from h_mean_rows[mean_first .. mean_first + mean_count) */
    int32_t mean_count;     /*   before this step (at most the detector's mean_frames): the first processed frame after frames
                               were only stored */
    uint32_t flags;         /* CPT_MOTION_* */
} cpt_motion_clip_step;
typedef struct {
    cpt_motion *m;
    void *d_background_state;  /* the WeightedBackground state record (cpt_state_bytes) the detector shares with the
                                  streaming extractor */
    const int32_t *ring_rows;  /* cpt_motion_clips: host [ring_frames], row of d_frames each ring slot holds afterwards,
                                  -1 = unchanged; NULL = none */
    double init_average;       /* WeightedBackground(init_average=...) until the background has seen a frame */
    int32_t delta_thresh;
    int32_t first_step;        /* cpt_motion_clips: this detector's steps are h_steps[first_step .. first_step + n_steps) */
    int32_t n_steps;
    int32_t reserved;
} cpt_motion_clip;
cpt_motion *cpt_motion_open(cpt_ctx *ctx, int ring_frames, int mean_frames, int diff_frames, int weight_slot);
void cpt_motion_close(cpt_motion *m);
/* SlidingWindow.update_current_frame / add without processing: host frame -> ring slot. */
int cpt_motion_store(cpt_motion *m, const uint16_t *h_pix, int slot);
/* One process_frame of detector h_clip->m (ring_rows, first_step and n_steps are not read): h_pix is stored in ring slot
 * -1 - h_step->frame, then the step runs on the ctx stream with every frame reference a ring slot and its mean rows in
 * h_mean_rows[0 .. n_mean_rows), n_mean_rows <= 64.  Waits and returns the result; CPT_ERR_INVALID for a reference, slot or
 * row out of range (checked before anything changes) and for a step whose running mean left the uint16 range. */
int cpt_motion_step(const cpt_motion_clip *h_clip, const uint16_t *h_pix, const cpt_motion_clip_step *h_step,
                    const int32_t *h_mean_rows, int n_mean_rows, cpt_motion_result *h_result);

/* Whole recordings, many detectors, one launch (cptvmotiondetector.py:135-205, motiondetector.py:160-244 for every frame
 * of each detector's frame list): one CTA per detector runs that detector's steps in order.  d_frames is
 * [n_frames][H][W] uint16 in device memory.  After the steps, each ring slot with ring_rows[slot] >= 0 takes that row, so
 * the ring holds what the per-frame calls would have left; the running sum, the delta ring and the background state
 * record are updated in place as by those calls.  Every detector must belong to ctx and appear once, with its own state
 * record.  Every index (frame references, delta-ring slots, mean rows, ring_rows, step ranges) is checked before anything
 * is launched: CPT_ERR_INVALID.  h_results[i] is step i's result as cpt_motion_step returns it; a step whose running mean
 * left the uint16 range has error = 1 (the call itself returns CPT_OK). */
int cpt_motion_clips(cpt_ctx *ctx, const cpt_motion_clip *h_clips, int n, const uint16_t *d_frames, int64_t n_frames,
                     const cpt_motion_clip_step *h_steps, int n_steps, const int32_t *h_mean_rows, int n_mean_rows,
                     cpt_motion_result *h_results);

/* ---- IRMotionDetector (piclassifier/irmotiondetector.py:55-153), streaming, 640x480 BGR frames ----
 * Per frame the reference does cv2.cvtColor(BGR2GRAY), feeds the grey frame to its background model (OpenCV's MOG2, on the
 * host through cv2 or on the device through cpt_mog2 below), then absdiff(oldest grey, grey) -> threshold 12 -> erode with a
 * k x k box (15 idle / 10 while recording) -> count, and the same erode + count on the background model's foreground mask.
 * The detector owns a ring of grey frames on the device (SlidingWindow of preview_secs * fps frames).  With a host
 * background model each frame is cpt_ir_motion_gray, the model, then cpt_ir_motion_detect; with the device MOG2 it is one
 * cpt_ir_motion_step (below).
 *   cpt_ir_motion_gray       h_bgr [H][W][3] -> grey (OpenCV's fixed point: (B*3735 + G*19235 + R*9798 + 2^14) >> 15) into
 *                            ring slot slot_new; h_gray_out (may be NULL) receives it for a host background model
 *   cpt_ir_motion_detect     *h_diff_pixels = count(erode(|ring[slot_oldest] - ring[slot_new]| > threshold)); with h_mask (the
 *                            background model's foreground mask, [H][W], non-zero = set; may be NULL) *h_mask_pixels =
 *                            count(erode(h_mask)).  Pixels outside the image do not constrain the erosion (cv2's default). */
typedef struct cpt_ir_motion cpt_ir_motion;
cpt_ir_motion *cpt_ir_motion_open(cpt_ctx *ctx, int width, int height, int ring_frames);
void cpt_ir_motion_close(cpt_ir_motion *m);
int cpt_ir_motion_gray(cpt_ir_motion *m, const uint8_t *h_bgr, int slot_new, uint8_t *h_gray_out);
int cpt_ir_motion_detect(cpt_ir_motion *m, int slot_new, int slot_oldest, int threshold, int erode_k, const uint8_t *h_mask,
                         int32_t *h_diff_pixels, int32_t *h_mask_pixels);

/* Whole IR recordings, many detectors, with each frame's trigger decided on the device (irmotiondetector.py:103-153 for
 * every frame of each detector's frame list, with the device MOG2 of cpt_mog2 as background model).  The host plans the
 * ring cursors and which frames detect; the device runs, for every step: grey into ring slot slot_new, the MOG2 update of
 * the clip's model with learning rate 0 while the clip's movement flag is set and cv2's automatic rate otherwise, the
 * foreground mask into the clip's d_mask, and with detect the two eroded counts (box erode_recording while recording,
 * erode_idle otherwise) and the trigger rule: the mask count is min(diff, mask) while recording, triggered moves by one
 * within [0, max_triggered], movement starts at triggered >= trigger_frames and ends at triggered <= 0.  Steps of one clip
 * run in order; the movement flag each step reads is the one the clip's previous step left, with no host round trip.
 * h_frames holds n_frames addresses of [H][W][3] uint8 BGR frames: device memory, or host memory with host_frames = 1
 * (copied with cudaMemcpyAsync, in chunks of about 256 MB of the context's scratch).  Each clip's model advances its frame
 * count as cpt_mog2_apply with learning rates -1 / 0 would.  Every handle (on ctx, one geometry, each ir / MOG2 handle and
 * mask once), frame row, ring slot, step range and erosion size is checked before anything is launched or changed:
 * CPT_ERR_INVALID.  The call synchronises once, at the end; movement / triggered of each clip record then hold the
 * clip's state after its last step. */
typedef struct {
    int64_t row;          /* the step's BGR frame: h_frames[row] */
    int32_t slot_new;     /* ring slot the grey frame goes to (SlidingWindow.last_index after add) */
    int32_t slot_oldest;  /* the ring slot it is compared with (SlidingWindow.oldest_index; == slot_new in a ring of one) */
    int32_t detect;       /* 1: erode, count and decide (num_frames > MIN_FRAMES); 0: grey and MOG2 only */
    int32_t reserved;
} cpt_ir_motion_clip_step;
typedef struct {
    cpt_ir_motion *m;     /* the detector's grey ring */
    struct cpt_mog2 *mog2; /* its background model (cpt_mog2 below), of the same geometry */
    uint8_t *d_mask;      /* [H][W]: each step's foreground mask (0 / 255); the last one stays */
    int32_t first_step;   /* this clip's steps: h_steps[first_step .. first_step + n_steps) */
    int32_t n_steps;
    int32_t movement;     /* movement_detected on entry; on return, after the last step */
    int32_t triggered;    /* triggered on entry; on return, after the last step */
} cpt_ir_motion_clip;
typedef struct {
    int32_t threshold;        /* |oldest grey - grey| > threshold is a changed pixel (THRESHOLD) */
    int32_t trigger_frames;   /* TRIGGER_FRAMES */
    int32_t max_triggered;    /* the cap of triggered */
    int32_t erode_idle;       /* erosion box while not recording, 1..64 */
    int32_t erode_recording;  /* erosion box while recording, 1..64 */
    int32_t host_frames;      /* 1: h_frames are host addresses */
} cpt_ir_motion_clip_params;
typedef struct {
    int32_t movement;     /* movement_detected after the step */
    int32_t triggered;    /* triggered after the step */
    int32_t diff_pixels;  /* eroded counts before the min rule; -1 for a step without detect */
    int32_t mask_pixels;
} cpt_ir_motion_clip_result;
int cpt_ir_motion_clips(cpt_ctx *ctx, cpt_ir_motion_clip *h_clips, int n, const uint8_t *const *h_frames, int64_t n_frames,
                        const cpt_ir_motion_clip_step *h_steps, int n_steps, const cpt_ir_motion_clip_params *params,
                        cpt_ir_motion_clip_result *h_results);
/* One step of cpt_ir_motion_clips for the one clip h_clip (first_step and n_steps are not read, nor h_step->row or
 * params->host_frames): the host BGR frame h_bgr [H][W][3] goes through the detector's pinned staging with the step's
 * records in one copy; grey, MOG2 update, mask, erosion and trigger rule run as in cpt_ir_motion_clips, with the same
 * checks.  Waits; *h_result is the step's result and h_clip->movement / triggered hold the state after it. */
int cpt_ir_motion_step(cpt_ir_motion_clip *h_clip, const uint8_t *h_bgr, const cpt_ir_motion_clip_step *h_step,
                       const cpt_ir_motion_clip_params *params, cpt_ir_motion_clip_result *h_result);

/* ---- OpenCV's BackgroundSubtractorMOG2 (track/cliptracker.py:560-609 CVBackground; the IR detector's background model) ----
 * cv2.createBackgroundSubtractorMOG2(history, varThreshold, detectShadows=False) on one uint8 channel with five modes, bit for
 * bit: every foreground mask of apply() and getBackgroundImage().  The model's state (61 bytes per pixel) stays on the
 * device; one cpt_mog2_apply runs any number of consecutive frames (one launch per 256 frames, a new launch where a frame
 * re-initialises the model).  Launches go on the ctx stream and do not synchronise. */
typedef struct cpt_mog2_params {       /* cv2.createBackgroundSubtractorMOG2 defaults in brackets */
    int history;                       /* [500]; the reference's CVBackground uses 1000 */
    double var_threshold;              /* Tb [16] */
    double background_ratio;           /* TB [0.9] */
    float var_threshold_gen;           /* Tg [9] */
    float var_init, var_min, var_max;  /* [15, 4, 75] */
    float complexity_reduction;        /* fCT [0.05f] -- prune = (float)(-lr * (double)fCT) */
    int detect_shadows;                /* must be 0: the reference creates MOG2 with detectShadows=False */
} cpt_mog2_params;
typedef struct cpt_mog2 cpt_mog2;
cpt_mog2 *cpt_mog2_open(cpt_ctx *ctx, int width, int height, const cpt_mog2_params *p);
void cpt_mog2_close(cpt_mog2 *m);
/* n_frames uint8 frames at d_frames (frame_stride bytes apart) -> n_frames masks (0 / 255) at d_masks (may be NULL);
 * h_learning_rates[n_frames]: cv2's learningRate argument per frame (-1 = automatic, >= 1 re-initialises the model) */
int cpt_mog2_apply(cpt_mog2 *m, const uint8_t *d_frames, int n_frames, int64_t frame_stride,
                   const double *h_learning_rates, uint8_t *d_masks);
int cpt_mog2_background(cpt_mog2 *m, uint8_t *d_out);   /* getBackgroundImage: d_out [H][W] uint8 */
int cpt_mog2_frames(const cpt_mog2 *m);                 /* nframes as cv2 counts it (frames since the last initialisation) */

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
