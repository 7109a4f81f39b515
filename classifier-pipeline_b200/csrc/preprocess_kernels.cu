// preprocess_kernels.cu -- classifier-input preprocessing (K9, K10 of SURVEY.md section 8a) and its C ABI.
//
// Interpreter.preprocess_segments (ml_tools/interpreter.py:365-474) for many tracks at once:
//   track_limits_kernel      get_limits with diff_norm (interpreter.py:315-363): track-wide min / max of
//                            region.subimage(frame.filtered)
//   sample_median_kernel     pass 1: np.median(frame.thermal) per unique track-frame and the
//                            clip_thermals_at_zero test (interpreter.py:389-399)
//   segment_tiles_kernel     pass 2 + tiling fused: crop by region (frame.py:203-236), cv2.resize INTER_LINEAR to the
//                            aspect-preserving size, paste into the frame_size x frame_size tile
//                            (imageprocessing.py:11-70), thermal -= median, clip, normalise (preprocess.py:56-113)
//                            and write the tile straight into its cell of the (rows*size, cols*size, 2) segment
//                            image (preprocess_movement / square_clip, preprocess.py:151-202,
//                            imageprocessing.py:85-104): one CTA per (segment, tile); the crop is read from
//                            HBM/L2 once, the only large traffic is the coalesced float2 output rows.
// The same entry points also run on an extraction's own buffers, where a frame's thermal row (its row of the input) and its
// filtered row (its row of every per-frame output) differ, and reuse the per-frame statistics the extraction has already
// computed when the caller passes them:
//   sample_crop_median_kernel        pass 1 with the frame medians of cpt_frame_medians: only the crop is read
//   track_thermal_limits_stats_kernel  thermal_diff_norm limits from cpt_frame_info.thermal_min / thermal_max: no frame read
#include <cfloat>

#include "cptrack_internal.cuh"
#include "median.cuh"
#include "resize_cv.cuh"

namespace cpt {

namespace {

__device__ __forceinline__ void atomic_min_float(float *addr, float v) {
    int *a = reinterpret_cast<int *>(addr);
    int old = *a;
    while (v < __int_as_float(old)) {
        const int assumed = old;
        old = atomicCAS(a, assumed, __float_as_int(v));
        if (old == assumed) break;
    }
}

__device__ __forceinline__ void atomic_max_float(float *addr, float v) {
    int *a = reinterpret_cast<int *>(addr);
    int old = *a;
    while (v > __int_as_float(old)) {
        const int assumed = old;
        old = atomicCAS(a, assumed, __float_as_int(v));
        if (old == assumed) break;
    }
}

template <typename T, typename Op>
__device__ __forceinline__ T block_reduce(T v, T *scratch32, Op op, T identity) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
    for (int off = 16; off; off >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, off));
    __syncthreads();  // scratch may still be read from a previous reduction
    if (lane == 0) scratch32[warp] = v;
    __syncthreads();
    v = (lane < nwarps) ? scratch32[lane] : identity;
    for (int off = 16; off; off >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, off));
    return v;
}

// min, max and a second min in one pass over the block (one pair of barriers instead of three)
__device__ __forceinline__ void block_reduce_min_max_min(float &a, float &b, float &c, float *scratch96) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
    for (int off = 16; off; off >>= 1) {
        a = fminf(a, __shfl_xor_sync(0xffffffffu, a, off));
        b = fmaxf(b, __shfl_xor_sync(0xffffffffu, b, off));
        c = fminf(c, __shfl_xor_sync(0xffffffffu, c, off));
    }
    __syncthreads();  // scratch may still be read from a previous reduction
    if (lane == 0) { scratch96[warp] = a; scratch96[32 + warp] = b; scratch96[64 + warp] = c; }
    __syncthreads();
    a = (lane < nwarps) ? scratch96[lane] : FLT_MAX;
    b = (lane < nwarps) ? scratch96[32 + lane] : -FLT_MAX;
    c = (lane < nwarps) ? scratch96[64 + lane] : FLT_MAX;
    for (int off = 16; off; off >>= 1) {
        a = fminf(a, __shfl_xor_sync(0xffffffffu, a, off));
        b = fmaxf(b, __shfl_xor_sync(0xffffffffu, b, off));
        c = fminf(c, __shfl_xor_sync(0xffffffffu, c, off));
    }
}

struct MinF { __device__ float operator()(float a, float b) const { return fminf(a, b); } };
struct MaxF { __device__ float operator()(float a, float b) const { return fmaxf(a, b); } };

}  // namespace

// ------------------------------------------------------------------------------------------------
__global__ void track_norm_reset_kernel(cpt_track_norm *tracks, int n_tracks) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_tracks) {
        tracks[i].filtered_min = FLT_MAX;  // "None" until a region is seen
        tracks[i].filtered_max = 0.0f;     // interpreter.py:317 max_diff = 0
        tracks[i].clip_at_zero = 1;
        tracks[i].has_limits = 0;
        tracks[i].thermal_min = FLT_MAX;
        tracks[i].thermal_max = -FLT_MAX;
        tracks[i].has_thermal_limits = 0;
        tracks[i].reserved = 0;
    }
}

// thermal_diff_norm is on: until a region of the track is seen the limits are (None, None) -- per-tile extrema, no clip
__global__ void track_thermal_on_kernel(cpt_track_norm *tracks, int n_tracks) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_tracks) tracks[i].has_thermal_limits = 2;
}

// one warp per non-blank region of a track (a crop is a few hundred pixels: a warp's worth of work, and many warps in
// flight hide the cold reads; a 128-thread CTA per region with two block reductions took 1.6 ms for 450 k regions)
constexpr int kLimitsThreads = 256;
// filtered_rows (may be NULL: the region's frame): the filtered row of every region
__global__ void __launch_bounds__(kLimitsThreads) track_limits_kernel(const float *filtered, const int64_t *filtered_rows, int W, int H,
                                                                      const cpt_sample *regions, int n_regions, cpt_track_norm *tracks) {
    const int idx = blockIdx.x * (kLimitsThreads / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (idx >= n_regions) return;
    const cpt_sample r = regions[idx];
    const int64_t row = filtered_rows ? filtered_rows[idx] : r.frame;
    if (r.width <= 0 || r.height <= 0 || r.frame < 0 || row < 0) return;  // (a row without a frame or an area is nobody's region)
    const float *f = filtered + (size_t)row * W * H;
    float mn = FLT_MAX, mx = -FLT_MAX;
    const int n = r.width * r.height;
    const uint32_t rcp = 0xffffffffu / (uint32_t)r.width + 1u;  // i / width == umulhi(i, rcp) (wraps to 0 for width == 1)
    for (int i = lane; i < n; i += 32) {
        const int yy = r.width == 1 ? i : (int)__umulhi((uint32_t)i, rcp), xx = i - yy * r.width;
        const float v = __ldg(f + (r.y + yy) * W + r.x + xx);
        mn = fminf(mn, v);
        mx = fmaxf(mx, v);
    }
    for (int off = 16; off; off >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, off));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
    }
    if (lane == 0) {
        cpt_track_norm *t = tracks + r.track;
        atomic_min_float(&t->filtered_min, mn);
        atomic_max_float(&t->filtered_max, mx);
        t->has_limits = 1;
    }
}

// one CTA per unique track-frame
__global__ void __launch_bounds__(256) sample_median_kernel(const uint16_t *thermal, int W, int H, cpt_sample *samples,
                                                            cpt_track_norm *tracks) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint16_t *px = reinterpret_cast<uint16_t *>(smem_raw);
    uint32_t *bins = reinterpret_cast<uint32_t *>(smem_raw + (((size_t)W * H * sizeof(uint16_t) + 15) & ~(size_t)15));
    __shared__ int red[80];
    cpt_sample *sp = samples + blockIdx.x;
    const cpt_sample r = *sp;
    if (r.frame < 0) return;  // (a malformed table must not make the kernel read in front of the frames)
    const int npx = W * H;
    const uint16_t *src = thermal + (size_t)r.frame * npx;
    for (int i = threadIdx.x; i < npx / 8; i += blockDim.x) *reinterpret_cast<uint4 *>(px + i * 8) = ldg16(src + i * 8);
    for (int i = (npx / 8) * 8 + threadIdx.x; i < npx; i += blockDim.x) px[i] = src[i];
    __syncthreads();
    const int frame2 = rect_median_sum(px, W, 0, 0, W, H, bins, red);  // 2 * median
    int crop2 = 0;
    const bool has_crop = r.width > 0 && r.height > 0;
    if (has_crop) crop2 = rect_median_sum(px, W, r.x, r.y, r.width, r.height, bins, red);
    if (threadIdx.x == 0) {
        sp->median = 0.5f * (float)frame2;
        // np.median(float32(sub_thermal) - median) <= 0  (interpreter.py:393-399); every value is a multiple of 0.5
        if (has_crop && crop2 <= frame2) atomicAnd(&tracks[r.track].clip_at_zero, 0);
    }
}

// pass 1 when the frame medians are known (cpt_frame_medians over the same thermal rows): sample.median is looked up and only
// the crop is read for the clip_thermals_at_zero test -- a few hundred pixels instead of the 19 200 of a frame, so a small CTA
// that reads them straight from L2 (no staging; the two passes of median.cuh touch the crop twice)
constexpr int kCropMedianThreads = 128;
__global__ void __launch_bounds__(kCropMedianThreads) sample_crop_median_kernel(const uint16_t *thermal, int W, int H,
                                                                               const float *frame_medians, cpt_sample *samples,
                                                                               cpt_track_norm *tracks) {
    __shared__ uint32_t bins[kMedianBins];
    __shared__ int red[80];
    cpt_sample *sp = samples + blockIdx.x;
    const cpt_sample r = *sp;
    if (r.frame < 0) return;
    const float median = __ldg(frame_medians + r.frame);
    const bool has_crop = r.width > 0 && r.height > 0;
    int crop2 = 0;
    if (has_crop)
        crop2 = rect_median_sum<kCropMedianThreads>(thermal + (size_t)r.frame * W * H, W, r.x, r.y, r.width, r.height, bins, red);
    if (threadIdx.x == 0) {
        sp->median = median;
        // the same integer test as sample_median_kernel: 2 * median is exact (a multiple of 0.5 below 2^16)
        if (has_crop && crop2 <= __float2int_rn(2.0f * median)) atomicAnd(&tracks[r.track].clip_at_zero, 0);
    }
}

// get_limits with thermal_diff_norm: one CTA per non-blank region of a track -- the extrema of frame.thermal - median over
// the whole frame (interpreter.py:338-345; float32 arithmetic on integer / half-integer values: exact)
__global__ void __launch_bounds__(256) track_thermal_limits_kernel(const uint16_t *thermal, int W, int H, const cpt_sample *regions,
                                                                   cpt_track_norm *tracks) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint16_t *px = reinterpret_cast<uint16_t *>(smem_raw);
    uint32_t *bins = reinterpret_cast<uint32_t *>(smem_raw + (((size_t)W * H * sizeof(uint16_t) + 15) & ~(size_t)15));
    __shared__ int red[80];
    __shared__ float scratch3[96];
    const cpt_sample r = regions[blockIdx.x];
    if (r.width <= 0 || r.height <= 0 || r.frame < 0) return;
    const int npx = W * H;
    const uint16_t *src = thermal + (size_t)r.frame * npx;
    float mn = FLT_MAX, mx = -FLT_MAX, unused = FLT_MAX;
    for (int i = threadIdx.x; i < npx / 8; i += blockDim.x) {
        const uint4 q = ldg16(src + i * 8);
        *reinterpret_cast<uint4 *>(px + i * 8) = q;
        const uint32_t ws[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float lo = (float)(ws[k] & 0xffffu), hi = (float)(ws[k] >> 16);
            mn = fminf(mn, fminf(lo, hi));
            mx = fmaxf(mx, fmaxf(lo, hi));
        }
    }
    for (int i = (npx / 8) * 8 + threadIdx.x; i < npx; i += blockDim.x) {
        const uint16_t v = src[i];
        px[i] = v;
        mn = fminf(mn, (float)v);
        mx = fmaxf(mx, (float)v);
    }
    block_reduce_min_max_min(mn, mx, unused, scratch3);  // (its barriers also publish the staged frame)
    const int frame2 = rect_median_sum(px, W, 0, 0, W, H, bins, red);  // 2 * median
    if (threadIdx.x == 0) {
        const float median = 0.5f * (float)frame2;
        cpt_track_norm *t = tracks + r.track;
        atomic_min_float(&t->thermal_min, __fsub_rn(mn, median));
        atomic_max_float(&t->thermal_max, __fsub_rn(mx, median));
        t->has_thermal_limits = 1;
    }
}

// the same limits from the extraction's per-frame statistics: frame extrema from cpt_frame_info (indexed by the filtered row,
// like every per-frame output) and the median from cpt_frame_medians (indexed by the thermal row); one thread per region
__global__ void track_thermal_limits_stats_kernel(const cpt_sample *regions, const int64_t *filtered_rows, int n_regions,
                                                  const float *frame_medians, const cpt_frame_info *info, cpt_track_norm *tracks) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_regions) return;
    const cpt_sample r = regions[idx];
    const int64_t row = filtered_rows ? filtered_rows[idx] : r.frame;
    if (r.width <= 0 || r.height <= 0 || r.frame < 0 || row < 0) return;
    const float median = __ldg(frame_medians + r.frame);
    cpt_track_norm *t = tracks + r.track;
    atomic_min_float(&t->thermal_min, __fsub_rn((float)info[row].thermal_min, median));
    atomic_max_float(&t->thermal_max, __fsub_rn((float)info[row].thermal_max, median));
    t->has_thermal_limits = 1;
}

// ------------------------------------------------------------------------------------------------
// normalize(data, min, max, new_max=255) of imageprocessing.py:151-169 on fp32
__device__ __forceinline__ float normalize255(float v, float mn, float mx) {
    if (mx == mn) return (mx == 0.0f) ? 0.0f : __fdiv_rn(v, mx);
    return __fdiv_rn(__fmul_rn(255.0f, __fsub_rn(v, mn)), __fsub_rn(mx, mn));
}

struct SegmentArgs {
    const uint16_t *thermal;
    const float *filtered;
    const int64_t *filtered_rows;    // [n_samples] filtered row of every sample, or NULL: the sample's frame
    const cpt_sample *samples;
    const cpt_track_norm *tracks;
    const int32_t *segment_samples;  // [n_segments][tiles]
    float *out;                      // [n_segments][rows*size][cols*size][2]
    int W, H;
    int tiles, per_row, size;
    int crop_x, crop_y, crop_w, crop_h;
    int preprocess_fn;
};

constexpr int kMaxTile = 64;  // frame_size <= 64

constexpr int kTileThreads = 128;  // (64 x-taps + 64 y-taps are set up by threads 0..127)
__global__ void __launch_bounds__(kTileThreads) segment_tiles_kernel(const SegmentArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *tile_t = reinterpret_cast<float *>(smem_raw);   // [size*size] thermal
    float *tile_f = tile_t + a.size * a.size;              // [size*size] filtered
    __shared__ float scratch[32], scratch3[96];
    __shared__ ResizeTaps tx[kMaxTile], ty[kMaxTile];
    const int seg = blockIdx.x / a.tiles, tile = blockIdx.x - seg * a.tiles;
    const int sidx = a.segment_samples[blockIdx.x];
    const cpt_sample r = a.samples[sidx];
    const int64_t frow = a.filtered_rows ? a.filtered_rows[sidx] : r.frame;
    if (r.frame < 0 || frow < 0 || r.width <= 0 || r.height <= 0) return;  // (malformed table: the tile is left as it is)
    const cpt_track_norm tn = a.tracks[r.track];
    const int size = a.size, n = size * size, tid = threadIdx.x;
    const int sw = r.width, sh = r.height;
    const uint16_t *th = a.thermal + (size_t)r.frame * a.W * a.H + r.y * a.W + r.x;
    const float *fl = a.filtered + (size_t)frow * a.W * a.H + r.y * a.W + r.x;

    // ---- target size and paste offsets (imageprocessing.py:24-59)
    const double scale = fmin((double)size / (double)sh, (double)size / (double)sw);
    const int fw = min(max((int)rint((double)sw * scale), 1), size);
    const int fh = min(max((int)rint((double)sh * scale), 1), size);
    int ox = (size - fw) / 2, oy = (size - fh) / 2;
    if (a.crop_w > 0) {  // keep_edge=True with a crop rectangle
        if (r.x <= a.crop_x) ox = min(0, size - fw);
        else if (r.x + sw >= a.crop_x + a.crop_w) ox = max(size - fw, 0);
        if (r.y <= a.crop_y) oy = min(0, size - fh);
        else if (r.y + sh >= a.crop_y + a.crop_h) oy = max(size - fh, 0);
    }
    // cv2.resize INTER_LINEAR (resize_cv.cuh); a same-size resize is a copy, as cv2 makes it
    const bool thin = sw == 1 || sh == 1, copy = fw == sw && fh == sh;
    if (tid < fw) tx[tid] = linear_taps(tid, fw, sw, thin, true);
    if (tid >= 64 && tid - 64 < fh) ty[tid - 64] = linear_taps(tid - 64, fh, sh, thin, !thin);

    // (index arithmetic without divisions: i / sw by a reciprocal multiply, i / size by a shift for the usual power of two)
    const uint32_t sw_rcp = 0xffffffffu / (uint32_t)sw + 1u;  // i / sw == umulhi(i, sw_rcp) for i * sw < 2^32 (wraps to 0 for sw == 1)
    const int size_shift = (size & (size - 1)) == 0 ? __ffs(size) - 1 : -1;
    // ---- pad value of the thermal tile: min of the crop (imageprocessing.py:36-37)
    float pad = FLT_MAX;
    for (int i = tid; i < sw * sh; i += blockDim.x) {
        const int yy = sw == 1 ? i : (int)__umulhi((uint32_t)i, sw_rcp), xx = i - yy * sw;
        pad = fminf(pad, (float)__ldg(th + yy * a.W + xx));
    }
    pad = block_reduce(pad, scratch, MinF(), FLT_MAX);  // (also orders the tap tables before their use)

    // ---- resize + paste, thermal -= median, clip unless thermal limits were asked for (preprocess.py:90-93)
    const bool clip0 = tn.clip_at_zero != 0 && tn.has_thermal_limits == 0;
    const bool per_tile = (a.preprocess_fn & CPT_PREPROCESS_PER_TILE) != 0;  // diff_norm off: Frame.normalize, both channels
    float tmin = FLT_MAX, tmax = -FLT_MAX, fmin_ = FLT_MAX, fmax_ = -FLT_MAX;
    for (int i = tid; i < n; i += blockDim.x) {
        const int y = size_shift >= 0 ? (i >> size_shift) : i / size, x = i - y * size;
        const int dx = x - ox, dy = y - oy;
        float t = pad, f = 0.0f;
        if (dx >= 0 && dx < fw && dy >= 0 && dy < fh) {
            if (copy) {
                t = (float)__ldg(th + dy * a.W + dx);
                f = __ldg(fl + dy * a.W + dx);
            } else {
                const ResizeTaps X = tx[dx], Y = ty[dy];
                const uint16_t *r0 = th + Y.i0 * a.W, *r1 = th + Y.i1 * a.W;
                t = lerp_cv(lerp_cv((float)__ldg(r0 + X.i0), (float)__ldg(r0 + X.i1), X.w, thin),
                            lerp_cv((float)__ldg(r1 + X.i0), (float)__ldg(r1 + X.i1), X.w, thin), Y.w, thin);
                const float *g0 = fl + Y.i0 * a.W, *g1 = fl + Y.i1 * a.W;
                f = lerp_cv(lerp_cv(__ldg(g0 + X.i0), __ldg(g0 + X.i1), X.w, thin),
                            lerp_cv(__ldg(g1 + X.i0), __ldg(g1 + X.i1), X.w, thin), Y.w, thin);
            }
        }
        t = __fsub_rn(t, r.median);
        if (clip0) t = fmaxf(t, 0.0f);
        tile_t[i] = t;
        tile_f[i] = f;
        tmin = fminf(tmin, t);
        tmax = fmaxf(tmax, t);
        fmin_ = fminf(fmin_, f);
        fmax_ = fmaxf(fmax_, f);
    }
    block_reduce_min_max_min(tmin, tmax, fmin_, scratch3);
    float lo = tn.filtered_min, hi = tn.filtered_max;
    if (!tn.has_limits) lo = fmin_;  // min=None: the tile's own minimum
    if (per_tile) {
        fmax_ = block_reduce(fmax_, scratch, MaxF(), -FLT_MAX);
        lo = fmin_;
        hi = fmax_;
    } else if (tn.has_thermal_limits == 1) {
        tmin = tn.thermal_min;  // (only used together with filtered limits: preprocess.py:96-110)
        tmax = tn.thermal_max;
    }

    // ---- normalise and write the cell: image[row*size + y][col*size + x][channel]
    const int row = tile / a.per_row, col = tile - row * a.per_row;
    const int img_w = a.per_row * size, img_h = ((a.tiles + a.per_row - 1) / a.per_row) * size;
    float2 *img = reinterpret_cast<float2 *>(a.out) + (size_t)seg * img_w * img_h;
    for (int i = tid; i < n; i += blockDim.x) {
        const int y = size_shift >= 0 ? (i >> size_shift) : i / size, x = i - y * size;
        float t = normalize255(tile_t[i], tmin, tmax), f = normalize255(tile_f[i], lo, hi);
        if (a.preprocess_fn & CPT_PREPROCESS_INC3) {  // x /= 127.5; x -= 1.0 (preprocess.py:19-22)
            t = __fsub_rn(__fdiv_rn(t, 127.5f), 1.0f);
            f = __fsub_rn(__fdiv_rn(f, 127.5f), 1.0f);
        }
        img[(size_t)(row * size + y) * img_w + col * size + x] = make_float2(t, f);
    }
}

}  // namespace cpt

// ================================================================================================
using cpt::fail;

extern "C" {

int cpt_preprocess_limits(cpt_ctx *c, const float *d_filtered, const int64_t *d_filtered_rows, const cpt_sample *d_regions,
                          int n_regions, cpt_track_norm *d_tracks, int n_tracks) {
    if (!c || !d_tracks) return fail(CPT_ERR_INVALID, "null argument");
    if (n_regions < 0 || n_tracks < 0) return fail(CPT_ERR_INVALID, "negative count");
    if (n_tracks == 0) return CPT_OK;
    CUDA_TRY(cudaSetDevice(c->device));
    cpt::track_norm_reset_kernel<<<(n_tracks + 255) / 256, 256, 0, c->stream>>>(d_tracks, n_tracks);
    if (n_regions > 0) {
        if (!d_filtered || !d_regions) return fail(CPT_ERR_INVALID, "null filtered / regions");
        cpt::track_limits_kernel<<<(n_regions + cpt::kLimitsThreads / 32 - 1) / (cpt::kLimitsThreads / 32), cpt::kLimitsThreads, 0, c->stream>>>(
            d_filtered, d_filtered_rows, c->g.W, c->g.H, d_regions, n_regions, d_tracks);
    }
    CUDA_TRY(cudaGetLastError());
    return CPT_OK;
}

int cpt_preprocess_thermal_limits(cpt_ctx *c, const uint16_t *d_thermal, const int64_t *d_filtered_rows, const cpt_sample *d_regions,
                                  int n_regions, cpt_track_norm *d_tracks, int n_tracks, const float *d_frame_medians,
                                  const cpt_frame_info *d_frame_info) {
    if (!c || !d_tracks) return fail(CPT_ERR_INVALID, "null argument");
    if (n_regions < 0 || n_tracks < 0) return fail(CPT_ERR_INVALID, "negative count");
    if (n_tracks == 0) return CPT_OK;
    CUDA_TRY(cudaSetDevice(c->device));
    cpt::track_thermal_on_kernel<<<(n_tracks + 255) / 256, 256, 0, c->stream>>>(d_tracks, n_tracks);
    if (n_regions > 0) {
        if (!d_regions) return fail(CPT_ERR_INVALID, "null regions");
        if (d_frame_medians && d_frame_info) {
            cpt::track_thermal_limits_stats_kernel<<<(n_regions + 255) / 256, 256, 0, c->stream>>>(d_regions, d_filtered_rows, n_regions,
                                                                                              d_frame_medians, d_frame_info, d_tracks);
        } else {
            if (!d_thermal) return fail(CPT_ERR_INVALID, "null thermal");
            const size_t smem = (((size_t)c->g.npx * sizeof(uint16_t) + 15) & ~(size_t)15) + cpt::kMedianBins * sizeof(uint32_t);
            cpt::track_thermal_limits_kernel<<<n_regions, 256, smem, c->stream>>>(d_thermal, c->g.W, c->g.H, d_regions, d_tracks);
        }
    }
    CUDA_TRY(cudaGetLastError());
    return CPT_OK;
}

int cpt_preprocess_medians(cpt_ctx *c, const uint16_t *d_thermal, const float *d_frame_medians, cpt_sample *d_samples, int n_samples,
                           cpt_track_norm *d_tracks) {
    if (!c) return fail(CPT_ERR_INVALID, "null ctx");
    if (n_samples < 0) return fail(CPT_ERR_INVALID, "negative count");
    if (n_samples == 0) return CPT_OK;
    if (!d_thermal || !d_samples || !d_tracks) return fail(CPT_ERR_INVALID, "null argument");
    CUDA_TRY(cudaSetDevice(c->device));
    if (d_frame_medians) {
        cpt::sample_crop_median_kernel<<<n_samples, cpt::kCropMedianThreads, 0, c->stream>>>(d_thermal, c->g.W, c->g.H, d_frame_medians,
                                                                                          d_samples, d_tracks);
    } else {
        const size_t smem = (((size_t)c->g.npx * sizeof(uint16_t) + 15) & ~(size_t)15) + cpt::kMedianBins * sizeof(uint32_t);
        cpt::sample_median_kernel<<<n_samples, 256, smem, c->stream>>>(d_thermal, c->g.W, c->g.H, d_samples, d_tracks);
    }
    CUDA_TRY(cudaGetLastError());
    return CPT_OK;
}

int cpt_preprocess_segments(cpt_ctx *c, const uint16_t *d_thermal, const float *d_filtered, const int64_t *d_filtered_rows,
                            const cpt_sample *d_samples, const cpt_track_norm *d_tracks, const int32_t *d_segment_samples,
                            int n_segments, int tiles_per_segment, int frames_per_row, int frame_size,
                            const int32_t *crop_rectangle, int preprocess_fn, float *d_out) {
    if (!c) return fail(CPT_ERR_INVALID, "null ctx");
    if (n_segments < 0) return fail(CPT_ERR_INVALID, "negative count");
    if (n_segments == 0) return CPT_OK;
    if (!d_thermal || !d_filtered || !d_samples || !d_tracks || !d_segment_samples || !d_out)
        return fail(CPT_ERR_INVALID, "null argument");
    if (tiles_per_segment < 1 || frames_per_row < 1 || frame_size < 1 || frame_size > cpt::kMaxTile)
        return fail(CPT_ERR_INVALID, "bad tiling (frame_size must be in [1,%d])", cpt::kMaxTile);
    if (preprocess_fn & ~(CPT_PREPROCESS_INC3 | CPT_PREPROCESS_PER_TILE)) return fail(CPT_ERR_INVALID, "preprocess_fn: unknown flag");
    if ((long long)n_segments * tiles_per_segment > 0x7fffffffll) return fail(CPT_ERR_INVALID, "too many tiles for one launch");
    CUDA_TRY(cudaSetDevice(c->device));
    cpt::SegmentArgs a{};
    a.thermal = d_thermal; a.filtered = d_filtered; a.filtered_rows = d_filtered_rows; a.samples = d_samples; a.tracks = d_tracks;
    a.segment_samples = d_segment_samples; a.out = d_out;
    a.W = c->g.W; a.H = c->g.H;
    a.tiles = tiles_per_segment; a.per_row = frames_per_row; a.size = frame_size;
    if (crop_rectangle) {
        a.crop_x = crop_rectangle[0]; a.crop_y = crop_rectangle[1]; a.crop_w = crop_rectangle[2]; a.crop_h = crop_rectangle[3];
    }
    a.preprocess_fn = preprocess_fn;
    const size_t smem = (size_t)2 * frame_size * frame_size * sizeof(float);
    cpt::segment_tiles_kernel<<<(unsigned)(n_segments * tiles_per_segment), cpt::kTileThreads, smem, c->stream>>>(a);
    CUDA_TRY(cudaGetLastError());
    return CPT_OK;
}

}  // extern "C"
