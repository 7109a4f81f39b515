// detect_kernels.cu -- imageprocessing.detect_objects (ml_tools/imageprocessing.py:240-248) for one image of any size,
// and detect_objects_ir for a batch of frames of one geometry (the extraction kernel fuses the same steps for 160x120 clips
// in shared memory; this is the stand-alone primitive, also the building block for the 640x480 IR frames of SURVEY.md
// section 8f-4):
//   close_init_kernel       cv2.morphologyEx(MORPH_CLOSE, <tuple>): the tuple becomes a 2x1 element, i.e.
//                           C[y] = M[y-1] | (M[y] & M[y-2]), C[0] = C[1] = M[0]; seeds the union-find
//   merge / flatten         8-connected label equivalence in global memory (union by smaller index, atomicMin); flatten
//                           also takes each component's least 2x2 block key (block-raster order)
//   mark / scan / rank      OpenCV label numbering: a bitmap over the block keys, a popcount prefix per frame, and the
//                           rank of each component's key in it
//   stats_kernel            per-component bbox / area / centroid sums with atomics on the label's row
//   write_stats_kernel      cv2-shaped stats rows and centroids
//   relabel_kernel          int32 label image
// The passes that both the single-image call and the batch run take the frame from blockIdx.y: pixel indices are per
// frame (int, a frame holds at most 2^26 pixels) and the frame's base offset is size_t.
#include <algorithm>
#include <climits>
#include <cmath>

#include "cptrack_internal.cuh"

namespace cpt {

namespace {

struct CompStats {
    int area, min_x, max_x, min_y, max_y;
    unsigned long long sum_x, sum_y;
};

__device__ __forceinline__ int reflect(int p, int n) {
    if (n == 1) return 0;
    while (p < 0 || p >= n) p = (p < 0) ? -p : 2 * n - 2 - p;
    return p;
}

__device__ __forceinline__ int find_root(const int *parent, int a) {
    while (true) {
        const int p = parent[a];
        if (p == a) return a;
        a = p;
    }
}

__device__ __forceinline__ void unite(int *parent, int a, int b) {
    while (true) {
        a = find_root(parent, a);
        b = find_root(parent, b);
        if (a == b) return;
        if (a < b) { const int t = a; a = b; b = t; }
        const int old = atomicMin(parent + a, b);  // a > b: hang the larger root under the smaller index
        if (old == a) return;
        a = old;
    }
}

// offset of frame blockIdx.y in arrays of `per_frame` elements per frame
__device__ __forceinline__ size_t frame_off(size_t per_frame) { return (size_t)blockIdx.y * per_frame; }

// 32-bit words of the per-frame bitmap over the 2x2 block keys
__host__ __device__ __forceinline__ int key_words(int W, int H) { return (((W + 1) >> 1) * ((H + 1) >> 1) + 31) >> 5; }

}  // namespace

// cv2.GaussianBlur(u8, (k, k), 0) for k in {3, 5, 7, 15}: OpenCV's 8-bit path uses fixed-point taps that sum to 256 and
// rounds once, (sum_y K_y sum_x K_x U + 2^15) >> 16, BORDER_REFLECT_101 (taps of 15 probed from cv2 4.13: a column of 255
// blurs to exactly these values; 3 / 5 / 7 are the exact binary fractions of getGaussianKernel's fixed tables).
__constant__ int kGaussTaps[4][15] = {
    {64, 128, 64}, {16, 64, 96, 64, 16}, {8, 28, 56, 72, 56, 28, 8}, {1, 3, 6, 12, 20, 30, 36, 40, 36, 30, 20, 12, 6, 3, 1}};

__global__ void __launch_bounds__(256) gauss_blur_kernel(const uint8_t *img, int W, int H, int ksize, int table, uint8_t *out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W * H) return;
    const int y = i / W, x = i - y * W, r = ksize >> 1;
    int acc = 0;
    for (int dy = -r; dy <= r; ++dy) {
        const uint8_t *row = img + reflect(y + dy, H) * W;
        int h = 0;
        for (int dx = -r; dx <= r; ++dx) h += kGaussTaps[table][dx + r] * (int)__ldg(row + reflect(x + dx, W));
        acc += kGaussTaps[table][dy + r] * h;
    }
    out[i] = (uint8_t)((acc + 32768) >> 16);
}

// cv2.morphologyEx(u8, MORPH_OPEN, <tuple>) on a grey image: the tuple becomes a 2x1 element (rows y-1, y), so
// E[y] = min(I[y-1], I[y]), O[y] = max(E[y-1], E[y]); rows outside the image do not constrain (ml_tools/imageprocessing.py:189)
__global__ void __launch_bounds__(256) open_gray_kernel(const uint8_t *img, int W, int H, uint8_t *out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W * H) return;
    img += frame_off((size_t)W * H);
    out += frame_off((size_t)W * H);
    const int y = i / W;
    const int a = img[i], b = y >= 1 ? img[i - W] : a, c = y >= 2 ? img[i - 2 * W] : b;
    const int e1 = min(b, a), e0 = y >= 1 ? min(c, b) : e1;  // E[y], E[y-1]
    out[i] = (uint8_t)max(e0, e1);
}

__global__ void __launch_bounds__(256) threshold_kernel(const uint8_t *img, int n, int ithresh, uint8_t *mask) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    img += frame_off(n);
    mask += frame_off(n);
    mask[i] = img[i] > ithresh ? 1 : 0;
}

// cv2.dilate(mask, <tuple>): D[y] = M[y-1] | M[y]
__global__ void __launch_bounds__(256) dilate_rows_kernel(const uint8_t *mask, int W, int H, uint8_t *out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W * H) return;
    out[i] = (uint8_t)(mask[i] | (i >= W ? mask[i - W] : 0));
}

__global__ void __launch_bounds__(256) or_mask_kernel(uint8_t *mask, const uint8_t *other, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) mask[i] = (uint8_t)((mask[i] | (other[i] ? 1 : 0)) ? 1 : 0);
}

__global__ void __launch_bounds__(256) histogram_kernel(const uint8_t *img, int n, unsigned int *hist) {
    __shared__ unsigned int h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) atomicAdd(&h[img[i]], 1u);
    __syncthreads();
    if (h[threadIdx.x]) atomicAdd(&hist[threadIdx.x], h[threadIdx.x]);
}

__global__ void __launch_bounds__(256) mask_out_kernel(const uint8_t *mask, int n, uint8_t *out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = mask[i] ? 255 : 0;
}

// seeds parent (own index or -1) and the least-key holder of every pixel (INT_MAX) for flatten_kernel
__global__ void __launch_bounds__(256) close_init_kernel(const uint8_t *mask, int W, int H, int close, int *parent, int *key_of) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W * H) return;
    mask += frame_off((size_t)W * H);
    parent += frame_off((size_t)W * H);
    key_of += frame_off((size_t)W * H);
    const int y = i / W;
    int c;
    if (!close) c = mask[i];
    else if (y == 0) c = mask[i];
    else if (y == 1) c = mask[i - W];
    else c = mask[i - W] | (mask[i] & mask[i - 2 * W]);
    parent[i] = c ? i : -1;
    key_of[i] = INT_MAX;
}

__global__ void __launch_bounds__(256) parent_to_mask_kernel(const int *parent, int n, uint8_t *mask) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) mask[i] = parent[i] >= 0 ? 1 : 0;
}

__global__ void __launch_bounds__(256) merge_kernel(int *parent, int W, int H) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W * H) return;
    parent += frame_off((size_t)W * H);
    if (parent[i] < 0) return;
    const int y = i / W, x = i - y * W;
    if (x > 0 && parent[i - 1] >= 0) unite(parent, i, i - 1);
    if (y > 0) {
        if (parent[i - W] >= 0) unite(parent, i, i - W);
        if (x > 0 && parent[i - W - 1] >= 0) unite(parent, i, i - W - 1);
        if (x + 1 < W && parent[i - W + 1] >= 0) unite(parent, i, i - W + 1);
    }
}

// parent -> root; the root's key_of entry takes the least 2x2 block key (block-raster order) of the component's pixels.
// Keys are unique per component: any two set pixels of one 2x2 block are 8-connected.
__global__ void __launch_bounds__(256) flatten_kernel(int *parent, int W, int H, int *key_of) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W * H) return;
    parent += frame_off((size_t)W * H);
    key_of += frame_off((size_t)W * H);
    if (parent[i] < 0) return;
    const int r = find_root(parent, i);
    parent[i] = r;
    const int y = i / W, x = i - y * W;
    atomicMin(key_of + r, (y >> 1) * ((W + 1) >> 1) + (x >> 1));
}

__global__ void __launch_bounds__(256) mark_kernel(const int *parent, const int *key_of, int W, int H, uint32_t *bitmap) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W * H) return;
    parent += frame_off((size_t)W * H);
    if (parent[i] != i) return;
    const int k = key_of[frame_off((size_t)W * H) + i];
    atomicOr(bitmap + frame_off(key_words(W, H)) + (k >> 5), 1u << (k & 31));
}

// one block of kScanThreads per frame: exclusive popcount prefix of the frame's bitmap words; the frame's component count
// to n_roots[f] and, when counts is given, cv2's label count (background included) to counts[f]
constexpr int kScanThreads = 1024;
__global__ void __launch_bounds__(kScanThreads) scan_kernel(const uint32_t *bitmap, int words, int *prefix, int *n_roots, int32_t *counts) {
    __shared__ int warp_sums[kScanThreads / 32];
    bitmap += frame_off(words);
    prefix += frame_off(words);
    const int per = (words + kScanThreads - 1) / kScanThreads;
    const int w0 = min(words, threadIdx.x * per), w1 = min(words, w0 + per);
    int own = 0;
    for (int w = w0; w < w1; ++w) own += __popc(bitmap[w]);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = own;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += v;
    }
    if (lane == 31) warp_sums[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int s = warp_sums[lane];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, s, d);
            if (lane >= d) s += v;
        }
        warp_sums[lane] = s;  // inclusive over warps
    }
    __syncthreads();
    int run = incl - own + (warp > 0 ? warp_sums[warp - 1] : 0);
    for (int w = w0; w < w1; ++w) {
        prefix[w] = run;
        run += __popc(bitmap[w]);
    }
    if (threadIdx.x == 0) {
        const int n = warp_sums[kScanThreads / 32 - 1];
        n_roots[blockIdx.y] = n;
        if (counts) counts[blockIdx.y] = n + 1;
    }
}

__device__ __forceinline__ void reset_stats(CompStats *s) {
    CompStats c;
    c.area = 0; c.min_x = INT_MAX; c.max_x = -1; c.min_y = INT_MAX; c.max_y = -1; c.sum_x = 0; c.sum_y = 0;
    *s = c;
}

// each root's key_of entry becomes its label (rank of the key + 1); the stats rows the frame will fill are reset
__global__ void __launch_bounds__(256) rank_kernel(const int *parent, int *key_of, int W, int H, const uint32_t *bitmap, const int *prefix,
                                                   int max_components, CompStats *stats) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W * H) return;
    parent += frame_off((size_t)W * H);
    key_of += frame_off((size_t)W * H);
    stats += frame_off((size_t)max_components + 1);
    if (i == 0) reset_stats(stats);
    if (parent[i] != i) return;
    const int k = key_of[i], words = key_words(W, H);
    const size_t w = frame_off(words) + (k >> 5);
    const int label = prefix[w] + __popc(bitmap[w] & ((1u << (k & 31)) - 1u)) + 1;
    key_of[i] = label;
    if (label <= max_components) reset_stats(stats + label);
}

// Row 0 (the background) takes one set of atomics per warp: most pixels of a frame are background.
__global__ void __launch_bounds__(256) stats_kernel(const int *parent, const int *label_of, int W, int H, int max_components, int sums,
                                                    CompStats *stats) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int npx = W * H;
    parent += frame_off(npx);
    label_of += frame_off(npx);
    stats += frame_off((size_t)max_components + 1);
    const bool in = i < npx;
    const int y = in ? i / W : 0, x = i - y * W;
    int label = -1;
    if (in) label = parent[i] < 0 ? 0 : label_of[parent[i]];
    const bool bg = label == 0;
    const unsigned bgm = __ballot_sync(0xffffffffu, bg);
    if (bgm) {
        const int mnx = __reduce_min_sync(0xffffffffu, bg ? x : INT_MAX), mxx = __reduce_max_sync(0xffffffffu, bg ? x : -1);
        const int mny = __reduce_min_sync(0xffffffffu, bg ? y : INT_MAX), mxy = __reduce_max_sync(0xffffffffu, bg ? y : -1);
        unsigned sx = 0, sy = 0;
        if (sums) {  // 32 coordinates below 2^26 fit in 32 bits
            sx = __reduce_add_sync(0xffffffffu, bg ? (unsigned)x : 0u);
            sy = __reduce_add_sync(0xffffffffu, bg ? (unsigned)y : 0u);
        }
        if ((threadIdx.x & 31) == __ffs(bgm) - 1) {
            atomicAdd(&stats->area, __popc(bgm));
            atomicMin(&stats->min_x, mnx);
            atomicMax(&stats->max_x, mxx);
            atomicMin(&stats->min_y, mny);
            atomicMax(&stats->max_y, mxy);
            if (sums) {
                atomicAdd(&stats->sum_x, (unsigned long long)sx);
                atomicAdd(&stats->sum_y, (unsigned long long)sy);
            }
        }
    }
    if (label < 1 || label > max_components) return;
    CompStats *s = stats + label;
    atomicAdd(&s->area, 1);
    atomicMin(&s->min_x, x);
    atomicMax(&s->max_x, x);
    atomicMin(&s->min_y, y);
    atomicMax(&s->max_y, y);
    if (sums) {
        atomicAdd(&s->sum_x, (unsigned long long)x);
        atomicAdd(&s->sum_y, (unsigned long long)y);
    }
}

// rows 0 .. min(n, max_components) of the frame in cv2's shape; out_centroids may be NULL
__global__ void __launch_bounds__(256) write_stats_kernel(const CompStats *stats, const int *n_roots, int max_components, int32_t *out_stats,
                                                          double *out_centroids) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s > min(n_roots[blockIdx.y], max_components)) return;
    const size_t row = frame_off((size_t)max_components + 1) + s;
    const CompStats c = stats[row];
    int32_t *o = out_stats + row * 5;
    double *ce = out_centroids ? out_centroids + row * 2 : nullptr;
    if (c.area > 0) {
        o[0] = c.min_x; o[1] = c.min_y; o[2] = c.max_x - c.min_x + 1; o[3] = c.max_y - c.min_y + 1; o[4] = c.area;
        if (ce) {
            ce[0] = (double)c.sum_x / (double)c.area;
            ce[1] = (double)c.sum_y / (double)c.area;
        }
    } else {  // only the background of an all-foreground image: cv2 4.13 reports [-1, INT_MAX, 0, 0, 0] and a NaN centroid
        o[0] = -1; o[1] = INT_MAX; o[2] = 0; o[3] = 0; o[4] = 0;
        if (ce) ce[0] = ce[1] = nan("");
    }
}

__global__ void __launch_bounds__(256) relabel_kernel(const int *parent, const int *label_of, int n, int32_t *labels) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    parent += frame_off(n);
    label_of += frame_off(n);
    labels[frame_off(n) + i] = parent[i] < 0 ? 0 : label_of[parent[i]];
}

namespace {

// Scratch of the components passes for `frames` frames: per frame a grey and a mask image, parent and key / label (4 B per
// pixel each), the key bitmap and its prefix, the stats rows and the component count.  `extra` adds what only the
// single-image call uses: a second grey and mask image and the Otsu histogram.
struct DetectScratch {
    uint8_t *grey, *mask, *grey_b, *mask_b;
    int *parent, *key_of, *prefix, *n_roots;
    uint32_t *bitmap;
    CompStats *stats;
    unsigned int *hist;
};

inline size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

size_t detect_scratch_bytes(int W, int H, int frames, int max_components, bool extra, DetectScratch *out = nullptr, uint8_t *base = nullptr) {
    const size_t npx = (size_t)W * H, F = (size_t)frames, words = (size_t)key_words(W, H);
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += align256(bytes); return base + o; };
    DetectScratch s{};
    s.grey = take(F * npx);
    s.mask = take(F * npx);
    s.parent = (int *)take(F * npx * 4);
    s.key_of = (int *)take(F * npx * 4);
    s.bitmap = (uint32_t *)take(F * words * 4);
    s.prefix = (int *)take(F * words * 4);
    s.stats = (CompStats *)take(F * ((size_t)max_components + 1) * sizeof(CompStats));
    s.n_roots = (int *)take(F * 4);
    if (extra) {
        s.grey_b = take(npx);
        s.mask_b = take(npx);
        s.hist = (unsigned int *)take(256 * sizeof(unsigned int));
    }
    if (out) *out = s;
    return off;
}

// The components passes from the seeded mask (close_init_kernel done) to the outputs, for gridDim.y = frames frames.
// counts, centroids and labels may be NULL.
cudaError_t components_passes(const DetectScratch &s, int W, int H, int frames, int max_components, int32_t *counts, int32_t *out_stats,
                       double *out_centroids, int32_t *labels, cudaStream_t st) {
    const int npx = W * H, words = key_words(W, H);
    const dim3 grid((npx + 255) / 256, frames), slots(max_components / 256 + 1, frames);
    merge_kernel<<<grid, 256, 0, st>>>(s.parent, W, H);
    flatten_kernel<<<grid, 256, 0, st>>>(s.parent, W, H, s.key_of);
    const cudaError_t e = cudaMemsetAsync(s.bitmap, 0, (size_t)frames * words * 4, st);
    if (e != cudaSuccess) return e;
    mark_kernel<<<grid, 256, 0, st>>>(s.parent, s.key_of, W, H, s.bitmap);
    scan_kernel<<<dim3(1, frames), kScanThreads, 0, st>>>(s.bitmap, words, s.prefix, s.n_roots, counts);
    rank_kernel<<<grid, 256, 0, st>>>(s.parent, s.key_of, W, H, s.bitmap, s.prefix, max_components, s.stats);
    stats_kernel<<<grid, 256, 0, st>>>(s.parent, s.key_of, W, H, max_components, out_centroids != nullptr, s.stats);
    write_stats_kernel<<<slots, 256, 0, st>>>(s.stats, s.n_roots, max_components, out_stats, out_centroids);
    if (labels) relabel_kernel<<<grid, 256, 0, st>>>(s.parent, s.key_of, npx, labels);
    return cudaGetLastError();
}

}  // namespace

}  // namespace cpt

using cpt::fail;

extern "C" {

// cv2.threshold(u8, ., 255, THRESH_BINARY + THRESH_OTSU): OpenCV's getThreshVal_Otsu_8u on the image's histogram
static int otsu_threshold(const unsigned int *hist, long long n) {
    const double scale = 1.0 / (double)n;
    double mu = 0;
    for (int i = 0; i < 256; ++i) mu += (double)i * (double)hist[i];
    mu *= scale;
    double mu1 = 0, q1 = 0, max_sigma = 0;
    int max_val = 0;
    const double eps = 1.1920928955078125e-07;  // FLT_EPSILON
    for (int i = 0; i < 256; ++i) {
        const double p_i = (double)hist[i] * scale;
        mu1 *= q1;
        q1 += p_i;
        const double q2 = 1.0 - q1;
        if (std::min(q1, q2) < eps || std::max(q1, q2) > 1.0 - eps) continue;
        mu1 = (mu1 + i * p_i) / q1;
        const double mu2 = (mu - q1 * mu1) / q2;
        const double sigma = q1 * q2 * (mu1 - mu2) * (mu1 - mu2);
        if (sigma > max_sigma) {
            max_sigma = sigma;
            max_val = i;
        }
    }
    return max_val;
}

// cv2.threshold on 8-bit images floors the threshold; >= 255 leaves no foreground, < 0 all of it
static int int_threshold(double threshold) {
    const double fl = std::floor(threshold);
    return fl >= 255.0 ? 255 : (fl < -1.0 ? -1 : (int)fl);
}

int cpt_detect_objects(cpt_ctx *c, const uint8_t *d_image, int width, int height, double threshold, int blur_ksize,
                       uint32_t steps, const uint8_t *d_or_mask, int max_components, int32_t *d_labels, int32_t *d_stats,
                       double *d_centroids, uint8_t *d_mask_out, int32_t *h_count, double *h_threshold_used) {
    const bool mask_only = (steps & CPT_DETECT_MASK_ONLY) != 0;
    if (!c || !d_image || !h_count) return fail(CPT_ERR_INVALID, "null argument");
    if (!mask_only && (!d_labels || !d_stats || !d_centroids)) return fail(CPT_ERR_INVALID, "null output");
    if (mask_only && !d_mask_out) return fail(CPT_ERR_INVALID, "CPT_DETECT_MASK_ONLY needs d_mask_out");
    if (width < 1 || height < 1 || (long long)width * height > (1ll << 26)) return fail(CPT_ERR_INVALID, "bad image size");
    int table = -1;
    if (blur_ksize == 3) table = 0; else if (blur_ksize == 5) table = 1; else if (blur_ksize == 7) table = 2; else if (blur_ksize == 15) table = 3;
    if (blur_ksize != 0 && table < 0) return fail(CPT_ERR_UNSUPPORTED, "GaussianBlur kernel size must be 3, 5, 7, 15 or 0 (none)");
    if (max_components < 1) return fail(CPT_ERR_INVALID, "max_components < 1");
    CUDA_TRY(cudaSetDevice(c->device));
    const int npx = width * height;
    CUDA_TRY(c->detect_scratch.ensure(cpt::detect_scratch_bytes(width, height, 1, max_components, true)));
    cpt::DetectScratch s;
    cpt::detect_scratch_bytes(width, height, 1, max_components, true, &s, c->detect_scratch);
    uint8_t *grey_a = s.grey, *grey_b = s.grey_b, *mask_a = s.mask, *mask_b = s.mask_b;
    const int grid = (npx + 255) / 256;
    cudaStream_t st = c->stream;
    // ---- grey stages: morphological open (tuple kernel), Gaussian blur
    const uint8_t *grey = d_image;
    if (steps & CPT_DETECT_OPEN_GRAY) {
        cpt::open_gray_kernel<<<grid, 256, 0, st>>>(grey, width, height, grey_a);
        grey = grey_a;
    }
    if (blur_ksize) {
        uint8_t *dst = grey == grey_a ? grey_b : grey_a;
        cpt::gauss_blur_kernel<<<grid, 256, 0, st>>>(grey, width, height, blur_ksize, table, dst);
        grey = dst;
    }
    // ---- threshold
    if (steps & CPT_DETECT_OTSU) {
        unsigned int h_hist[256];
        CUDA_TRY(cudaMemsetAsync(s.hist, 0, sizeof(h_hist), st));
        cpt::histogram_kernel<<<std::min(grid, 1024), 256, 0, st>>>(grey, npx, s.hist);
        CUDA_TRY(cudaMemcpyAsync(h_hist, s.hist, sizeof(h_hist), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        threshold = (double)otsu_threshold(h_hist, npx);
    }
    if (h_threshold_used) *h_threshold_used = threshold;
    uint8_t *mask = mask_a;
    cpt::threshold_kernel<<<grid, 256, 0, st>>>(grey, npx, int_threshold(threshold), mask);
    // ---- binary stages: dilate, (close is fused with the union-find seeding below), OR with a second mask
    if (steps & CPT_DETECT_DILATE) {
        cpt::dilate_rows_kernel<<<grid, 256, 0, st>>>(mask, width, height, mask_b);
        mask = mask_b;
    }
    const int close = (steps & CPT_DETECT_CLOSE) ? 1 : 0;
    if (d_or_mask || mask_only) {
        // materialise the closed mask so that the other mask can be OR-ed in / the mask handed out
        uint8_t *dst = mask == mask_a ? mask_b : mask_a;
        cpt::close_init_kernel<<<grid, 256, 0, st>>>(mask, width, height, close, s.parent, s.key_of);
        cpt::parent_to_mask_kernel<<<grid, 256, 0, st>>>(s.parent, npx, dst);
        mask = dst;
        if (d_or_mask) cpt::or_mask_kernel<<<grid, 256, 0, st>>>(mask, d_or_mask, npx);
        if (mask_only) {
            cpt::mask_out_kernel<<<grid, 256, 0, st>>>(mask, npx, d_mask_out);
            CUDA_TRY(cudaGetLastError());
            *h_count = 0;
            return CPT_OK;
        }
        cpt::close_init_kernel<<<grid, 256, 0, st>>>(mask, width, height, 0, s.parent, s.key_of);
    } else {
        cpt::close_init_kernel<<<grid, 256, 0, st>>>(mask, width, height, close, s.parent, s.key_of);
    }
    CUDA_TRY(cpt::components_passes(s, width, height, 1, max_components, nullptr, d_stats, d_centroids, d_labels, st));
    int n = 0;
    CUDA_TRY(cudaMemcpyAsync(&n, s.n_roots, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    if (n > max_components) return fail(CPT_ERR_INVALID, "%d components exceed max_components %d", n, max_components);
    *h_count = n + 1;  // cv2 counts the background label
    return CPT_OK;
}

int cpt_detect_objects_batch(cpt_ctx *c, const uint8_t *d_frames, int n_frames, int width, int height, double threshold, uint32_t steps,
                             int max_components, int32_t *d_counts, int32_t *d_stats, double *d_centroids, int32_t *d_labels) {
    if (!c || !d_frames || !d_counts || !d_stats) return fail(CPT_ERR_INVALID, "null argument");
    if (n_frames < 0) return fail(CPT_ERR_INVALID, "n_frames < 0");
    if (width < 1 || height < 1 || (long long)width * height > (1ll << 26)) return fail(CPT_ERR_INVALID, "bad image size");
    if (max_components < 1) return fail(CPT_ERR_INVALID, "max_components < 1");
    if (steps & ~CPT_DETECT_OPEN_GRAY) return fail(CPT_ERR_UNSUPPORTED, "cpt_detect_objects_batch: steps must be CPT_DETECT_OPEN_GRAY or 0");
    if (n_frames == 0) return CPT_OK;
    CUDA_TRY(cudaSetDevice(c->device));
    // frames per chunk: the scratch stays near kChunkBytes whatever the call's length (at least one frame)
    constexpr size_t kChunkBytes = 256u << 20;
    const size_t per_frame = cpt::detect_scratch_bytes(width, height, 1, max_components, false);
    const int chunk = (int)std::max<size_t>(1, std::min<size_t>({kChunkBytes / per_frame, (size_t)n_frames, 65535}));
    CUDA_TRY(c->detect_scratch.ensure(cpt::detect_scratch_bytes(width, height, chunk, max_components, false)));
    cpt::DetectScratch s;
    cpt::detect_scratch_bytes(width, height, chunk, max_components, false, &s, c->detect_scratch);
    const size_t npx = (size_t)width * height, rows = (size_t)max_components + 1;
    const int ithresh = int_threshold(threshold);
    cudaStream_t st = c->stream;
    for (int f0 = 0; f0 < n_frames; f0 += chunk) {
        const int nf = std::min(chunk, n_frames - f0);
        const dim3 grid((unsigned)((npx + 255) / 256), nf);
        const uint8_t *grey = d_frames + (size_t)f0 * npx;
        if (steps & CPT_DETECT_OPEN_GRAY) {
            cpt::open_gray_kernel<<<grid, 256, 0, st>>>(grey, width, height, s.grey);
            grey = s.grey;
        }
        cpt::threshold_kernel<<<grid, 256, 0, st>>>(grey, (int)npx, ithresh, s.mask);
        cpt::close_init_kernel<<<grid, 256, 0, st>>>(s.mask, width, height, 0, s.parent, s.key_of);
        CUDA_TRY(cpt::components_passes(s, width, height, nf, max_components, d_counts + f0, d_stats + (size_t)f0 * rows * 5,
                                        d_centroids ? d_centroids + (size_t)f0 * rows * 2 : nullptr,
                                        d_labels ? d_labels + (size_t)f0 * npx : nullptr, st));
    }
    CUDA_TRY(cudaGetLastError());
    return CPT_OK;
}

}  // extern "C"
