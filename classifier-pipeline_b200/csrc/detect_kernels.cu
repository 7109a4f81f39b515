// detect_kernels.cu -- imageprocessing.detect_objects (ml_tools/imageprocessing.py:240-248) for ONE image of any
// size (the extraction kernel fuses the same steps for 160x120 clips in shared memory; this is the stand-alone
// primitive, also the building block for the 640x480 IR frames of SURVEY.md section 8f-4):
//   blur_threshold_kernel   cv2.GaussianBlur(u8, (5,5), 0): (sum k_i k_j U + 128) >> 8, BORDER_REFLECT_101, then
//                           cv2.threshold: U > floor(thresh)
//   close_init_kernel       cv2.morphologyEx(MORPH_CLOSE, <tuple>): the tuple becomes a 2x1 element, i.e.
//                           C[y] = M[y-1] | (M[y] & M[y-2]), C[0] = C[1] = M[0]; seeds the union-find
//   merge / flatten         8-connected label equivalence in global memory (union by smaller index, atomicMin)
//   stats_kernel            per-component bbox / area / centroid sums with atomics on the root's slot
//   order_kernel            OpenCV label numbering: rank of the component's first 2x2 block in block-raster order
//   relabel_kernel          int32 label image
#include <algorithm>
#include <climits>
#include <cmath>

#include "cptrack_internal.cuh"

namespace cpt {

namespace {

struct CompStats {
    int area, min_x, max_x, min_y, max_y, key;
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

}  // namespace

__global__ void __launch_bounds__(256) blur_threshold_kernel(const uint8_t *img, int W, int H, int ithresh, int blur, uint8_t *mask) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W * H) return;
    const int y = i / W, x = i - y * W;
    int v;
    if (blur) {
        const int k[5] = {1, 4, 6, 4, 1};
        int acc = 0;
#pragma unroll
        for (int dy = -2; dy <= 2; ++dy) {
            const uint8_t *row = img + reflect(y + dy, H) * W;
            int r = 0;
#pragma unroll
            for (int dx = -2; dx <= 2; ++dx) r += k[dx + 2] * (int)__ldg(row + reflect(x + dx, W));
            acc += k[dy + 2] * r;
        }
        v = (acc + 128) >> 8;
    } else {
        v = img[i];
    }
    mask[i] = v > ithresh ? 1 : 0;
}

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
    const int y = i / W;
    const int a = img[i], b = y >= 1 ? img[i - W] : a, c = y >= 2 ? img[i - 2 * W] : b;
    const int e1 = min(b, a), e0 = y >= 1 ? min(c, b) : e1;  // E[y], E[y-1]
    out[i] = (uint8_t)max(e0, e1);
}

__global__ void __launch_bounds__(256) threshold_kernel(const uint8_t *img, int n, int ithresh, uint8_t *mask) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) mask[i] = img[i] > ithresh ? 1 : 0;
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

__global__ void __launch_bounds__(256) close_init_kernel(const uint8_t *mask, int W, int H, int close, int *parent) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W * H) return;
    const int y = i / W;
    int c;
    if (!close) c = mask[i];
    else if (y == 0) c = mask[i];
    else if (y == 1) c = mask[i - W];
    else c = mask[i - W] | (mask[i] & mask[i - 2 * W]);
    parent[i] = c ? i : -1;
}

__global__ void __launch_bounds__(256) parent_to_mask_kernel(const int *parent, int n, uint8_t *mask) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) mask[i] = parent[i] >= 0 ? 1 : 0;
}

__global__ void __launch_bounds__(256) merge_kernel(int *parent, int W, int H) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W * H || parent[i] < 0) return;
    const int y = i / W, x = i - y * W;
    if (x > 0 && parent[i - 1] >= 0) unite(parent, i, i - 1);
    if (y > 0) {
        if (parent[i - W] >= 0) unite(parent, i, i - W);
        if (x > 0 && parent[i - W - 1] >= 0) unite(parent, i, i - W - 1);
        if (x + 1 < W && parent[i - W + 1] >= 0) unite(parent, i, i - W + 1);
    }
}

// slot 0 of `stats` is the background (label 0); component slots are claimed by their root pixel
__global__ void __launch_bounds__(256) flatten_claim_kernel(int *parent, int W, int H, int *slot_of, int *n_roots, int max_components) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W * H) return;
    slot_of[i] = -1;
    if (parent[i] < 0) return;
    const int r = find_root(parent, i);
    parent[i] = r;
    if (r == i) {
        const int s = atomicAdd(n_roots, 1);
        slot_of[i] = s < max_components ? s + 1 : -2;  // -2: overflow
    }
}

__global__ void __launch_bounds__(256) stats_kernel(const int *parent, const int *slot_of, int W, int H, CompStats *stats) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W * H) return;
    const int y = i / W, x = i - y * W;
    int slot = 0;
    if (parent[i] >= 0) {
        slot = slot_of[parent[i]];
        if (slot < 0) return;
    }
    CompStats *s = stats + slot;
    atomicAdd(&s->area, 1);
    atomicMin(&s->min_x, x);
    atomicMax(&s->max_x, x);
    atomicMin(&s->min_y, y);
    atomicMax(&s->max_y, y);
    atomicMin(&s->key, (y >> 1) * ((W + 1) >> 1) + (x >> 1));
    atomicAdd(&s->sum_x, (unsigned long long)x);
    atomicAdd(&s->sum_y, (unsigned long long)y);
}

__global__ void stats_reset_kernel(CompStats *stats, int n, int *n_roots) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *n_roots = 0;
    if (i >= n) return;
    CompStats s;
    s.area = 0; s.min_x = INT_MAX; s.max_x = -1; s.min_y = INT_MAX; s.max_y = -1; s.key = INT_MAX; s.sum_x = 0; s.sum_y = 0;
    stats[i] = s;
}

// rank of every component slot (1..n) by key -> label number; writes the cv2-shaped outputs
__global__ void __launch_bounds__(256) order_kernel(const CompStats *stats, int n, int *label_of_slot, int32_t *out_stats, double *out_centroids) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;  // slot 0..n
    if (s > n) return;
    int label = 0;
    if (s > 0) {
        const int key = stats[s].key;
        int rank = 0;
        for (int q = 1; q <= n; ++q) rank += stats[q].key < key;
        label = rank + 1;
    }
    label_of_slot[s] = label;
    const CompStats c = stats[s];
    int32_t *o = out_stats + label * 5;
    if (c.area > 0) {
        o[0] = c.min_x; o[1] = c.min_y; o[2] = c.max_x - c.min_x + 1; o[3] = c.max_y - c.min_y + 1; o[4] = c.area;
        out_centroids[label * 2] = (double)c.sum_x / (double)c.area;
        out_centroids[label * 2 + 1] = (double)c.sum_y / (double)c.area;
    } else {  // only the background of an all-foreground image: cv2 reports an empty box and a NaN centroid
        o[0] = INT_MAX; o[1] = INT_MAX; o[2] = 0; o[3] = 0; o[4] = 0;
        out_centroids[label * 2] = nan("");
        out_centroids[label * 2 + 1] = nan("");
    }
}

__global__ void __launch_bounds__(256) relabel_kernel(const int *parent, const int *slot_of, const int *label_of_slot, int n, int32_t *labels) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    labels[i] = parent[i] < 0 ? 0 : label_of_slot[slot_of[parent[i]]];
}

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

int cpt_detect_objects_ex(cpt_ctx *c, const uint8_t *d_image, int width, int height, double threshold, int blur_ksize,
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
    // scratch: grey A | grey B | mask A | mask B | parent int | slot_of int | stats | label_of_slot | n_roots | histogram
    const size_t img_bytes = ((size_t)npx + 255) & ~(size_t)255;
    const size_t off_parent = 4 * img_bytes;
    const size_t off_slot = off_parent + (size_t)npx * 4;
    const size_t off_stats = off_slot + (size_t)npx * 4;
    const size_t off_label = off_stats + (size_t)(max_components + 1) * sizeof(cpt::CompStats);
    const size_t off_count = off_label + (size_t)(max_components + 1) * 4;
    const size_t off_hist = off_count + 256;
    const size_t total = off_hist + 256 * sizeof(unsigned int);
    CUDA_TRY(c->detect_scratch.ensure(total));
    uint8_t *base = c->detect_scratch;
    uint8_t *grey_a = base, *grey_b = base + img_bytes, *mask_a = base + 2 * img_bytes, *mask_b = base + 3 * img_bytes;
    int *parent = (int *)(base + off_parent), *slot_of = (int *)(base + off_slot);
    cpt::CompStats *stats = (cpt::CompStats *)(base + off_stats);
    int *label_of_slot = (int *)(base + off_label), *n_roots = (int *)(base + off_count);
    unsigned int *hist = (unsigned int *)(base + off_hist);
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
    // ---- threshold (cv2.threshold on 8-bit images floors the threshold; >= 255 leaves no foreground, < 0 all of it)
    if (steps & CPT_DETECT_OTSU) {
        unsigned int h_hist[256];
        CUDA_TRY(cudaMemsetAsync(hist, 0, sizeof(h_hist), st));
        cpt::histogram_kernel<<<std::min(grid, 1024), 256, 0, st>>>(grey, npx, hist);
        CUDA_TRY(cudaMemcpyAsync(h_hist, hist, sizeof(h_hist), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        threshold = (double)otsu_threshold(h_hist, npx);
    }
    if (h_threshold_used) *h_threshold_used = threshold;
    const double fl = std::floor(threshold);
    const int ithresh = fl >= 255.0 ? 255 : (fl < -1.0 ? -1 : (int)fl);
    uint8_t *mask = mask_a;
    cpt::threshold_kernel<<<grid, 256, 0, st>>>(grey, npx, ithresh, mask);
    // ---- binary stages: dilate, (close is fused with the union-find seeding below), OR with a second mask
    if (steps & CPT_DETECT_DILATE) {
        cpt::dilate_rows_kernel<<<grid, 256, 0, st>>>(mask, width, height, mask_b);
        mask = mask_b;
    }
    const int close = (steps & CPT_DETECT_CLOSE) ? 1 : 0;
    if (d_or_mask || mask_only) {
        // materialise the closed mask so that the other mask can be OR-ed in / the mask handed out
        uint8_t *dst = mask == mask_a ? mask_b : mask_a;
        cpt::close_init_kernel<<<grid, 256, 0, st>>>(mask, width, height, close, parent);
        cpt::parent_to_mask_kernel<<<grid, 256, 0, st>>>(parent, npx, dst);
        mask = dst;
        if (d_or_mask) cpt::or_mask_kernel<<<grid, 256, 0, st>>>(mask, d_or_mask, npx);
        if (mask_only) {
            cpt::mask_out_kernel<<<grid, 256, 0, st>>>(mask, npx, d_mask_out);
            CUDA_TRY(cudaGetLastError());
            *h_count = 0;
            return CPT_OK;
        }
        cpt::close_init_kernel<<<grid, 256, 0, st>>>(mask, width, height, 0, parent);
    } else {
        cpt::close_init_kernel<<<grid, 256, 0, st>>>(mask, width, height, close, parent);
    }
    cpt::merge_kernel<<<grid, 256, 0, st>>>(parent, width, height);
    cpt::stats_reset_kernel<<<(max_components + 256) / 256, 256, 0, st>>>(stats, max_components + 1, n_roots);
    cpt::flatten_claim_kernel<<<grid, 256, 0, st>>>(parent, width, height, slot_of, n_roots, max_components);
    cpt::stats_kernel<<<grid, 256, 0, st>>>(parent, slot_of, width, height, stats);
    int n = 0;
    CUDA_TRY(cudaMemcpyAsync(&n, n_roots, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (n > max_components) return fail(CPT_ERR_INVALID, "%d components exceed max_components %d", n, max_components);
    cpt::order_kernel<<<(n + 256) / 256, 256, 0, st>>>(stats, n, label_of_slot, d_stats, d_centroids);
    cpt::relabel_kernel<<<grid, 256, 0, st>>>(parent, slot_of, label_of_slot, npx, d_labels);
    CUDA_TRY(cudaGetLastError());
    *h_count = n + 1;  // cv2 counts the background label
    return CPT_OK;
}

int cpt_detect_objects_u8(cpt_ctx *c, const uint8_t *d_image, int width, int height, double threshold, int blur_ksize,
                          int close, int max_components, int32_t *d_labels, int32_t *d_stats, double *d_centroids,
                          int32_t *h_count) {
    return cpt_detect_objects_ex(c, d_image, width, height, threshold, blur_ksize, close ? CPT_DETECT_CLOSE : 0u, nullptr, max_components,
                                 d_labels, d_stats, d_centroids, nullptr, h_count, nullptr);
}

}  // extern "C"
