// ir_kernels.cu -- the device half of IRMotionDetector.process_frame (piclassifier/irmotiondetector.py:103-153) for
// 640x480 BGR frames: grey conversion, |oldest - current| > 12, erosion with a k x k box and the count of surviving pixels
// (for the frame difference and for the foreground mask of the host's background model).
//   bgr_to_gray_kernel   cv2.cvtColor(BGR2GRAY) in OpenCV's 8-bit fixed point
//   delta_mask_kernel    cv2.absdiff + cv2.threshold(THRESH_BINARY)
//   erode_rows_kernel    one thread per image row: a pixel survives the horizontal pass iff its k-wide window (anchor k / 2,
//                        pixels outside the image count as set) is all set -- run lengths along the row
//   erode_cols_kernel    one thread per column: the vertical pass on the row result, counting the survivors
// and the rectangle merging of the IR tracker's detection half for a batch of frames:
//   ir_merge_kernel      track/irtrackextractor.py merge_components on every frame's stats rows, one warp per frame
#include <algorithm>

#include "cptrack_internal.cuh"

namespace cpt {

__global__ void __launch_bounds__(256) bgr_to_gray_kernel(const uint8_t *bgr, int n, uint8_t *gray) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int b = bgr[3 * i], g = bgr[3 * i + 1], r = bgr[3 * i + 2];
    gray[i] = (uint8_t)((b * 3735 + g * 19235 + r * 9798 + (1 << 14)) >> 15);
}

__global__ void __launch_bounds__(256) delta_mask_kernel(const uint8_t *a, const uint8_t *b, int n, int threshold, uint8_t *mask) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) mask[i] = abs((int)a[i] - (int)b[i]) > threshold ? 1 : 0;
}

// window of output x: input columns x - a .. x - a + k - 1 with a = k / 2 (cv2's default anchor)
__global__ void __launch_bounds__(128) erode_rows_kernel(const uint8_t *mask, int W, int H, int k, uint8_t *out) {
    const int y = blockIdx.x * blockDim.x + threadIdx.x;
    if (y >= H) return;
    const uint8_t *row = mask + (size_t)y * W;
    uint8_t *o = out + (size_t)y * W;
    const int a = k / 2, right = k - 1 - a;
    // run = number of consecutive set pixels ending at column c (columns left of the image count as set: a long run)
    int run = k;
    for (int c = 0; c < W + right; ++c) {
        const int v = c < W ? (row[c] != 0) : 1;
        run = v ? min(run + 1, 2 * k) : 0;
        const int x = c - right;  // the output whose window ends at column c
        if (x >= 0) o[x] = run >= k ? 1 : 0;
    }
}

__global__ void __launch_bounds__(128) erode_cols_kernel(const uint8_t *rows_ok, int W, int H, int k, int *count) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    int mine = 0;
    if (x < W) {
        const int a = k / 2, below = k - 1 - a;
        int run = k;
        for (int r = 0; r < H + below; ++r) {
            const int v = r < H ? (rows_ok[(size_t)r * W + x] != 0) : 1;
            run = v ? min(run + 1, 2 * k) : 0;
            if (r - below >= 0 && run >= k) ++mine;
        }
    }
    mine = __reduce_add_sync(0xffffffffu, mine);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(count, mine);
}

// merge_components' pair test (track/irtrackextractor.py): rect a = the scanning rectangle, b = the other one.  The squared
// distance wraps in 32 bits as numpy's int32 arithmetic on the stats rows does.
__device__ __forceinline__ bool ir_rects_merge(int ax, int ay, int aw, int ah, int bx, int by, int bw, int bh, double max_gap) {
    bool within = false;
    if (bw + aw > max(bx + bw, aw + ax) - min(bx, ax)) within = bh + ah > max(by + bh, ay + ah) - min(by, ay);
    int x1 = 0, x2 = 0, y1 = 0, y2 = 0;
    if (aw + bw > max(ax + aw, bw + bx) - min(ax, bx)) {
    } else if (ax < bx) {
        x1 = ax + aw; x2 = bx;
    } else {
        x1 = bx + bw; x2 = ax;
    }
    if (ah + bh > max(ay + ah, by + bh) - min(ay, by)) {
    } else if (ay < by) {
        y1 = ay + ah; y2 = by;
    } else {
        y1 = by + bh; y2 = ay;
    }
    const unsigned dx = (unsigned)(x1 - x2), dy = (unsigned)(y1 - y2);
    const int d2 = (int)(dx * dx + dy * dy);
    return sqrt((double)d2) < max_gap || within;
}

// One warp per frame.  stats [frame][max_components + 1][5] with row 0 the background, counts = cv2's label count.  The
// list lives in the frame's output rows (merged, [max_components][5]) and in order[max_components] (the label of each list
// position; negative once deleted), so no list length is too long: every step is a warp-wide pass over the list, 32
// positions at a time.  A deletion only marks the position, which keeps the survivors in the order the Python list keeps
// them.
__global__ void __launch_bounds__(128) ir_merge_kernel(const int32_t *stats, const int32_t *counts, int n_frames, int max_components,
                                                       int min_mass, int min_size, double max_gap, int *order, int32_t *merged,
                                                       int32_t *merged_counts) {
    const int f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (f >= n_frames) return;  // whole warps
    const unsigned below = (1u << lane) - 1u;
    const int n = counts[f];
    if (n < 1 || n - 1 > max_components) {  // overflowed: the list is truncated, never merge it
        if (lane == 0) merged_counts[f] = -1;
        return;
    }
    stats += (size_t)f * ((size_t)max_components + 1) * 5;
    merged += (size_t)f * (size_t)max_components * 5;
    int *ord = order + (size_t)f * max_components;
    // filter, in label order
    int m = 0;
    for (int b = 0; b < n - 1; b += 32) {
        const int l = b + lane + 1;
        bool keep = false;
        if (l < n) {
            const int32_t *r = stats + l * 5;
            keep = r[4] > min_mass || (r[2] > min_size && r[3] > min_size);
        }
        const unsigned k = __ballot_sync(0xffffffffu, keep);
        if (keep) ord[m + __popc(k & below)] = l;
        m += __popc(k);
    }
    __syncwarp();
    // stable sort by area, descending: the rank counts larger areas and equal areas earlier in the list
    for (int b = 0; b < m; b += 32) {
        const int i = b + lane;
        if (i < m) {
            const int li = ord[i], ai = stats[li * 5 + 4];
            int rank = 0;
            for (int j = 0; j < m; ++j) {
                const int aj = stats[ord[j] * 5 + 4];
                rank += aj > ai || (aj == ai && j < i);
            }
            merged[rank * 5] = li;
        }
    }
    __syncwarp();
    for (int p = lane; p < m; p += 32) {
        const int l = merged[p * 5];
        ord[p] = l;
        for (int k = 0; k < 5; ++k) merged[p * 5 + k] = stats[l * 5 + k];
    }
    __syncwarp();
    // the scan: the current rectangle's original against every live original; merges fold in list order
    int cur = 0;
    while (cur < m) {
        const int32_t *rc = stats + ord[cur] * 5;
        const int rx = rc[0], ry = rc[1], rw = rc[2], rh = rc[3];
        int mx = merged[cur * 5], my = merged[cur * 5 + 1], mw = merged[cur * 5 + 2], mh = merged[cur * 5 + 3], ma = merged[cur * 5 + 4];
        bool any = false;
        for (int b = 0; b < m; b += 32) {
            const int p = b + lane;
            const int l = p < m ? ord[p] : 0;
            int x2 = 0, y2 = 0, w2 = 0, h2 = 0, a2 = 0;
            bool hit = false;
            if (l > 0) {
                const int32_t *r2 = stats + l * 5;
                x2 = r2[0]; y2 = r2[1]; w2 = r2[2]; h2 = r2[3]; a2 = r2[4];
                hit = x2 != rx && ir_rects_merge(rx, ry, rw, rh, x2, y2, w2, h2, max_gap);
            }
            unsigned hits = __ballot_sync(0xffffffffu, hit);
            any |= hits != 0;
            if (hit) ord[p] = -l;
            while (hits) {
                const int k = __ffs(hits) - 1;
                hits &= hits - 1;
                const int X = __shfl_sync(0xffffffffu, x2, k), Y = __shfl_sync(0xffffffffu, y2, k);
                const int W2 = __shfl_sync(0xffffffffu, w2, k), H2 = __shfl_sync(0xffffffffu, h2, k), A2 = __shfl_sync(0xffffffffu, a2, k);
                const int cur_right = mx + mw;
                mx = min(mx, X);
                my = min(my, Y);
                mw = max(cur_right, X + W2) - mx;
                mh = max(my + mh, Y + H2) - my;  // the bottom edge from the updated y, as the reference writes it
                ma += A2;
            }
        }
        if (any && lane == 0) {
            merged[cur * 5] = mx; merged[cur * 5 + 1] = my; merged[cur * 5 + 2] = mw; merged[cur * 5 + 3] = mh; merged[cur * 5 + 4] = ma;
        }
        __syncwarp();
        // a merge restarts the scan at the first live rectangle, otherwise it moves to the next live one
        const int start = any ? 0 : cur + 1;
        cur = m;
        for (int b = start; b < m; b += 32) {
            const int p = b + lane;
            const unsigned live = __ballot_sync(0xffffffffu, p < m && ord[p] > 0);
            if (live) {
                cur = b + __ffs(live) - 1;
                break;
            }
        }
    }
    // compact the live rows in place (a row only moves down, and a chunk is read before it is written)
    int out = 0;
    for (int b = 0; b < m; b += 32) {
        const int p = b + lane;
        const bool live = p < m && ord[p] > 0;
        int row[5];
        if (live)
            for (int k = 0; k < 5; ++k) row[k] = merged[p * 5 + k];
        const unsigned lv = __ballot_sync(0xffffffffu, live);
        __syncwarp();
        if (live)
            for (int k = 0; k < 5; ++k) merged[(out + __popc(lv & below)) * 5 + k] = row[k];
        out += __popc(lv);
        __syncwarp();
    }
    if (lane == 0) merged_counts[f] = out;
}

}  // namespace cpt

using cpt::fail;

struct cpt_ir_motion {
    cpt_ctx *ctx;
    int W, H, ring_frames;
    uint8_t *d_bgr, *d_ring, *d_mask, *d_rows, *d_in_mask;
    int *d_counts;   // [2]
    uint8_t *h_pin;  // pinned staging: bgr in, grey / counts out
};

extern "C" {

cpt_ir_motion *cpt_ir_motion_open(cpt_ctx *c, int width, int height, int ring_frames) {
    if (!c || width < 1 || height < 1 || ring_frames < 1 || (long long)width * height > (1ll << 24)) {
        fail(CPT_ERR_INVALID, "bad IR motion detector geometry");
        return nullptr;
    }
    if (cudaSetDevice(c->device) != cudaSuccess) {
        fail(CPT_ERR_CUDA, "cudaSetDevice failed");
        return nullptr;
    }
    cpt_ir_motion *m = new cpt_ir_motion();
    m->ctx = c; m->W = width; m->H = height; m->ring_frames = ring_frames;
    const size_t n = (size_t)width * height;
    if (cudaMalloc(&m->d_bgr, 3 * n) != cudaSuccess || cudaMalloc(&m->d_ring, n * ring_frames) != cudaSuccess ||
        cudaMalloc(&m->d_mask, n) != cudaSuccess || cudaMalloc(&m->d_rows, n) != cudaSuccess || cudaMalloc(&m->d_in_mask, n) != cudaSuccess ||
        cudaMalloc(&m->d_counts, 2 * sizeof(int)) != cudaSuccess || cudaHostAlloc((void **)&m->h_pin, 3 * n + 64, cudaHostAllocDefault) != cudaSuccess) {
        fail(CPT_ERR_NOMEM, "IR motion detector allocation failed");
        cpt_ir_motion_close(m);
        return nullptr;
    }
    cudaMemset(m->d_ring, 0, n * ring_frames);
    return m;
}

void cpt_ir_motion_close(cpt_ir_motion *m) {
    if (!m) return;
    cudaSetDevice(m->ctx->device);
    cudaStreamSynchronize(m->ctx->stream);
    cudaFree(m->d_bgr); cudaFree(m->d_ring); cudaFree(m->d_mask); cudaFree(m->d_rows); cudaFree(m->d_in_mask); cudaFree(m->d_counts);
    cudaFreeHost(m->h_pin);
    delete m;
}

int cpt_ir_motion_gray(cpt_ir_motion *m, const uint8_t *h_bgr, int slot_new, uint8_t *h_gray_out) {
    if (!m || !h_bgr) return fail(CPT_ERR_INVALID, "null argument");
    if (slot_new < 0 || slot_new >= m->ring_frames) return fail(CPT_ERR_INVALID, "ring slot out of range");
    cpt_ctx *c = m->ctx;
    CUDA_TRY(cudaSetDevice(c->device));
    const int n = m->W * m->H;
    CUDA_TRY(cudaStreamSynchronize(c->stream));  // without h_gray_out the previous frame's copy from h_pin may still run
    memcpy(m->h_pin, h_bgr, 3 * (size_t)n);
    CUDA_TRY(cudaMemcpyAsync(m->d_bgr, m->h_pin, 3 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    uint8_t *gray = m->d_ring + (size_t)slot_new * n;
    cpt::bgr_to_gray_kernel<<<(n + 255) / 256, 256, 0, c->stream>>>(m->d_bgr, n, gray);
    CUDA_TRY(cudaGetLastError());
    if (h_gray_out) {
        CUDA_TRY(cudaMemcpyAsync(m->h_pin, gray, n, cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(cudaStreamSynchronize(c->stream));
        memcpy(h_gray_out, m->h_pin, n);
    }
    return CPT_OK;
}

const uint8_t *cpt_ir_motion_ring_slot(cpt_ir_motion *m, int slot) {
    if (!m) {
        fail(CPT_ERR_INVALID, "null argument");
        return nullptr;
    }
    if (slot < 0 || slot >= m->ring_frames) {
        fail(CPT_ERR_INVALID, "ring slot out of range");
        return nullptr;
    }
    return m->d_ring + (size_t)slot * m->W * m->H;
}

int cpt_ir_motion_detect_ex(cpt_ir_motion *m, int slot_new, int slot_oldest, int threshold, int erode_k, const uint8_t *d_mask,
                            int32_t *h_diff_pixels, int32_t *h_mask_pixels) {
    if (!m || !h_diff_pixels) return fail(CPT_ERR_INVALID, "null argument");
    if (slot_new < 0 || slot_new >= m->ring_frames || slot_oldest < 0 || slot_oldest >= m->ring_frames)
        return fail(CPT_ERR_INVALID, "ring slot out of range");
    if (erode_k < 1 || erode_k > 64) return fail(CPT_ERR_INVALID, "erosion box must be 1..64 pixels");
    if (d_mask && !h_mask_pixels) return fail(CPT_ERR_INVALID, "h_mask_pixels is required with a mask");
    cpt_ctx *c = m->ctx;
    CUDA_TRY(cudaSetDevice(c->device));
    const int n = m->W * m->H;
    cudaStream_t st = c->stream;
    CUDA_TRY(cudaMemsetAsync(m->d_counts, 0, 2 * sizeof(int), st));
    cpt::delta_mask_kernel<<<(n + 255) / 256, 256, 0, st>>>(m->d_ring + (size_t)slot_oldest * n, m->d_ring + (size_t)slot_new * n, n, threshold, m->d_mask);
    cpt::erode_rows_kernel<<<(m->H + 127) / 128, 128, 0, st>>>(m->d_mask, m->W, m->H, erode_k, m->d_rows);
    cpt::erode_cols_kernel<<<(m->W + 127) / 128, 128, 0, st>>>(m->d_rows, m->W, m->H, erode_k, m->d_counts);
    if (d_mask) {
        cpt::erode_rows_kernel<<<(m->H + 127) / 128, 128, 0, st>>>(d_mask, m->W, m->H, erode_k, m->d_rows);
        cpt::erode_cols_kernel<<<(m->W + 127) / 128, 128, 0, st>>>(m->d_rows, m->W, m->H, erode_k, m->d_counts + 1);
    }
    CUDA_TRY(cudaGetLastError());
    int32_t *h_counts = reinterpret_cast<int32_t *>(m->h_pin + 3 * (size_t)n);
    CUDA_TRY(cudaMemcpyAsync(h_counts, m->d_counts, 2 * sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    *h_diff_pixels = h_counts[0];
    if (h_mask_pixels) *h_mask_pixels = d_mask ? h_counts[1] : 0;
    return CPT_OK;
}

int cpt_ir_motion_detect(cpt_ir_motion *m, int slot_new, int slot_oldest, int threshold, int erode_k, const uint8_t *h_mask,
                         int32_t *h_diff_pixels, int32_t *h_mask_pixels) {
    if (!m) return fail(CPT_ERR_INVALID, "null argument");
    if (h_mask && !h_mask_pixels) return fail(CPT_ERR_INVALID, "h_mask_pixels is required with h_mask");
    if (h_mask) {
        // the host mask goes through pinned staging into the detector's own device buffer
        const int n = m->W * m->H;
        CUDA_TRY(cudaSetDevice(m->ctx->device));
        CUDA_TRY(cudaStreamSynchronize(m->ctx->stream));  // h_pin may still be the source of an earlier copy
        memcpy(m->h_pin, h_mask, n);
        CUDA_TRY(cudaMemcpyAsync(m->d_in_mask, m->h_pin, n, cudaMemcpyHostToDevice, m->ctx->stream));
    }
    return cpt_ir_motion_detect_ex(m, slot_new, slot_oldest, threshold, erode_k, h_mask ? m->d_in_mask : nullptr, h_diff_pixels,
                                   h_mask_pixels);
}

int cpt_ir_merge_components(cpt_ctx *c, const int32_t *d_stats, const int32_t *d_counts, int n_frames, int max_components, int min_mass,
                            int min_size, double max_gap, int32_t *d_merged, int32_t *d_merged_counts) {
    if (!c || !d_stats || !d_counts || !d_merged || !d_merged_counts) return fail(CPT_ERR_INVALID, "null argument");
    if (n_frames < 0) return fail(CPT_ERR_INVALID, "n_frames < 0");
    if (max_components < 1) return fail(CPT_ERR_INVALID, "max_components < 1");
    if (n_frames == 0) return CPT_OK;
    CUDA_TRY(cudaSetDevice(c->device));
    // frames per launch: the list-order scratch stays near 64 MB whatever the call's length
    const int chunk = (int)std::max<long long>(1, std::min<long long>(n_frames, (16ll << 20) / max_components));
    CUDA_TRY(c->merge_order.ensure((size_t)chunk * max_components));
    const size_t rows = (size_t)max_components + 1;
    for (int f0 = 0; f0 < n_frames; f0 += chunk) {
        const int nf = std::min(chunk, n_frames - f0);
        cpt::ir_merge_kernel<<<(nf + 3) / 4, 128, 0, c->stream>>>(d_stats + (size_t)f0 * rows * 5, d_counts + f0, nf, max_components, min_mass,
                                                                   min_size, max_gap, c->merge_order,
                                                                   d_merged + (size_t)f0 * max_components * 5, d_merged_counts + f0);
    }
    CUDA_TRY(cudaGetLastError());
    return CPT_OK;
}

}  // extern "C"
