// ir_kernels.cu -- the device half of IRMotionDetector.process_frame (piclassifier/irmotiondetector.py:103-153) for
// 640x480 BGR frames: grey conversion, |oldest - current| > 12, erosion with a k x k box and the count of surviving pixels
// (for the frame difference and for the foreground mask of the host's background model).
//   bgr_to_gray_kernel   cv2.cvtColor(BGR2GRAY) in OpenCV's 8-bit fixed point
//   delta_mask_kernel    cv2.absdiff + cv2.threshold(THRESH_BINARY)
//   erode_rows_kernel    one thread per image row: a pixel survives the horizontal pass iff its k-wide window (anchor k / 2,
//                        pixels outside the image count as set) is all set -- run lengths along the row
//   erode_cols_kernel    one thread per column: the vertical pass on the row result, counting the survivors
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

}  // extern "C"
