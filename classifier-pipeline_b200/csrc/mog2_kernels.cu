// mog2_kernels.cu -- OpenCV's BackgroundSubtractorMOG2 (cv2.createBackgroundSubtractorMOG2(detectShadows=False), one
// channel, five modes) on the device, bit for bit: the background model of track/cliptracker.py:560-609 (CVBackground) and
// of IRMotionDetector.
//   mog2_apply_kernel        apply() for T consecutive frames of one model: one thread per pixel, the pixel's modes in
//                            registers for all T frames, the state read once at the start and written once at the end
//   mog2_background_kernel   getBackgroundImage()
// The per-pixel update, the state layout and the learning-rate rule are in mog2.cuh, shared with the IR motion detector's
// kernel of whole clips (ir_kernels.cu).
#include "mog2.cuh"

namespace cpt {

constexpr int kMog2MaxT = 256;  // frames per launch: the per-frame rates travel as kernel parameters (2 KB)

struct Mog2Rates {
    float alpha[kMog2MaxT];  // alphaT = (float)learning rate
    float prune[kMog2MaxT];  // (float)(-learning rate * (double)complexity_reduction)
};

// fresh != 0: the model starts empty (cv2's initialisation: zero modes) and the state is not read.  masks may be null.
__global__ void __launch_bounds__(256) mog2_apply_kernel(float *__restrict__ state, int64_t npx, const uint8_t *__restrict__ frames,
                                                          int64_t frame_stride, int T, int fresh, Mog2Consts c, Mog2Rates r,
                                                          uint8_t *__restrict__ masks) {
    const int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= npx) return;
    float w[kMog2Modes], v[kMog2Modes], m[kMog2Modes];
    int nmodes;
    mog2_load(state, npx, x, fresh, w, v, m, nmodes);
    const uint8_t *f = frames + x;
    uint8_t next = __ldg(f);
    for (int t = 0; t < T; ++t) {
        const float data = (float)next;
        if (t + 1 < T) next = __ldg(f + (int64_t)(t + 1) * frame_stride);  // the next frame's byte is in flight during the update
        const int bg = mog2_pixel(w, v, m, nmodes, data, r.alpha[t], r.prune[t], c);
        if (masks) masks[(int64_t)t * npx + x] = bg ? 0 : 255;
    }
    mog2_store(state, npx, x, w, v, m, nmodes);
}

__global__ void __launch_bounds__(256) mog2_background_kernel(const float *__restrict__ state, int64_t npx, float TB,
                                                               uint8_t *__restrict__ out) {
    const int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= npx) return;
    const float *sw = state, *sm = state + 2 * kMog2Modes * npx;
    const int used = reinterpret_cast<const uint8_t *>(state + 3 * kMog2Modes * npx)[x];
    float meanVal = 0.f, totalWeight = 0.f;
#pragma unroll
    for (int j = 0; j < kMog2Modes; ++j) {
        if (j >= used) break;
        const float wj = sw[j * npx + x];
        meanVal = __fadd_rn(meanVal, __fmul_rn(wj, sm[j * npx + x]));
        totalWeight = __fadd_rn(totalWeight, wj);
        if (totalWeight > TB) break;
    }
    const float inv = fabsf(totalWeight) > FLT_EPSILON ? __fdiv_rn(1.f, totalWeight) : 0.f;
    const int r = __float2int_rn(__fmul_rn(meanVal, inv));
    out[x] = (uint8_t)(r < 0 ? 0 : r > 255 ? 255 : r);
}

}  // namespace cpt

using cpt::fail;

extern "C" {

cpt_mog2 *cpt_mog2_open(cpt_ctx *ctx, int width, int height, const cpt_mog2_params *p) {
    if (!ctx || !p) {
        fail(CPT_ERR_INVALID, "null argument");
        return nullptr;
    }
    if (width < 1 || height < 1 || (long long)width * height > (1ll << 28)) {
        fail(CPT_ERR_INVALID, "bad MOG2 geometry %d x %d", width, height);
        return nullptr;
    }
    if (p->detect_shadows != 0) {
        fail(CPT_ERR_INVALID, "MOG2 shadow detection is not supported (detect_shadows must be 0)");
        return nullptr;
    }
    if (p->history < 1 || !(p->complexity_reduction >= 0.f) || !(p->var_min > 0.f) || !(p->var_max >= p->var_min)) {
        fail(CPT_ERR_INVALID, "bad MOG2 parameters (history >= 1, complexity_reduction >= 0, 0 < var_min <= var_max)");
        return nullptr;
    }
    if (cudaSetDevice(ctx->device) != cudaSuccess) {
        fail(CPT_ERR_CUDA, "cudaSetDevice failed");
        return nullptr;
    }
    cpt_mog2 *m = new cpt_mog2();
    m->ctx = ctx; m->W = width; m->H = height; m->npx = (int64_t)width * height;
    m->history = p->history;
    m->complexity_reduction = p->complexity_reduction;
    m->c = cpt::Mog2Consts{(float)p->var_threshold, (float)p->background_ratio, p->var_threshold_gen, p->var_init, p->var_min, p->var_max};
    m->nframes = 0;
    const size_t bytes = cpt::mog2_state_bytes(m->npx);
    if (cudaMalloc(&m->d_state, bytes) != cudaSuccess) {
        fail(CPT_ERR_NOMEM, "MOG2 state allocation failed");
        delete m;
        return nullptr;
    }
    if (cudaMemsetAsync(m->d_state, 0, bytes, ctx->stream) != cudaSuccess) {
        fail(CPT_ERR_CUDA, "cudaMemsetAsync failed");
        cpt_mog2_close(m);
        return nullptr;
    }
    return m;
}

void cpt_mog2_close(cpt_mog2 *m) {
    if (!m) return;
    cudaSetDevice(m->ctx->device);
    cudaStreamSynchronize(m->ctx->stream);
    cudaFree(m->d_state);
    delete m;
}

int cpt_mog2_apply(cpt_mog2 *m, const uint8_t *d_frames, int n_frames, int64_t frame_stride, const double *h_learning_rates,
                   uint8_t *d_masks) {
    if (!m || (n_frames > 0 && (!d_frames || !h_learning_rates))) return fail(CPT_ERR_INVALID, "null argument");
    if (n_frames < 0) return fail(CPT_ERR_INVALID, "n_frames must be >= 0");
    if (n_frames > 1 && frame_stride < m->npx) return fail(CPT_ERR_INVALID, "frame_stride %lld is smaller than a %d x %d frame",
                                                           (long long)frame_stride, m->W, m->H);
    if (n_frames == 0) return CPT_OK;
    cpt_ctx *c = m->ctx;
    CUDA_TRY(cudaSetDevice(c->device));
    static_assert(sizeof(cpt::Mog2Rates) <= 4000, "kernel parameters");
    cpt::Mog2Rates r;
    const int blocks = (int)((m->npx + 255) / 256);
    int i = 0;
    // one launch per run of at most kMog2MaxT frames; a frame that re-initialises the model (cv2: nframes == 0 or a
    // learning rate >= 1) starts a new launch that does not read the state
    while (i < n_frames) {
        const int first = i;
        int fresh = 0, t = 0;
        while (i < n_frames && t < cpt::kMog2MaxT) {
            const double lr_arg = h_learning_rates[i];
            if (cpt::mog2_reinitialises(m->nframes, lr_arg)) {
                if (t > 0) break;
                fresh = 1;
            }
            cpt::mog2_next_rate(*m, m->nframes, lr_arg, r.alpha[t], r.prune[t]);
            ++t;
            ++i;
        }
        cpt::mog2_apply_kernel<<<blocks, 256, 0, c->stream>>>(m->d_state, m->npx, d_frames + (int64_t)first * frame_stride, frame_stride,
                                                              t, fresh, m->c, r, d_masks ? d_masks + (int64_t)first * m->npx : nullptr);
        CUDA_TRY(cudaGetLastError());
    }
    return CPT_OK;
}

int cpt_mog2_background(cpt_mog2 *m, uint8_t *d_out) {
    if (!m || !d_out) return fail(CPT_ERR_INVALID, "null argument");
    cpt_ctx *c = m->ctx;
    CUDA_TRY(cudaSetDevice(c->device));
    cpt::mog2_background_kernel<<<(int)((m->npx + 255) / 256), 256, 0, c->stream>>>(m->d_state, m->npx, m->c.TB, d_out);
    CUDA_TRY(cudaGetLastError());
    return CPT_OK;
}

int cpt_mog2_frames(const cpt_mog2 *m) {
    if (!m) return fail(CPT_ERR_INVALID, "null argument");
    return m->nframes;
}

}  // extern "C"
