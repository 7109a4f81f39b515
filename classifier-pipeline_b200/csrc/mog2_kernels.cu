// mog2_kernels.cu -- OpenCV's BackgroundSubtractorMOG2 (cv2.createBackgroundSubtractorMOG2(detectShadows=False), one
// channel, five modes) on the device, bit for bit: the background model of track/cliptracker.py:560-609 (CVBackground) and
// of IRMotionDetector.
//   mog2_apply_kernel        apply() for T consecutive frames of one model: one thread per pixel, the pixel's modes in
//                            registers for all T frames, the state read once at the start and written once at the end
//   mog2_background_kernel   getBackgroundImage()
// Every product, sum and quotient is a separately rounded intrinsic: cv2 evaluates a*b+c as two rounded operations, and a
// fused multiply-add gives different background pixels.  The library is built with one set of nvcc flags, so the
// rounding is pinned here rather than with -fmad=false.
#include <algorithm>
#include <cfloat>

#include "cptrack_internal.cuh"

namespace cpt {

constexpr int kMog2Modes = 5;
constexpr int kMog2MaxT = 256;  // frames per launch: the per-frame rates travel as kernel parameters (2 KB)

struct Mog2Consts {
    float Tb, TB, Tg, var_init, var_min, var_max;
};
struct Mog2Rates {
    float alpha[kMog2MaxT];  // alphaT = (float)learning rate
    float prune[kMog2MaxT];  // (float)(-learning rate * (double)complexity_reduction)
};

// State in HBM, structure of arrays over the npx pixels: float weight[5][npx], var[5][npx], mean[5][npx], then
// uint8 used[npx] (the mode count).
__host__ __device__ inline size_t mog2_state_bytes(int64_t npx) { return (size_t)npx * (3 * kMog2Modes * sizeof(float) + 1); }

template <int N>
__device__ __forceinline__ void swap_mode(float (&w)[N], float (&v)[N], float (&m)[N], int i) {
    float t = w[i]; w[i] = w[i - 1]; w[i - 1] = t;
    t = v[i]; v[i] = v[i - 1]; v[i - 1] = t;
    t = m[i]; m[i] = m[i - 1]; m[i - 1] = t;
}

// One apply() of one pixel.  Indices into w / v / m are compile-time constants after unrolling (a runtime index would put
// the arrays in local memory): the loops of the scalar algorithm become predicated chains with the same break conditions.
// Returns 1 when the pixel is background.
__device__ __forceinline__ int mog2_pixel(float (&w)[kMog2Modes], float (&v)[kMog2Modes], float (&m)[kMog2Modes], int &nmodes,
                                          float data, float alphaT, float prune, const Mog2Consts &c) {
    const float alpha1 = __fsub_rn(1.f, alphaT);
    int background = 0, fits = 0;
    float totalWeight = 0.f;
#pragma unroll
    for (int mode = 0; mode < kMog2Modes; ++mode) {
        if (mode >= nmodes) break;  // nmodes shrinks inside the loop (a pruned mode stays in place with weight 0)
        float weight = __fadd_rn(__fmul_rn(alpha1, w[mode]), prune);
        int swap_count = 0;
        if (!fits) {
            const float var = v[mode];
            const float d = __fsub_rn(m[mode], data);
            const float dist2 = __fmul_rn(d, d);
            if (totalWeight < c.TB && dist2 < __fmul_rn(c.Tb, var)) background = 1;
            if (dist2 < __fmul_rn(c.Tg, var)) {
                fits = 1;
                weight = __fadd_rn(weight, alphaT);
                const float k = __fdiv_rn(alphaT, weight);
                m[mode] = __fsub_rn(m[mode], __fmul_rn(k, d));
                float varnew = __fadd_rn(var, __fmul_rn(k, __fsub_rn(dist2, var)));
                varnew = varnew > c.var_min ? varnew : c.var_min;
                varnew = varnew < c.var_max ? varnew : c.var_max;
                v[mode] = varnew;
                // bubble the mode up while its new weight is >= the one above (equal weights swap)
                bool moving = true;
#pragma unroll
                for (int i = mode; i > 0; --i) {
                    moving = moving && !(weight < w[i - 1]);
                    if (moving) {
                        swap_mode(w, v, m, i);
                        ++swap_count;
                    }
                }
            }
        }
        if (weight < -prune) {
            weight = 0.f;
            --nmodes;
        }
#pragma unroll
        for (int j = 0; j <= mode; ++j)
            if (j == mode - swap_count) w[j] = weight;
        totalWeight = __fadd_rn(totalWeight, weight);
    }
    // cv2 4.x renormalises with 0 when every mode it visited was pruned (a learning rate near 1 prunes all modes before the
    // fitting one); 1 / totalWeight would turn the remaining weights into NaN
    const float invWeight = fabsf(totalWeight) > FLT_EPSILON ? __fdiv_rn(1.f, totalWeight) : 0.f;
#pragma unroll
    for (int j = 0; j < kMog2Modes; ++j)
        if (j < nmodes) w[j] = __fmul_rn(w[j], invWeight);
    if (!fits && alphaT > 0.f) {
        const int mode = nmodes == kMog2Modes ? kMog2Modes - 1 : nmodes++;
#pragma unroll
        for (int j = 0; j < kMog2Modes; ++j) {
            if (nmodes == 1) {
                if (j == mode) w[j] = 1.f;
            } else if (j == mode) {
                w[j] = alphaT;
            } else if (j < nmodes - 1) {
                w[j] = __fmul_rn(w[j], alpha1);
            }
            if (j == mode) {
                m[j] = data;
                v[j] = c.var_init;
            }
        }
        bool moving = true;
#pragma unroll
        for (int i = kMog2Modes - 1; i > 0; --i) {
            if (i < nmodes) {
                moving = moving && !(alphaT < w[i - 1]);
                if (moving) swap_mode(w, v, m, i);
            }
        }
    }
    return background;
}

// fresh != 0: the model starts empty (cv2's initialisation: zero modes) and the state is not read.  masks may be null.
__global__ void __launch_bounds__(256) mog2_apply_kernel(float *__restrict__ state, int64_t npx, const uint8_t *__restrict__ frames,
                                                          int64_t frame_stride, int T, int fresh, Mog2Consts c, Mog2Rates r,
                                                          uint8_t *__restrict__ masks) {
    const int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= npx) return;
    float *sw = state, *sv = state + kMog2Modes * npx, *sm = state + 2 * kMog2Modes * npx;
    uint8_t *used = reinterpret_cast<uint8_t *>(state + 3 * kMog2Modes * npx);
    float w[kMog2Modes], v[kMog2Modes], m[kMog2Modes];
    int nmodes = 0;
    if (fresh) {
#pragma unroll
        for (int j = 0; j < kMog2Modes; ++j) w[j] = v[j] = m[j] = 0.f;
    } else {
#pragma unroll
        for (int j = 0; j < kMog2Modes; ++j) {
            w[j] = sw[j * npx + x];
            v[j] = sv[j * npx + x];
            m[j] = sm[j * npx + x];
        }
        nmodes = used[x];
    }
    const uint8_t *f = frames + x;
    uint8_t next = __ldg(f);
    for (int t = 0; t < T; ++t) {
        const float data = (float)next;
        if (t + 1 < T) next = __ldg(f + (int64_t)(t + 1) * frame_stride);  // the next frame's byte is in flight during the update
        const int bg = mog2_pixel(w, v, m, nmodes, data, r.alpha[t], r.prune[t], c);
        if (masks) masks[(int64_t)t * npx + x] = bg ? 0 : 255;
    }
#pragma unroll
    for (int j = 0; j < kMog2Modes; ++j) {
        sw[j * npx + x] = w[j];
        sv[j * npx + x] = v[j];
        sm[j * npx + x] = m[j];
    }
    used[x] = (uint8_t)nmodes;
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

struct cpt_mog2 {
    cpt_ctx *ctx;
    int W, H;
    int64_t npx;
    int history;
    float complexity_reduction;
    cpt::Mog2Consts c;
    int nframes;     // cv2's nframes: frames since the last initialisation
    float *d_state;  // mog2_state_bytes(npx)
};

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
            if (m->nframes == 0 || lr_arg >= 1) {
                if (t > 0) break;
                fresh = 1;
                m->nframes = 0;
            }
            ++m->nframes;
            const double lr = (lr_arg >= 0 && m->nframes > 1) ? lr_arg : 1.0 / (double)std::min(2 * m->nframes, m->history);
            r.alpha[t] = (float)lr;
            r.prune[t] = (float)(-lr * (double)m->complexity_reduction);
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
