// mog2.cuh -- OpenCV's BackgroundSubtractorMOG2 (detectShadows=False, one uint8 channel, five modes), shared by the model's
// own kernels (mog2_kernels.cu) and the IR motion detector's per-frame kernel of whole clips (ir_kernels.cu): the state
// layout, the per-pixel update and cv2's learning-rate rule.  Every product, sum and quotient is a separately rounded
// intrinsic: cv2 evaluates a*b+c as two rounded operations, and a fused multiply-add gives different background pixels.
// The library is built with one set of nvcc flags, so the rounding is pinned here rather than with -fmad=false.
#pragma once

#include <algorithm>
#include <cfloat>

#include "cptrack_internal.cuh"

namespace cpt {

constexpr int kMog2Modes = 5;

struct Mog2Consts {
    float Tb, TB, Tg, var_init, var_min, var_max;
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

// The modes of pixel x: read from the state, or an empty model (cv2's initialisation: zero modes) when fresh.
__device__ __forceinline__ void mog2_load(const float *__restrict__ state, int64_t npx, int64_t x, bool fresh, float (&w)[kMog2Modes],
                                          float (&v)[kMog2Modes], float (&m)[kMog2Modes], int &nmodes) {
    nmodes = 0;
    if (fresh) {
#pragma unroll
        for (int j = 0; j < kMog2Modes; ++j) w[j] = v[j] = m[j] = 0.f;
        return;
    }
    const float *sw = state, *sv = state + kMog2Modes * npx, *sm = state + 2 * kMog2Modes * npx;
#pragma unroll
    for (int j = 0; j < kMog2Modes; ++j) {
        w[j] = sw[j * npx + x];
        v[j] = sv[j * npx + x];
        m[j] = sm[j * npx + x];
    }
    nmodes = reinterpret_cast<const uint8_t *>(state + 3 * kMog2Modes * npx)[x];
}

__device__ __forceinline__ void mog2_store(float *__restrict__ state, int64_t npx, int64_t x, const float (&w)[kMog2Modes],
                                           const float (&v)[kMog2Modes], const float (&m)[kMog2Modes], int nmodes) {
    float *sw = state, *sv = state + kMog2Modes * npx, *sm = state + 2 * kMog2Modes * npx;
#pragma unroll
    for (int j = 0; j < kMog2Modes; ++j) {
        sw[j * npx + x] = w[j];
        sv[j * npx + x] = v[j];
        sm[j * npx + x] = m[j];
    }
    reinterpret_cast<uint8_t *>(state + 3 * kMog2Modes * npx)[x] = (uint8_t)nmodes;
}

}  // namespace cpt

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

namespace cpt {

// cv2's learning-rate rule (BackgroundSubtractorMOG2Impl::apply), the one copy of it: a frame with learningRate lr_arg
// re-initialises the model when nframes == 0 or lr_arg >= 1 ...
inline bool mog2_reinitialises(int nframes, double lr_arg) { return nframes == 0 || lr_arg >= 1; }

// ... and one apply() advances nframes and runs with alphaT = (float)lr and prune = (float)(-lr * (double)fCT), where lr is
// lr_arg, or the automatic 1 / min(2 * nframes, history) for a negative lr_arg and on the first frame after initialisation.
inline void mog2_next_rate(const cpt_mog2 &m, int &nframes, double lr_arg, float &alpha, float &prune) {
    if (mog2_reinitialises(nframes, lr_arg)) nframes = 0;
    ++nframes;
    const double lr = (lr_arg >= 0 && nframes > 1) ? lr_arg : 1.0 / (double)std::min(2 * nframes, m.history);
    alpha = (float)lr;
    prune = (float)(-lr * (double)m.complexity_reduction);
}

}  // namespace cpt
