// median.cuh -- np.median of the uint16 values of a rectangle of a frame staged in shared memory, by one CTA of
// 256 threads (K8 ClipStats median, clip.py:474-487; the per-frame / per-crop medians of
// Interpreter.preprocess_segments, interpreter.py:389-399).  Returned as the SUM of the two middle order
// statistics (== 2 * median), so the result stays an integer.
//   narrow rectangles (max - min < 2048, i.e. every real thermal frame): one pass into a 2048-bin histogram of
//     (value - min) -- the contention of a coarse radix pass on a single bucket is what made the two-pass version slow --
//     then a block-wide prefix scan locates both ranks;
//   wide rectangles: two 256-bin radix passes (high byte, then low byte within the selected bucket).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace cpt {

constexpr int kMedianBins = 2048;
constexpr int kMedianThreads = 256;

// bins: kMedianBins uint32 of shared scratch; red: 80 ints of shared scratch.  Every thread of the CTA must call; the CTA
// has kThreads threads (64..256; a crop of a few hundred pixels wants fewer than a whole frame).  px may point to shared or
// global memory.
template <int kThreads = kMedianThreads>
__device__ inline int rect_median_sum(const uint16_t *px, int W, int x0, int y0, int w, int h, uint32_t *bins, int *red) {
    static_assert(kThreads % 32 == 0 && kThreads >= 64 && kThreads <= 256 && kMedianBins % kThreads == 0, "CTA size");
    constexpr int kWarps = kThreads / 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, n = w * h;
    // ---- range of the rectangle
    int mn = 65535, mx = 0;
    for (int i = tid; i < n; i += kThreads) {
        const int yy = i / w, xx = i - yy * w;
        const int v = px[(y0 + yy) * W + x0 + xx];
        mn = min(mn, v);
        mx = max(mx, v);
    }
    mn = __reduce_min_sync(0xffffffffu, mn);
    mx = __reduce_max_sync(0xffffffffu, mx);
    __syncthreads();  // scratch may still be read by a previous call
    if (lane == 0) { red[warp] = mn; red[8 + warp] = mx; }
    __syncthreads();
    mn = red[lane % kWarps];
    mx = red[8 + lane % kWarps];
    mn = __reduce_min_sync(0xffffffffu, mn);
    mx = __reduce_max_sync(0xffffffffu, mx);
    const int r_lo = (n - 1) / 2, r_hi = n / 2;
    if (mx - mn < kMedianBins) {
        for (int i = tid; i < kMedianBins; i += kThreads) bins[i] = 0;
        __syncthreads();
        for (int i = tid; i < n; i += kThreads) {
            const int yy = i / w, xx = i - yy * w;
            atomicAdd(&bins[px[(y0 + yy) * W + x0 + xx] - mn], 1u);
        }
        __syncthreads();
        // thread t owns bins [kPer t, kPer (t + 1)): block-wide inclusive scan of the per-thread counts
        constexpr int kPer = kMedianBins / kThreads;
        uint32_t c[kPer], loc = 0;
#pragma unroll
        for (int j = 0; j < kPer; ++j) { c[j] = bins[tid * kPer + j]; loc += c[j]; }
        uint32_t incl = loc;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, incl, off);
            if (lane >= off) incl += v;
        }
        if (lane == 31) red[16 + warp] = (int)incl;
        __syncthreads();
        uint32_t before = 0;
        for (int q = 0; q < warp; ++q) before += (uint32_t)red[16 + q];
        incl += before;
        uint32_t excl = incl - loc;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const uint32_t rank = (uint32_t)(k == 0 ? r_lo : r_hi);
            if (rank >= excl && rank < incl) {
                uint32_t acc = excl;
                int bin = 0;
#pragma unroll
                for (int j = 0; j < kPer; ++j) {
                    if (rank >= acc && rank < acc + c[j]) bin = j;
                    acc += c[j];
                }
                red[32 + k] = mn + tid * kPer + bin;
            }
        }
        __syncthreads();
        return red[32] + red[33];
    }
    // ---- wide range: radix select on the high byte, then on the low byte inside the selected bucket(s)
    uint32_t *h0 = bins, *h1 = bins + 256;
    for (int i = tid; i < 512; i += kThreads) bins[i] = 0;
    __syncthreads();
    for (int i = tid; i < n; i += kThreads) {
        const int yy = i / w, xx = i - yy * w;
        atomicAdd(&h0[px[(y0 + yy) * W + x0 + xx] >> 8], 1u);
    }
    __syncthreads();
    if (tid < 2) {
        const int rank = tid == 0 ? r_lo : r_hi;
        int acc = 0, b = 0;
        for (; b < 255; ++b) {
            const int cnt = (int)h0[b];
            if (rank < acc + cnt) break;
            acc += cnt;
        }
        red[40 + tid] = b;           // bucket
        red[42 + tid] = rank - acc;  // rank inside the bucket
    }
    __syncthreads();
    const int b_lo = red[40], b_hi = red[41];
    for (int i = tid; i < 512; i += kThreads) bins[i] = 0;
    __syncthreads();
    for (int i = tid; i < n; i += kThreads) {
        const int yy = i / w, xx = i - yy * w;
        const int v = px[(y0 + yy) * W + x0 + xx], hb = v >> 8;
        if (hb == b_lo) atomicAdd(&h0[v & 0xff], 1u);
        if (hb == b_hi) atomicAdd(&h1[v & 0xff], 1u);
    }
    __syncthreads();
    if (tid < 2) {
        const uint32_t *hh = tid == 0 ? h0 : h1;
        const int rank = red[42 + tid];
        int acc = 0, b = 0;
        for (; b < 255; ++b) {
            const int cnt = (int)hh[b];
            if (rank < acc + cnt) break;
            acc += cnt;
        }
        red[32 + tid] = (red[40 + tid] << 8) | b;
    }
    __syncthreads();
    return red[32] + red[33];
}

}  // namespace cpt
