// background_step.cuh -- WeightedBackground.process_frame (piclassifier/motiondetector.py:197-244) on one state
// record by one CTA; shared by background_step_kernel (aux_kernels.cu) and motion_phases (motion_kernels.cu).
#pragma once
#include "cptrack_kernels.cuh"

namespace cpt {

// `frame(p)` returns the int32 value (np.int32(frame)) of full-frame pixel p; only crop pixels are asked for.
// Every thread of the CTA must call; red_sum[32] / red_changed are shared scratch.  State layout as the
// extraction kernel's, so a record can move between the kernels.
template <typename FrameFn>
__device__ __forceinline__ void background_step(const Geometry &g, uint8_t *st_raw, FrameFn frame, const WeightTable &wt,
                                                unsigned long long *red_sum, int *red_changed) {
    StateHeader *hdr = reinterpret_cast<StateHeader *>(st_raw);
    uint16_t *B = reinterpret_cast<uint16_t *>(st_raw + sizeof(StateHeader));
    uint16_t *K = B + g.npx;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool first = hdr->initialised == 0;
    if (tid == 0) *red_changed = 0;
    __syncthreads();
    unsigned long long sum = 0;
    int changed = 0;
    for (int i = tid; i < g.ncrop; i += blockDim.x) {
        const int y = i / g.crop_w + g.edge, x = i - (y - g.edge) * g.crop_w + g.edge;
        const int p = y * g.W + x;
        const int a = frame(p);
        int b;
        if (first) {
            b = a;
            K[p] = 0;
        } else {
            b = B[p];
            const int k = K[p];
            const uint32_t e = __ldg(wt.thr + min(k, wt.max_count));
            const int thr = (int)(e & 0xffffu) - ((b < (int)(e >> 16)) ? 1 : 0);
            if (a - b >= thr) {
                K[p] = (uint16_t)(k + 1);  // keep the background, grow the weight
            } else {
                changed |= (b != a);
                b = a;
                K[p] = 0;
            }
        }
        B[p] = (uint16_t)b;
        sum += (unsigned long long)b;
    }
    for (int off = 16; off; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
    if (lane == 0) red_sum[warp] = sum;
    if (changed) *red_changed = 1;
    __syncthreads();
    if (tid == 0 && !first) hdr->frames_seen += 1;  // number of updates applied (bounds the weight counters)
    const bool any_changed = first || *red_changed;
    if (any_changed) {
        // edges: clamp the coordinate into the crop rectangle (rows, then columns: motiondetector.py:239-244)
        for (int i = tid; i < g.npx; i += blockDim.x) {
            const int y = i / g.W, x = i - y * g.W;
            const int sy = min(max(y, g.edge), g.H - 1 - g.edge), sx = min(max(x, g.edge), g.W - 1 - g.edge);
            if (sy != y || sx != x) B[i] = B[sy * g.W + sx];
        }
        if (tid == 0) {
            unsigned long long total = 0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) total += red_sum[w];
            const double mean = (double)total / (double)g.ncrop;
            hdr->average = first ? mean : rint(mean);  // np.average on init, int(round(.)) afterwards
            hdr->initialised = 1;
        }
    }
    __syncthreads();
}

}  // namespace cpt
