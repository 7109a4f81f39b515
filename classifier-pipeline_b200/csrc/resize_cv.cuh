// resize_cv.cuh -- the arithmetic of cv2.resize INTER_LINEAR on fp32 (cv2 4.13, x86 build with IPP), shared by
// resize_pad_kernel (image_kernels.cu) and segment_tiles_kernel (preprocess_kernels.cu).  The rules below were measured
// against live cv2 and are held to it bit for bit by tests/test_resize_cv2.py and tests/test_resize_gpu.py (DESIGN.md §4).
//   both source sides > 1 (IPP's linear resize): coordinate (d + 0.5) * (sn / dn) - 0.5 in double, weight fp32(f - floor f),
//     index clamped with the weight zeroed at both ends in both directions, each tap pair as fma(b - a, w, a);
//   a source side of 1 (OpenCV's resizeGeneric_): coordinate fp32((d + 0.5) * (1 / (dn / sn)) - 0.5), weight f - floor f in
//     fp32; horizontally the index is clamped with the weight zeroed, vertically only the row index is clamped; each tap
//     pair as fl(a * fl(1 - w)) + fl(b * w).
// Horizontal pass first, then vertical.  Every product and sum is a rounded intrinsic so nvcc cannot contract one into a
// fused multiply-add: the one fused multiply-add is the explicit __fmaf_rn of the two-sided form.
#pragma once

#include <cuda_runtime.h>

namespace cpt {

struct ResizeTaps {
    int i0, i1;
    float w;  // weight of i1 (lerp_cv applies it in the form of the path)
};

// taps of destination index d along an axis of sn source / dn destination pixels; thin: a source side is 1;
// zero_weight: the edge rule that zeroes the weight of a clamped index (every axis but the vertical one of a thin source)
__device__ __forceinline__ ResizeTaps linear_taps(int d, int dn, int sn, bool thin, bool zero_weight) {
    const double c = __dadd_rn((double)d, 0.5);
    int i0;
    float w;
    if (thin) {
        const float f = __double2float_rn(__dadd_rn(__dmul_rn(c, __ddiv_rn(1.0, __ddiv_rn((double)dn, (double)sn))), -0.5));
        const float fl = floorf(f);
        i0 = (int)fl;
        w = __fsub_rn(f, fl);
    } else {
        const double f = __dadd_rn(__dmul_rn(c, __ddiv_rn((double)sn, (double)dn)), -0.5);
        const double fl = floor(f);
        i0 = (int)fl;
        w = __double2float_rn(__dsub_rn(f, fl));
    }
    ResizeTaps t;
    if (zero_weight) {
        if (i0 < 0) { i0 = 0; w = 0.0f; }
        if (i0 >= sn - 1) { i0 = sn - 1; w = 0.0f; }
        t.i0 = i0;
        t.i1 = min(i0 + 1, sn - 1);
    } else {
        t.i0 = min(max(i0, 0), sn - 1);
        t.i1 = min(max(i0 + 1, 0), sn - 1);
    }
    t.w = w;
    return t;
}

__device__ __forceinline__ float lerp_cv(float a, float b, float w, bool thin) {
    return thin ? __fadd_rn(__fmul_rn(a, __fsub_rn(1.0f, w)), __fmul_rn(b, w)) : __fmaf_rn(__fsub_rn(b, a), w, a);
}

}  // namespace cpt
