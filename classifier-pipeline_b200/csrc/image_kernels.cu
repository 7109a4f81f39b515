// image_kernels.cu -- the ml_tools/imageprocessing.py helpers as stand-alone device primitives (the
// reference calls them on single numpy arrays; the extraction and preprocessing kernels fuse the same
// arithmetic for batches):
//   minmax_kernel / normalize_kernel   normalize()          imageprocessing.py:151-169
//   resize_pad_kernel                  resize_and_pad()     imageprocessing.py:11-70 (cv2.resize linear / nearest)
#include <algorithm>
#include <cfloat>

#include "cptrack_internal.cuh"

namespace cpt {

// ------------------------------------------------------------------------------------------------
// min / max of an fp32 array -> out[0], out[1] (initialised by the caller to +FLT_MAX / -FLT_MAX)
__global__ void __launch_bounds__(256) minmax_kernel(const float *in, long long n, float *out) {
    float mn = FLT_MAX, mx = -FLT_MAX;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float v = __ldg(in + i);
        mn = fminf(mn, v);
        mx = fmaxf(mx, v);
    }
    for (int off = 16; off; off >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, off));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
    }
    if ((threadIdx.x & 31) == 0) {
        // ordered-int trick: floats with the sign bit clear order as ints, floats with it set order reversed as unsigned.
        // The branch tests the sign bit, not v >= 0: -0.0 compares equal to 0 but its bits are INT_MIN as an int.
        int *o = reinterpret_cast<int *>(out);
        if (__float_as_int(mn) >= 0) atomicMin(o, __float_as_int(mn)); else atomicMax(reinterpret_cast<unsigned *>(o), __float_as_uint(mn));
        if (__float_as_int(mx) >= 0) atomicMax(o + 1, __float_as_int(mx)); else atomicMin(reinterpret_cast<unsigned *>(o + 1), __float_as_uint(mx));
    }
}

// normalize(): out = new_max * (float32(data) - min) / (max - min); the arithmetic type follows numpy's
// promotion of the operands (decided on the host): fp32 throughout, or fp64 on the fp32-rounded data.
// min == max: zeros when max == 0, else data / max.
__global__ void __launch_bounds__(256) normalize_kernel(const float *in, long long n, double mn, double mx, double new_max,
                                                        int use_f64, float *out32, double *out64) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float v = __ldg(in + i);
    if (use_f64) {
        double r;
        if (mx == mn) r = (mx == 0.0) ? 0.0 : (double)v / mx;
        else r = new_max * ((double)v - mn) / (mx - mn);
        out64[i] = r;
    } else {
        const float fmn = (float)mn, fmx = (float)mx;
        float r;
        if (fmx == fmn) r = (fmx == 0.0f) ? 0.0f : __fdiv_rn(v, fmx);
        else r = __fdiv_rn(__fmul_rn((float)new_max, __fsub_rn(v, fmn)), __fsub_rn(fmx, fmn));
        out32[i] = r;
    }
}

// ------------------------------------------------------------------------------------------------
// cv2.resize of an fp32 image (sw x sh) to (fw x fh), pasted at (ox, oy) into a (dw x dh) image filled with pad.
// interpolation 1 = INTER_LINEAR (half-pixel centres, fp32 taps, horizontal then vertical, each pair as
// fma(b - a, w, a) -- the form the x86 OpenCV 4.x build uses), 0 = INTER_NEAREST (floor(dst * src/dst)).
__global__ void __launch_bounds__(256) resize_pad_kernel(const float *src, int sw, int sh, int fw, int fh, int ox, int oy,
                                                         int dw, int dh, float pad, int interpolation, float *dst) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= dw * dh) return;
    const int y = i / dw, x = i - y * dw;
    const int dx = x - ox, dy = y - oy;
    float v = pad;
    if (dx >= 0 && dx < fw && dy >= 0 && dy < fh) {
        if (interpolation == 0) {
            const int sx = min((int)floor((double)dx * (1.0 / ((double)fw / (double)sw))), sw - 1);
            const int sy = min((int)floor((double)dy * (1.0 / ((double)fh / (double)sh))), sh - 1);
            v = __ldg(src + sy * sw + sx);
        } else {
            int x0, x1, y0, y1;
            float wx, wy;
            {
                const double fx = ((double)dx + 0.5) * (1.0 / ((double)fw / (double)sw)) - 0.5;
                if (sh == 1 && sw > 1) { const float ff = (float)fx, fl = floorf(ff); x0 = (int)fl; wx = __fsub_rn(ff, fl); }
                else { const double fl = floor(fx); x0 = (int)fl; wx = (float)(fx - fl); }
                if (x0 < 0) { x0 = 0; wx = 0.f; }
                if (x0 >= sw - 1) { x0 = sw - 1; wx = 0.f; }
                x1 = min(x0 + 1, sw - 1);
            }
            {
                const double fy = ((double)dy + 0.5) * (1.0 / ((double)fh / (double)sh)) - 0.5;
                if (sw == 1 && sh > 1) { const float ff = (float)fy, fl = floorf(ff); y0 = (int)fl; wy = __fsub_rn(ff, fl); }
                else { const double fl = floor(fy); y0 = (int)fl; wy = (float)(fy - fl); }
                if (y0 < 0) { y0 = 0; wy = 0.f; }
                if (y0 >= sh - 1) { y0 = sh - 1; wy = 0.f; }
                y1 = min(y0 + 1, sh - 1);
            }
            const float a = __ldg(src + y0 * sw + x0), b = __ldg(src + y0 * sw + x1);
            const float c = __ldg(src + y1 * sw + x0), d = __ldg(src + y1 * sw + x1);
            const float r0 = __fmaf_rn(__fsub_rn(b, a), wx, a), r1 = __fmaf_rn(__fsub_rn(d, c), wx, c);
            v = __fmaf_rn(__fsub_rn(r1, r0), wy, r0);
        }
    }
    dst[i] = v;
}

}  // namespace cpt

using cpt::fail;

extern "C" {

int cpt_minmax_f32(cpt_ctx *c, const float *d_in, int64_t n, float *d_out2) {
    if (!c || !d_in || !d_out2) return fail(CPT_ERR_INVALID, "null argument");
    if (n <= 0) return fail(CPT_ERR_INVALID, "empty array");
    CUDA_TRY(cudaSetDevice(c->device));
    const float init[2] = {FLT_MAX, -FLT_MAX};
    CUDA_TRY(cudaMemcpyAsync(d_out2, init, sizeof(init), cudaMemcpyHostToDevice, c->stream));
    const int grid = (int)std::min<long long>((n + 255) / 256, 4 * (long long)c->num_sms);
    cpt::minmax_kernel<<<grid, 256, 0, c->stream>>>(d_in, n, d_out2);
    CUDA_TRY(cudaGetLastError());
    return CPT_OK;
}

int cpt_normalize_f32(cpt_ctx *c, const float *d_in, int64_t n, double min, double max, double new_max, int use_f64,
                      void *d_out) {
    if (!c || !d_in || !d_out) return fail(CPT_ERR_INVALID, "null argument");
    if (n < 0) return fail(CPT_ERR_INVALID, "negative size");
    if (n == 0) return CPT_OK;
    CUDA_TRY(cudaSetDevice(c->device));
    cpt::normalize_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(d_in, n, min, max, new_max, use_f64,
                                                                              (float *)d_out, (double *)d_out);
    CUDA_TRY(cudaGetLastError());
    return CPT_OK;
}

int cpt_resize_pad_f32(cpt_ctx *c, const float *d_src, int src_w, int src_h, int resized_w, int resized_h, int offset_x,
                       int offset_y, int out_w, int out_h, float pad, int interpolation, float *d_out) {
    if (!c || !d_src || !d_out) return fail(CPT_ERR_INVALID, "null argument");
    if (src_w < 1 || src_h < 1 || resized_w < 1 || resized_h < 1 || out_w < 1 || out_h < 1)
        return fail(CPT_ERR_INVALID, "empty image");
    if (interpolation != 0 && interpolation != 1) return fail(CPT_ERR_UNSUPPORTED, "interpolation must be 0 (nearest) or 1 (linear)");
    CUDA_TRY(cudaSetDevice(c->device));
    const int n = out_w * out_h;
    cpt::resize_pad_kernel<<<(n + 255) / 256, 256, 0, c->stream>>>(d_src, src_w, src_h, resized_w, resized_h, offset_x, offset_y,
                                                                   out_w, out_h, pad, interpolation, d_out);
    CUDA_TRY(cudaGetLastError());
    return CPT_OK;
}

}  // extern "C"
