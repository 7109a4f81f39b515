// cptv_kernels.cu -- CPTV v2 frame decode on the device (K0 / SURVEY.md section 8f-2).  The reference reads clips with
// the third-party Rust decoder (cptv_rs_python_bindings.CptvReader, track/cliptrackextractor.py:108-129,160-165); the
// host here only inflates the gzip stream and walks the section headers (cptv/reader.py), the per-pixel work runs here:
//   cptv_unpack_kernel      one CTA per frame: int32 start value + (W*H - 1) two's-complement deltas of `bit_width`
//                           bits packed MSB first -> inclusive prefix sum along the boustrophedon scan (odd rows
//                           right to left) -> the frame's change image (int32)
//   cptv_accumulate_kernel  one thread per pixel and clip: frame t = frame t-1 + change t (uint16, modular like the
//                           host decoder's astype(uint16)); the first frame of a clip starts from zero
#include "cptrack_internal.cuh"

namespace cpt {

__device__ __forceinline__ int cptv_delta(const uint8_t *payload, int i, int w) {
    // i-th packed value (0-based) after the 4-byte start value
    if (i < 0) return (int)((uint32_t)payload[0] | ((uint32_t)payload[1] << 8) | ((uint32_t)payload[2] << 16) | ((uint32_t)payload[3] << 24));
    const long long bit = (long long)i * w;
    const uint8_t *p = payload + 4 + (bit >> 3);
    const uint32_t window = ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | (uint32_t)p[3];
    const uint32_t v = (window >> (32 - w - (int)(bit & 7))) & ((1u << w) - 1u);
    return (v & (1u << (w - 1))) ? (int)v - (1 << w) : (int)v;
}

__global__ void __launch_bounds__(256) cptv_unpack_kernel(const uint8_t *stream, const cpt_cptv_frame *table, int W, int H,
                                                          int32_t *change) {
    __shared__ int warp_sums[8];
    const cpt_cptv_frame fr = table[blockIdx.x];
    const uint8_t *payload = stream + fr.payload_offset;
    const int n = W * H, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int per = (n + 255) / 256, lo = tid * per, hi = min(lo + per, n);
    // pass 1: this thread's partial sum of its contiguous chunk of the scan order
    int sum = 0;
    for (int i = lo; i < hi; ++i) sum += cptv_delta(payload, i - 1, fr.bit_width);
    int incl = sum;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += v;
    }
    if (lane == 31) warp_sums[warp] = incl;
    __syncthreads();
    int before = 0;
    for (int q = 0; q < warp; ++q) before += warp_sums[q];
    int run = before + incl - sum;  // exclusive prefix of the chunk
    // pass 2: inclusive prefix along the snake scan, scattered to row-major order
    int32_t *out = change + (size_t)blockIdx.x * n;
    for (int i = lo; i < hi; ++i) {
        run += cptv_delta(payload, i - 1, fr.bit_width);
        const int y = i / W, x = i - y * W;
        out[y * W + ((y & 1) ? W - 1 - x : x)] = run;
    }
}

__global__ void __launch_bounds__(256) cptv_accumulate_kernel(const int32_t *change, const int32_t *clip_first, int npx,
                                                              uint16_t *frames) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x, clip = blockIdx.y;
    if (p >= npx) return;
    int cur = 0;
    for (int t = clip_first[clip]; t < clip_first[clip + 1]; ++t) {
        cur += change[(size_t)t * npx + p];
        frames[(size_t)t * npx + p] = (uint16_t)cur;
    }
}

}  // namespace cpt

using cpt::fail;

namespace cpt {
// the two decode launches on `stream`: packed frames of d_stream -> uint16 frames (scratch: n_frames * npx int32)
int cptv_decode_launch(cpt_ctx *c, const uint8_t *d_stream, const cpt_cptv_frame *d_table, int n_frames, const int32_t *d_clip_first,
                       int n_clips, uint16_t *d_frames, int32_t *scratch, cudaStream_t stream) {
    cptv_unpack_kernel<<<n_frames, 256, 0, stream>>>(d_stream, d_table, c->g.W, c->g.H, scratch);
    dim3 grid((c->g.npx + 255) / 256, n_clips);
    cptv_accumulate_kernel<<<grid, 256, 0, stream>>>(scratch, d_clip_first, c->g.npx, d_frames);
    CUDA_TRY(cudaGetLastError());
    return CPT_OK;
}
}  // namespace cpt

extern "C" {

int cpt_cptv_decode(cpt_ctx *c, const uint8_t *d_stream, const cpt_cptv_frame *d_table, int n_frames,
                    const int32_t *d_clip_first, int n_clips, uint16_t *d_frames) {
    if (!c) return fail(CPT_ERR_INVALID, "null ctx");
    if (n_frames < 0 || n_clips < 0) return fail(CPT_ERR_INVALID, "negative count");
    if (n_frames == 0 || n_clips == 0) return CPT_OK;
    if (!d_stream || !d_table || !d_clip_first || !d_frames) return fail(CPT_ERR_INVALID, "null argument");
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(c->cptv_scratch.ensure((size_t)n_frames * c->g.npx));
    return cpt::cptv_decode_launch(c, d_stream, d_table, n_frames, d_clip_first, n_clips, d_frames, c->cptv_scratch, c->stream);
}

}  // extern "C"
