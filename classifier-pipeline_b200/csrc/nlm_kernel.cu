// nlm_kernel.cu -- cv2.fastNlMeansDenoising(uint8, None) (K3 of SURVEY.md section 8a / Appendix B; the call site is
// track/cliptracker.py:116-117, active when TrackingConfig.denoise is set): h = 3, 7x7 template, 21x21 search.
// OpenCV's integer algorithm, bit for bit: for every pixel p and search offset o in [-10, 10]^2
//     dist = sum over the 7x7 template of (ext[p + o + t] - ext[p + t])^2        (ext: BORDER_REFLECT_101 by 13)
//     w = table[dist >> 6],  est += w * ext[p + o],  wsum += w;      out = (est + wsum / 2) / wsum
// with table[a] = rint(19096 * exp(-(a * 64 / 49) / 9)), zero below 0.001 * 19096 -- only a <= 47 is non-zero.
// Compute bound by design (441 offsets x 49 template pixels per output pixel).  nlm_quads_kernel, the kernel every
// image takes: a thread owns 4 adjacent columns x 10 rows, its 40 estimates and weight sums live in registers for
// all 441 offsets; per offset it walks down 10 + 6 rows of its columns -- per row three words of the image and of the
// shifted image (funnel shifts bring the shifted bytes into line), |a - b| on four bytes at a time, the squares summed
// by dp4a into the four 7-wide horizontal sums, a 7-deep register ring for the vertical running sum -- and then looks
// up the weight of each of its 10 x 4 pixels: about 27 instructions per pixel and offset, no barrier inside the search.
#include <algorithm>
#include <cmath>

#include "cptrack_internal.cuh"

namespace cpt {

constexpr int kNlmT = 3, kNlmS = 10, kNlmB = kNlmT + kNlmS;  // template / search / border radii
constexpr int kNlmWeights = 64;

__constant__ int c_nlm_weights[kNlmWeights];

__device__ __forceinline__ int nlm_reflect(int p, int n) {
    if (n == 1) return 0;
    while (p < 0 || p >= n) p = (p < 0) ? -p : 2 * n - 2 - p;
    return p;
}

// ---- the quad kernel -------------------------------------------------------------------------------------------------
constexpr int kNqCols = 160;                       // pixels per tile row: 40 threads x 4
constexpr int kNqQuads = kNqCols / 4;
constexpr int kNqRowsT = 10;                       // rows per thread
constexpr int kNqStrips = 4;                       // threads per column quad: 4 strips of kNqRowsT rows
constexpr int kNqRows = kNqRowsT * kNqStrips;      // 40 rows per tile: three tiles cover the 120 rows of a Lepton frame exactly
constexpr int kNqThreads = kNqQuads * kNqStrips;   // 160
constexpr int kNqPad = 16;                         // columns left / right of the tile in shared memory (>= 13, a multiple of 4)
constexpr int kNqExtW = kNqCols + 2 * kNqPad;      // 192 bytes per row
constexpr int kNqExtH = kNqRows + 2 * kNlmB;       // 58 rows
constexpr int kNqMinBlocks = 3;                    // CTAs per SM the register allocation allows

// info != nullptr: only the frames the extraction kernel marked for denoising (reserved[1] != 0) are processed
__global__ void __launch_bounds__(kNqThreads, kNqMinBlocks) nlm_quads_kernel(const uint8_t *src, int W, int H, uint8_t *dst, const cpt_frame_info *info) {
    if (info && info[blockIdx.z].reserved[1] == 0) return;
    __shared__ __align__(16) uint8_t ext[kNqExtH][kNqExtW];
    __shared__ int wtab[kNlmWeights];
    const int tid = threadIdx.x;
    const int x0t = blockIdx.x * kNqCols, y0t = blockIdx.y * kNqRows;
    const uint8_t *img = src + (size_t)blockIdx.z * W * H;
    for (int i = tid; i < kNqExtH * kNqExtW; i += kNqThreads) {
        const int ey = i / kNqExtW, ex = i - ey * kNqExtW;
        ext[ey][ex] = img[nlm_reflect(y0t + ey - kNlmB, H) * W + nlm_reflect(x0t + ex - kNqPad, W)];
    }
    if (tid < kNlmWeights) wtab[tid] = c_nlm_weights[tid];
    __syncthreads();
    const int ql = tid % kNqQuads, strip = tid / kNqQuads;
    const int lx = 4 * ql;                 // first column of the quad inside the tile
    const int er0 = kNqRowsT * strip + kNlmS;  // ext row of (first output row - 3): output row j's window is ext rows er0 + j .. er0 + j + 6
    uint32_t est[kNqRowsT][4], wsum[kNqRowsT][4];
#pragma unroll
    for (int j = 0; j < kNqRowsT; ++j)
#pragma unroll
        for (int i = 0; i < 4; ++i) { est[j][i] = 0u; wsum[j][i] = 0u; }
    // a: the thread's own columns x0 - 4 .. x0 + 7 as three aligned words per row (bytes 1 .. 10 are the template's reach)
    const uint8_t *arow = &ext[er0][lx + kNqPad - 4];
#pragma unroll 1
    for (int oy = -kNlmS; oy <= kNlmS; ++oy) {
#pragma unroll 1
        for (int ox = -kNlmS; ox <= kNlmS; ++ox) {
            // b: the same bytes of the image shifted by (ox, oy): four aligned words and a funnel shift per row
            const int sb = lx + kNqPad - 4 + ox;  // first byte wanted (>= 2)
            const uint8_t *brow = &ext[er0 + oy][sb & ~3];
            const uint32_t sh = (uint32_t)(sb & 3) * 8u;
            uint32_t ring[7][4];
            uint32_t V[4] = {0u, 0u, 0u, 0u};
            uint32_t bc[4] = {0u, 0u, 0u, 0u};  // the middle word of b of the last four rows: row rr - 3 holds the window's centre pixels
#pragma unroll
            for (int rr = 0; rr < kNqRowsT + 6; ++rr) {
                const uint32_t *ap = reinterpret_cast<const uint32_t *>(arow + rr * kNqExtW);
                const uint32_t *bp = reinterpret_cast<const uint32_t *>(brow + rr * kNqExtW);
                const uint32_t a0 = ap[0], a1 = ap[1], a2 = ap[2];
                const uint32_t r0 = bp[0], r1 = bp[1], r2 = bp[2], r3 = bp[3];
                const uint32_t b0 = __funnelshift_r(r0, r1, sh), b1 = __funnelshift_r(r1, r2, sh), b2 = __funnelshift_r(r2, r3, sh);
                const uint32_t d0 = __vabsdiffu4(a0, b0), d1 = __vabsdiffu4(a1, b1), d2 = __vabsdiffu4(a2, b2);
                // squares: byte k of word w is column x0 - 4 + 4 w + k; pixel i sums columns x0 + i - 3 .. x0 + i + 3
                const uint32_t mid = __dp4a(d1, d1, 0u);
                const uint32_t l3 = __dp4a(d0 & 0xff000000u, d0, 0u);          // column x0 - 1
                const uint32_t l2 = __dp4a(d0 & 0x00ff0000u, d0, l3);          // + x0 - 2
                const uint32_t l1 = __dp4a(d0 & 0x0000ff00u, d0, l2);          // + x0 - 3
                const uint32_t h0 = __dp4a(d2 & 0x000000ffu, d2, 0u);          // column x0 + 4
                const uint32_t h1 = __dp4a(d2 & 0x0000ff00u, d2, h0);          // + x0 + 5
                const uint32_t h2 = __dp4a(d2 & 0x00ff0000u, d2, h1);          // + x0 + 6
                const uint32_t Hs[4] = {mid + l1, mid + l2 + h0, mid + l3 + h1, mid + h2};
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    V[i] += Hs[i];
                    if (rr >= 7) V[i] -= ring[rr % 7][i];
                    ring[rr % 7][i] = Hs[i];
                }
                bc[rr & 3] = b1;
                if (rr >= 6) {
                    const int j = rr - 6;                    // output row: window rows rr - 6 .. rr, centre row rr - 3
                    const uint32_t cw = bc[(rr - 3) & 3];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const uint32_t a = min(V[i] >> 6, (uint32_t)(kNlmWeights - 1));  // (the table ends in zeros)
                        const uint32_t w = (uint32_t)wtab[a];
                        est[j][i] += w * ((cw >> (8 * i)) & 0xffu);
                        wsum[j][i] += w;
                    }
                }
            }
        }
    }
    const int x = x0t + lx, ybase = y0t + kNqRowsT * strip;
    uint8_t *out = dst + (size_t)blockIdx.z * W * H;
#pragma unroll
    for (int j = 0; j < kNqRowsT; ++j) {
        const int y = ybase + j;
        if (y >= H) continue;
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (x + i < W) out[y * W + x + i] = (uint8_t)((est[j][i] + wsum[j][i] / 2) / wsum[j][i]);
    }
}

}  // namespace cpt

using cpt::fail;

namespace cpt {

int nlm_prepare(cpt_ctx *c) {
    if (!c->nlm_table_ready) {
        // OpenCV FastNlMeansDenoisingInvoker: fixed_point_mult = INT_MAX / (21 * 21 * 255); template 49 -> shift 6
        const int fpm = 2147483647 / (21 * 21 * 255);
        const double mult = 64.0 / 49.0;
        int table[cpt::kNlmWeights];
        for (int a = 0; a < cpt::kNlmWeights; ++a) {
            const double w = std::exp(-(a * mult) / 9.0);
            int wi = (int)std::rint(fpm * w);
            if (wi < 0.001 * fpm) wi = 0;
            table[a] = wi;
        }
        if (table[cpt::kNlmWeights - 1] != 0) return fail(CPT_ERR_UNSUPPORTED, "internal: NLM weight table is longer than expected");
        CUDA_TRY(cudaMemcpyToSymbol(cpt::c_nlm_weights, table, sizeof(table)));
        c->nlm_table_ready = true;
    }
    return CPT_OK;
}

int nlm_launch(cpt_ctx *c, const uint8_t *d_src, int width, int height, long long n_frames, uint8_t *d_dst, const cpt_frame_info *info,
               cudaStream_t stream) {
    int rc = nlm_prepare(c);
    if (rc) return rc;
    for (long long f0 = 0; f0 < n_frames; f0 += 65535) {  // gridDim.z limit
        const int nz = (int)std::min<long long>(65535, n_frames - f0);
        const uint8_t *s0 = d_src + (size_t)f0 * width * height;
        uint8_t *d0 = d_dst + (size_t)f0 * width * height;
        const cpt_frame_info *i0 = info ? info + f0 : nullptr;
        dim3 grid((width + kNqCols - 1) / kNqCols, (height + kNqRows - 1) / kNqRows, nz);
        nlm_quads_kernel<<<grid, kNqThreads, 0, stream>>>(s0, width, height, d0, i0);
    }
    CUDA_TRY(cudaGetLastError());
    return CPT_OK;
}

}  // namespace cpt

extern "C" {

int cpt_nlm_denoise_u8(cpt_ctx *c, const uint8_t *d_src, int width, int height, int n_frames, uint8_t *d_dst) {
    if (!c || !d_src || !d_dst) return fail(CPT_ERR_INVALID, "null argument");
    if (width < 1 || height < 1 || n_frames < 0) return fail(CPT_ERR_INVALID, "bad size");
    if (n_frames == 0) return CPT_OK;
    CUDA_TRY(cudaSetDevice(c->device));
    return cpt::nlm_launch(c, d_src, width, height, n_frames, d_dst, nullptr, c->stream);
}

}  // extern "C"
