// cptrack.cu -- C ABI (include/cptrack.h) over the sm_100a kernels.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <functional>
#include <vector>

#include "cptrack_internal.cuh"

namespace cpt {
__global__ void extract_clips_kernel(const KernelArgs a);
__global__ void mask_components_kernel(const KernelArgs a, long long total_frames, const uint8_t *denoised);
__global__ void strip_sweep_kernel(const KernelArgs a);
__global__ void frame_scalars_kernel(const KernelArgs a);
size_t strip_sweep_smem_bytes();
__global__ void frame_regions_kernel(const KernelArgs a, long long total_frames);
__global__ void frame_components_kernel(const KernelArgs a, long long total_frames);
int cptv_decode_launch(cpt_ctx *c, const uint8_t *d_stream, const cpt_cptv_frame *d_table, int n_frames, const int32_t *d_clip_first,
                       int n_clips, uint16_t *d_frames, int32_t *scratch, cudaStream_t stream);
int nlm_launch(cpt_ctx *c, const uint8_t *d_src, int width, int height, long long n_frames, uint8_t *d_dst, const cpt_frame_info *info,
               cudaStream_t stream);
__global__ void region_variance_kernel(Geometry g, long long total_frames, const float *filtered, cpt_frame_info *info, cpt_region *regions);
__global__ void background_step_kernel(Geometry g, uint8_t *state, const int32_t *frames, const int *record_index, WeightTable wt);
__global__ void frame_median_kernel(const uint16_t *frames, int npx, float *out);
}

namespace {
thread_local char g_error[512] = "";
}  // namespace

namespace cpt {
char *error_buffer() { return g_error; }
}  // namespace cpt

using cpt::fail;
using cpt::HostWeightTable;

extern "C" {

const char *cpt_last_error(void) { return g_error; }

int cpt_version(void) { return 100; }

int cpt_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

cpt_ctx *cpt_ctx_create(int device, int width, int height, int edge_pixels, int max_regions) {
    if (width <= 0 || height <= 0 || width % 8 != 0 || width > cpt::kMaxW || height > cpt::kMaxH ||
        width * height > cpt::kMaxPx || (width * height) % 16 != 0) {
        fail(CPT_ERR_INVALID, "unsupported geometry %dx%d (need width%%8==0, width<=160, height<=120)", width, height);
        return nullptr;
    }
    if (edge_pixels < 0 || edge_pixels > 1 || height < 4) {
        fail(CPT_ERR_INVALID, "edge_pixels must be 0 or 1 (got %d) and height >= 4", edge_pixels);
        return nullptr;
    }
    if (max_regions < 1 || max_regions > CPT_MAX_COMPONENTS) {
        fail(CPT_ERR_INVALID, "max_regions must be in [1,%d]", CPT_MAX_COMPONENTS);
        return nullptr;
    }
    if (cudaSetDevice(device) != cudaSuccess) {
        fail(CPT_ERR_CUDA, "cudaSetDevice(%d) failed: %s", device, cudaGetErrorString(cudaGetLastError()));
        return nullptr;
    }
    cpt_ctx *c = new cpt_ctx();
    c->device = device;
    cpt::Geometry &g = c->g;
    g.W = width; g.H = height; g.edge = edge_pixels;
    g.npx = width * height; g.groups = g.npx / 8; g.gpr = width / 8;
    g.row_words = (width + 31) / 32; g.words = height * g.row_words;
    g.crop_w = width - 2 * edge_pixels; g.crop_h = height - 2 * edge_pixels; g.ncrop = g.crop_w * g.crop_h;
    g.block_w = (width + 1) / 2; g.max_regions = max_regions;
    g.gpr_magic = ((1u << 17) + g.gpr - 1) / g.gpr;
    g.rw_magic = ((1u << 13) + g.row_words - 1) / g.row_words;
    g.qpr = width / 4;
    {
        // strips of whole rows, at most kStripPxMax pixels, split evenly (a border row and the owned row next to it always
        // share a strip: every strip has at least two rows)
        const int rmax = std::max(cpt::kStripPxMax / width, 1);
        g.n_strips = (height + rmax - 1) / rmax;
    }
    g.qpr_magic = (uint32_t)(0xffffffffu / (uint32_t)std::max(g.qpr, 1)) + 1u;
    g.h_magic = (uint32_t)(0xffffffffu / (uint32_t)height) + 1u;
    g.qw_magic = (uint32_t)(0xffffffffu / (uint32_t)std::max(g.qpr / 4, 1)) + 1u;
    for (int st = 0; st < 20; ++st) g.strip_y0[st] = (uint8_t)(std::min(st, g.n_strips) * height / g.n_strips);
    g.rows_per_it = cpt::kPThreads / g.qpr;
    g.balanced = 0;
    g.bal_a_oy = g.bal_a_r = g.bal_b_oy = g.bal_b_r = -1;
    if (width == 160 && height == 120 && edge_pixels == 1) {
        const int R = g.rows_per_it, last = height - 2 * edge_pixels - 1, li = cpt::kQIter - 1;
        const int fr = last + 1 - li * R;  // first row group without a row of its own in the last iteration
        const int rb = last % R;           // row group of the last owned row
        if (last / R == li && li * R <= last && rb != 0 && fr > rb && fr + 1 < R) {
            g.balanced = 1;
            g.bal_a_oy = li * R; g.bal_a_r = fr;     // group 0 (top border row) hands over its last row
            g.bal_b_oy = rb; g.bal_b_r = fr + 1;     // group rb (bottom border row) hands over its first row
        }
    }
    if ((height - 2 * edge_pixels + g.rows_per_it - 1) / g.rows_per_it > cpt::kQIter) {
        fail(CPT_ERR_INVALID, "unsupported geometry %dx%d: too many sweep iterations", width, height);
        delete c;
        return nullptr;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
        fail(CPT_ERR_CUDA, "cudaGetDeviceProperties failed");
        delete c;
        return nullptr;
    }
    c->num_sms = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&c->d2h_stream, cudaStreamNonBlocking) != cudaSuccess) {
        fail(CPT_ERR_CUDA, "cudaStreamCreate failed");
        delete c;
        return nullptr;
    }
    c->stream = c->own_stream;
    if (cudaFuncSetAttribute(cpt::extract_clips_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)sizeof(cpt::Smem)) != cudaSuccess ||
        cudaFuncSetAttribute(cpt::strip_sweep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)cpt::strip_sweep_smem_bytes()) != cudaSuccess ||
        cudaFuncSetAttribute(cpt::frame_regions_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)sizeof(cpt::MaskSmem)) != cudaSuccess ||
        cudaFuncSetAttribute(cpt::frame_components_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)sizeof(cpt::CompSmem)) != cudaSuccess) {
        fail(CPT_ERR_CUDA, "cannot opt in to %zu bytes of shared memory: %s", sizeof(cpt::Smem),
             cudaGetErrorString(cudaGetLastError()));
        delete c;
        return nullptr;
    }
    if (cudaMalloc(&c->zero_frame, sizeof(uint16_t) * cpt::kMaxPx) != cudaSuccess ||
        cudaMemset(c->zero_frame, 0, sizeof(uint16_t) * cpt::kMaxPx) != cudaSuccess ||
        cudaMalloc(&c->work_counter, sizeof(int)) != cudaSuccess) {
        fail(CPT_ERR_NOMEM, "cudaMalloc failed");
        delete c;
        return nullptr;
    }
    g_error[0] = 0;
    return c;
}

void cpt_ctx_destroy(cpt_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (auto &t : c->tables) {
        cudaFree(t.d_thr);
    }
    for (int i = 0; i < 6; ++i)
        if (c->ev_k[i]) cudaEventDestroy(c->ev_k[i]);
    cudaFree(c->work_counter);
    cudaFree(c->zero_frame);
    cudaFree(c->debug);
    if (c->events)
        for (int i = 0; i < 2; ++i) {
            cudaEventDestroy(c->ev_h2d[i]);
            cudaEventDestroy(c->ev_compute[i]);
            cudaEventDestroy(c->ev_d2h[i]);
        }
    cudaStreamDestroy(c->own_stream);
    cudaStreamDestroy(c->copy_stream);
    cudaStreamDestroy(c->d2h_stream);
    delete c;  // (the scratch and staging buffers free themselves)
}

int cpt_ctx_set_stream(cpt_ctx *c, void *cuda_stream) {
    if (!c) return fail(CPT_ERR_INVALID, "null ctx");
    c->stream = (cudaStream_t)cuda_stream;  // NULL is the legacy default stream (what torch calls stream 0)
    return CPT_OK;
}

int cpt_ctx_synchronize(cpt_ctx *c) {
    if (!c) return fail(CPT_ERR_INVALID, "null ctx");
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return CPT_OK;
}

int cpt_build_weight_table(double weight_add, int n, uint32_t *thr_out, double *w_out) {
    if (n < 1 || !thr_out || !(weight_add >= 0.0)) return fail(CPT_ERR_INVALID, "bad weight table request");
    // background_weight accumulates by repeated += weight_add in fp64 (motiondetector.py:222-226);
    // entry layout and derivation: cptrack_kernels.cuh (WeightTable).
    volatile double acc = 0.0;
    for (int k = 0; k < n; ++k) {
        double w = acc;
        if (w_out) w_out[k] = w;
        double cw = std::ceil(w);
        double gap = cw - w;  // exact: cw and w agree in exponent range or gap is tiny
        uint32_t c = cw >= 65535.0 ? 65535u : (uint32_t)cw;
        uint32_t thr, bound = 0;
        if (c >= 65535u) {
            thr = 65535u;  // never keeps (d <= 65535 only when frame == 65535 and background == 0)
        } else if (gap == 0.0) {
            thr = c + 1u;
        } else {
            int ex;
            double m = std::frexp(gap, &ex);          // gap = m * 2^ex, m in [0.5, 1)
            int ceil_log2 = (m == 0.5) ? ex - 1 : ex;  // ceil(log2 gap)
            int E = ceil_log2 + 53;
            if (E >= 16) thr = c;
            else {
                thr = c + 1u;
                bound = 1u << std::max(E, 0);
            }
        }
        thr_out[k] = std::min(thr, 65535u) | (bound << 16);
        acc = acc + weight_add;
    }
    return CPT_OK;
}

int cpt_set_weight_table(cpt_ctx *c, int slot, double weight_add, int max_frames) {
    if (!c || slot < 0 || slot >= 4) return fail(CPT_ERR_INVALID, "weight table slot must be 0..3");
    if (max_frames < 1 || max_frames > 65534) return fail(CPT_ERR_INVALID, "max_frames must be in [1,65534]");
    if (!(weight_add >= 0.0)) return fail(CPT_ERR_INVALID, "weight_add must be >= 0");
    CUDA_TRY(cudaSetDevice(c->device));
    HostWeightTable &t = c->tables[slot];
    int n = max_frames + 1;
    t.w.assign(n, 0.0);
    std::vector<uint32_t> thr(n);
    cpt_build_weight_table(weight_add, n, thr.data(), t.w.data());
    thr[n - 1] = 0xffffu;  // a count can never pass the end of the table: the last entry never keeps
    cudaFree(t.d_thr);
    t.d_thr = nullptr;
    CUDA_TRY(cudaMalloc(&t.d_thr, sizeof(uint32_t) * n));
    CUDA_TRY(cudaMemcpy(t.d_thr, thr.data(), sizeof(uint32_t) * n, cudaMemcpyHostToDevice));
    t.max_count = max_frames;
    t.has_bounds = 0;
    t.max_bound = 0;
    t.linear_upto = n;
    for (int k = 0; k < n; ++k) {
        t.has_bounds |= (thr[k] >> 16) != 0;
        t.max_bound = std::max(t.max_bound, (int)(thr[k] >> 16));
        if (t.linear_upto == n && thr[k] != (uint32_t)(k + 1)) t.linear_upto = k;
    }
    return CPT_OK;
}

double cpt_weight_value(const cpt_ctx *c, int slot, int count) {
    if (!c || slot < 0 || slot >= 4) return NAN;
    const HostWeightTable &t = c->tables[slot];
    if (count < 0 || count >= (int)t.w.size()) return NAN;
    return t.w[count];
}

int cpt_device_alloc(cpt_ctx *c, void **d_ptr, uint64_t bytes) {
    if (!c || !d_ptr) return fail(CPT_ERR_INVALID, "null argument");
    CUDA_TRY(cudaSetDevice(c->device));
    cudaError_t e = cudaMalloc(d_ptr, bytes);
    if (e != cudaSuccess) return fail(CPT_ERR_NOMEM, "cudaMalloc(%llu): %s", (unsigned long long)bytes, cudaGetErrorString(e));
    return CPT_OK;
}

int cpt_device_free(cpt_ctx *c, void *d_ptr) {
    if (!c) return fail(CPT_ERR_INVALID, "null ctx");
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(cudaFree(d_ptr));
    return CPT_OK;
}

int cpt_host_alloc_pinned(void **h_ptr, uint64_t bytes) {
    if (!h_ptr) return fail(CPT_ERR_INVALID, "null argument");
    cudaError_t e = cudaHostAlloc(h_ptr, bytes, cudaHostAllocDefault);
    if (e != cudaSuccess) return fail(CPT_ERR_NOMEM, "cudaHostAlloc(%llu): %s", (unsigned long long)bytes, cudaGetErrorString(e));
    return CPT_OK;
}

int cpt_host_free_pinned(void *h_ptr) {
    CUDA_TRY(cudaFreeHost(h_ptr));
    return CPT_OK;
}

int cpt_copy_to_device(cpt_ctx *c, void *d_dst, const void *h_src, uint64_t bytes) {
    if (!c) return fail(CPT_ERR_INVALID, "null ctx");
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, c->stream));
    return CPT_OK;
}

int cpt_copy_to_host(cpt_ctx *c, void *h_dst, const void *d_src, uint64_t bytes) {
    if (!c) return fail(CPT_ERR_INVALID, "null ctx");
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, c->stream));
    return CPT_OK;
}

/* Debug builds only (-DCPT_PHASE_TIMING): allocate / read the per-CTA phase cycle counters. */
int cpt_debug_phase_cycles(cpt_ctx *c, long long *h_out32, int reset) {
    if (!c) return fail(CPT_ERR_INVALID, "null ctx");
    CUDA_TRY(cudaSetDevice(c->device));
    size_t bytes = sizeof(long long) * 32 * (size_t)c->num_sms;
    if (!c->debug) {
        CUDA_TRY(cudaMalloc(&c->debug, bytes));
        CUDA_TRY(cudaMemset(c->debug, 0, bytes));
    }
    CUDA_TRY(cudaDeviceSynchronize());
    if (h_out32) {
        std::vector<long long> all(32 * (size_t)c->num_sms);
        CUDA_TRY(cudaMemcpy(all.data(), c->debug, bytes, cudaMemcpyDeviceToHost));
        for (int i = 0; i < 32; ++i) {
            long long sum = 0;
            for (int b = 0; b < c->num_sms; ++b) sum += all[(size_t)b * 32 + i];
            h_out32[i] = sum;
        }
    }
    if (reset) CUDA_TRY(cudaMemset(c->debug, 0, bytes));
    return CPT_OK;
}

int cpt_debug_force_single_kernel(cpt_ctx *c, int enable) {
    if (!c) return fail(CPT_ERR_INVALID, "null ctx");
    c->force_single = enable != 0;
    return CPT_OK;
}

int cpt_debug_kernel_times_ex(cpt_ctx *c, int enable, float *h_ms, int n) {
    if (!c) return fail(CPT_ERR_INVALID, "null ctx");
    if (h_ms && (n < 1 || n > 5)) return fail(CPT_ERR_INVALID, "n must be in [1,5]");
    CUDA_TRY(cudaSetDevice(c->device));
    if (enable && !c->ev_k[0])
        for (int i = 0; i < 6; ++i) CUDA_TRY(cudaEventCreate(&c->ev_k[i]));
    if (h_ms) {
        for (int i = 0; i < n; ++i) h_ms[i] = 0.f;
        if (c->timed_valid) {
            CUDA_TRY(cudaEventSynchronize(c->ev_k[5]));
            for (int i = 0; i < n; ++i) CUDA_TRY(cudaEventElapsedTime(&h_ms[i], c->ev_k[i], c->ev_k[i + 1]));
        }
    }
    c->time_kernels = enable != 0;
    return CPT_OK;
}

uint64_t cpt_state_bytes(const cpt_ctx *c) { return c ? cpt::state_bytes(c->g.npx) : 0; }

static int launch_extract(cpt_ctx *c, const uint16_t *d_frames, const cpt_clip *d_clips, int n_clips,
                          const cpt_outputs *out, void *d_state, cudaStream_t stream, long long total_frames) {
    if (n_clips == 0) return CPT_OK;
    int grid = std::min(n_clips, c->num_sms);
    if (!out->d_filtered) CUDA_TRY(c->scratch.ensure((size_t)c->num_sms * 8 * c->g.npx));
    cpt::KernelArgs a{};
    a.g = c->g;
    a.frames = d_frames;
    a.clips = d_clips;
    a.n_clips = n_clips;
    a.regions = out->d_regions;
    a.info = out->d_info;
    a.filtered = out->d_filtered;
    a.labels = out->d_labels;
    a.scratch = out->d_filtered ? nullptr : static_cast<float *>(c->scratch);
    a.state = (uint8_t *)d_state;
    for (int i = 0; i < 4; ++i) a.tables[i] = c->tables[i].device();
    a.work_counter = c->work_counter;
    a.zero_frame = c->zero_frame;
    a.debug = c->debug;
    CUDA_TRY(cudaMemsetAsync(c->work_counter, 0, sizeof(int), stream));
    // with the filtered images kept and the frame count known, the per-region variances of all frames but the
    // first of each clip are computed by a second, wide launch
    a.defer_variance = (out->d_filtered != nullptr && total_frames > 1) ? 1 : 0;
    if (out->denoise) {
        // CPT_CLIP_DENOISE clips: normalised images -> cv2.fastNlMeansDenoising -> masks and components, as three
        // passes over all frames (the recurrence does not depend on the masks)
        if (total_frames < 1 || !out->d_filtered)
            return fail(CPT_ERR_INVALID, "denoise needs cpt_outputs.total_frames and d_filtered");
        for (auto &u8 : c->u8_frames) CUDA_TRY(u8.ensure((size_t)total_frames * c->g.npx));
        a.u8_frames = c->u8_frames[0];
        a.defer_variance = 1;
    }
    // Batch launches that keep the filtered images and carry no per-clip state take the split path: the recurrence as a
    // persistent sweep kernel, then one CTA per frame for masks / components.  A state record may be written (not
    // resumed from).  Everything else (streaming, resumed clips, regions-only launches) runs the single persistent
    // kernel with its three warp roles.
    const bool timed = c->time_kernels && c->ev_k[0];
    if (timed) CUDA_TRY(cudaEventRecord(c->ev_k[0], stream));
    // (the sweep kernel stages frame rows with 16-byte bulk copies: rows must be a multiple of 8 pixels)
    const bool split = !c->force_single && (d_state == nullptr || out->no_resume) && out->d_filtered != nullptr &&
                       total_frames > 0 && c->g.W % 8 == 0;
    if (split) {
        const size_t nf = (size_t)total_frames, nc = (size_t)n_clips;
        CUDA_TRY(c->qbytes.ensure(nf * c->g.H * c->g.qpr));
        CUDA_TRY(c->prec.ensure((nf + nc) * c->g.n_strips));
        CUDA_TRY(c->fhdr.ensure(nf));
        CUDA_TRY(c->maskbits.ensure(nf * cpt::kMaxWords));
        CUDA_TRY(c->fallback.ensure(nf + 1));
        a.qbytes = c->qbytes;
        a.prec = c->prec;
        a.fhdr = c->fhdr;
        a.maskbits = c->maskbits;
        a.fallback = c->fallback;
        CUDA_TRY(cudaMemsetAsync(c->fallback, 0, sizeof(int), stream));
        a.total_frames = total_frames;
        // the valid flag of every output frame starts cleared: frames no clip writes are skipped by the per-frame launches
        CUDA_TRY(cudaMemsetAsync(c->fhdr, 0, (size_t)total_frames * sizeof(cpt::FrameHdr), stream));
        const long long units = (long long)n_clips * c->g.n_strips;
        const int sgrid = (int)std::min<long long>(units, c->num_sms);
        cpt::strip_sweep_kernel<<<sgrid, cpt::kStripThreads, cpt::strip_sweep_smem_bytes(), stream>>>(a);
        CUDA_TRY(cudaGetLastError());
        if (timed) CUDA_TRY(cudaEventRecord(c->ev_k[1], stream));
        cpt::frame_scalars_kernel<<<(n_clips + 3) / 4, 128, 0, stream>>>(a);
        CUDA_TRY(cudaGetLastError());
        if (timed) CUDA_TRY(cudaEventRecord(c->ev_k[2], stream));
        cpt::frame_regions_kernel<<<(unsigned)total_frames, cpt::kFThreads, sizeof(cpt::MaskSmem), stream>>>(a, total_frames);
        CUDA_TRY(cudaGetLastError());
        cpt::frame_components_kernel<<<(unsigned)std::min<long long>(total_frames, 2LL * c->num_sms), cpt::kGThreads, sizeof(cpt::CompSmem), stream>>>(a, total_frames);
        CUDA_TRY(cudaGetLastError());
    } else {
        cpt::extract_clips_kernel<<<grid, cpt::kThreads, sizeof(cpt::Smem), stream>>>(a);
        CUDA_TRY(cudaGetLastError());
        if (timed) {
            CUDA_TRY(cudaEventRecord(c->ev_k[1], stream));
            CUDA_TRY(cudaEventRecord(c->ev_k[2], stream));
        }
    }
    if (timed) CUDA_TRY(cudaEventRecord(c->ev_k[3], stream));
    if (out->denoise) {
        int rc = cpt::nlm_launch(c, c->u8_frames[0], c->g.W, c->g.H, total_frames, c->u8_frames[1], out->d_info, stream);
        if (rc) return rc;
        if (cudaFuncSetAttribute(cpt::mask_components_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(cpt::Smem)) != cudaSuccess)
            return fail(CPT_ERR_CUDA, "cannot opt in to shared memory for mask_components_kernel");
        const int mgrid = (int)std::min<long long>(total_frames, c->num_sms);
        cpt::mask_components_kernel<<<mgrid, cpt::kThreads, sizeof(cpt::Smem), stream>>>(a, total_frames, c->u8_frames[1]);
        CUDA_TRY(cudaGetLastError());
    }
    if (timed) CUDA_TRY(cudaEventRecord(c->ev_k[4], stream));
    if (a.defer_variance) {
        constexpr int fpb = cpt::kVarThreads / 32;  // frames per block
        const unsigned blocks = (unsigned)((total_frames + fpb - 1) / fpb);
        cpt::region_variance_kernel<<<blocks, cpt::kVarThreads, 0, stream>>>(c->g, total_frames, out->d_filtered, out->d_info, out->d_regions);
        CUDA_TRY(cudaGetLastError());
    }
    if (timed) {
        CUDA_TRY(cudaEventRecord(c->ev_k[5], stream));
        c->timed_valid = true;
    }
    return CPT_OK;
}

int cpt_extract_batch(cpt_ctx *c, const uint16_t *d_frames, const cpt_clip *d_clips, int n_clips,
                      const cpt_outputs *out, void *d_state) {
    if (!c || !out) return fail(CPT_ERR_INVALID, "null argument");
    if (n_clips < 0) return fail(CPT_ERR_INVALID, "n_clips < 0");
    if (n_clips == 0) return CPT_OK;
    if (!d_frames || !d_clips) return fail(CPT_ERR_INVALID, "null frames / clips");
    if (!out->d_info || !out->d_regions) return fail(CPT_ERR_INVALID, "d_info and d_regions are required");
    if (!c->tables[0].d_thr && !c->tables[1].d_thr && !c->tables[2].d_thr && !c->tables[3].d_thr)
        return fail(CPT_ERR_INVALID, "no weight table set (cpt_set_weight_table)");
    CUDA_TRY(cudaSetDevice(c->device));
    if (out->total_frames < 0) return fail(CPT_ERR_INVALID, "total_frames < 0");
    return launch_extract(c, d_frames, d_clips, n_clips, out, d_state, c->stream, out->total_frames);
}

// One chunk of a host-staged call: clips [c0, c1), the input they read -- frames of the raw call, frame table rows of the
// packed call -- [in_lo, in_hi), the output frames they write [out_lo, out_hi) and, packed call only, the payload bytes of
// their rows [byte_lo, byte_hi)
struct Chunk {
    int c0, c1;
    int64_t in_lo, in_hi, out_lo, out_hi;
    uint64_t byte_lo, byte_hi;
};

static std::vector<Chunk> make_chunks(int n_clips, int chunk_clips) {
    std::vector<Chunk> chunks;
    for (int c0 = 0; c0 < n_clips; c0 = chunks.back().c1) chunks.push_back(Chunk{c0, c0 + std::min(chunk_clips, n_clips - c0)});
    return chunks;
}

using ChunkStep = std::function<int(int ch, int b)>;

// The pipeline of both host-staged calls, double-buffered over the chunks: chunk ch uses staging buffers b = ch & 1.
// `upload` enqueues the chunk's input on copy_stream; `decode` (packed call only) turns it into frames in stage_frames[b]
// on c->stream.  The extraction runs on c->stream and its outputs go back to the host on d2h_stream.  The clips come
// validated and the chunks with their input spans; this finds the output spans and rebases the clips to both.
static int run_host_staged(cpt_ctx *c, const cpt_clip *h_clips, std::vector<Chunk> &chunks, cpt_region *h_regions,
                           cpt_frame_info *h_info, float *h_filtered, uint8_t *h_labels, const ChunkStep &upload,
                           const ChunkStep &decode) {
    const size_t npx = c->g.npx;
    const int n_clips = chunks.back().c1;
    std::vector<cpt_clip> rebased(h_clips, h_clips + n_clips);
    size_t max_in = 1, max_out = 1;
    for (Chunk &k : chunks) {
        k.out_lo = INT64_MAX;
        k.out_hi = 0;
        for (int i = k.c0; i < k.c1; ++i) {
            k.out_lo = std::min(k.out_lo, h_clips[i].out_offset);
            k.out_hi = std::max(k.out_hi, h_clips[i].out_offset + h_clips[i].n_frames);
        }
        for (int i = k.c0; i < k.c1; ++i) {
            rebased[i].frame_offset -= k.in_lo;
            rebased[i].init_offset -= k.in_lo;
            rebased[i].out_offset -= k.out_lo;
        }
        max_in = std::max(max_in, (size_t)(k.in_hi - k.in_lo));
        max_out = std::max(max_out, (size_t)(k.out_hi - k.out_lo));
    }
    if (!c->events) {
        for (int i = 0; i < 2; ++i) {
            CUDA_TRY(cudaEventCreateWithFlags(&c->ev_h2d[i], cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&c->ev_compute[i], cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&c->ev_d2h[i], cudaEventDisableTiming));
        }
        c->events = true;
    }
    for (int b = 0; b < 2; ++b) {
        CUDA_TRY(c->stage_frames[b].ensure(max_in * npx));
        CUDA_TRY(c->stage_regions[b].ensure(max_out * c->g.max_regions));
        CUDA_TRY(c->stage_info[b].ensure(max_out));
        if (h_filtered) CUDA_TRY(c->stage_filtered[b].ensure(max_out * npx));
        if (h_labels) CUDA_TRY(c->stage_labels[b].ensure(max_out * npx));
    }
    // calls that do not return the filtered images still run the split plan (it keeps the whole GPU busy with (clip, strip)
    // units where the single persistent kernel has one CTA per clip): the images go to a scratch buffer
    if (!h_filtered) CUDA_TRY(c->scratch_filtered.ensure(max_out * npx));
    CUDA_TRY(c->d_clips.ensure(n_clips));
    CUDA_TRY(cudaMemcpyAsync(c->d_clips, rebased.data(), sizeof(cpt_clip) * n_clips, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    for (int ch = 0; ch < (int)chunks.size(); ++ch) {
        const Chunk &k = chunks[ch];
        const int b = ch & 1;
        // staging buffers b are free once the kernels of chunk ch-2 have run and its outputs have been copied back
        if (ch >= 2) CUDA_TRY(cudaStreamWaitEvent(c->copy_stream, c->ev_compute[b], 0));
        if (int rc = upload(ch, b)) return rc;
        CUDA_TRY(cudaEventRecord(c->ev_h2d[b], c->copy_stream));
        CUDA_TRY(cudaStreamWaitEvent(c->stream, c->ev_h2d[b], 0));
        if (ch >= 2) CUDA_TRY(cudaStreamWaitEvent(c->stream, c->ev_d2h[b], 0));
        if (decode)
            if (int rc = decode(ch, b)) return rc;
        int denoise = 0;  // (CPT_CLIP_DENOISE clips: the NLM, mask and component passes follow the chunk's launch)
        for (int i = k.c0; i < k.c1; ++i) denoise |= (h_clips[i].flags & CPT_CLIP_DENOISE) ? 1 : 0;
        const int64_t nf = k.out_hi - k.out_lo;
        cpt_outputs out{c->stage_regions[b], c->stage_info[b], h_filtered ? c->stage_filtered[b] : c->scratch_filtered,
                        h_labels ? static_cast<uint8_t *>(c->stage_labels[b]) : nullptr, nf, denoise, 1};
        if (int rc = launch_extract(c, c->stage_frames[b], c->d_clips + k.c0, k.c1 - k.c0, &out, nullptr, c->stream, nf)) return rc;
        CUDA_TRY(cudaEventRecord(c->ev_compute[b], c->stream));
        CUDA_TRY(cudaStreamWaitEvent(c->d2h_stream, c->ev_compute[b], 0));
        CUDA_TRY(cudaMemcpyAsync(h_regions + (size_t)k.out_lo * c->g.max_regions, c->stage_regions[b],
                                 (size_t)nf * c->g.max_regions * sizeof(cpt_region), cudaMemcpyDeviceToHost, c->d2h_stream));
        CUDA_TRY(cudaMemcpyAsync(h_info + k.out_lo, c->stage_info[b], (size_t)nf * sizeof(cpt_frame_info), cudaMemcpyDeviceToHost, c->d2h_stream));
        if (h_filtered)
            CUDA_TRY(cudaMemcpyAsync(h_filtered + (size_t)k.out_lo * npx, c->stage_filtered[b], (size_t)nf * npx * sizeof(float),
                                     cudaMemcpyDeviceToHost, c->d2h_stream));
        if (h_labels)
            CUDA_TRY(cudaMemcpyAsync(h_labels + (size_t)k.out_lo * npx, c->stage_labels[b], (size_t)nf * npx, cudaMemcpyDeviceToHost, c->d2h_stream));
        CUDA_TRY(cudaEventRecord(c->ev_d2h[b], c->d2h_stream));
    }
    CUDA_TRY(cudaStreamSynchronize(c->d2h_stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return CPT_OK;
}

int cpt_extract_batch_host(cpt_ctx *c, const uint16_t *h_frames, const cpt_clip *h_clips, int n_clips,
                           int64_t total_frames, cpt_region *h_regions, cpt_frame_info *h_info,
                           float *h_filtered, uint8_t *h_labels, int chunk_clips) {
    if (!c) return fail(CPT_ERR_INVALID, "null ctx");
    if (n_clips < 0 || total_frames < 0) return fail(CPT_ERR_INVALID, "negative sizes");
    if (n_clips == 0) return CPT_OK;
    if (!h_frames || !h_clips || !h_regions || !h_info) return fail(CPT_ERR_INVALID, "null host buffer");
    CUDA_TRY(cudaSetDevice(c->device));
    std::vector<Chunk> chunks = make_chunks(n_clips, chunk_clips > 0 ? chunk_clips : c->num_sms);
    for (Chunk &sp : chunks) {
        // the chunk's input: from the first frame its clips read to past the last
        sp.in_lo = INT64_MAX;
        for (int i = sp.c0; i < sp.c1; ++i) {
            const cpt_clip &k = h_clips[i];
            if (k.flags & CPT_CLIP_RESUME) return fail(CPT_ERR_INVALID, "CPT_CLIP_RESUME is not supported by the host-staged call");
            if (k.n_frames < 0 || k.frame_offset < 0 || k.init_offset < 0 || k.out_offset < 0 || k.ring_frames != 0)
                return fail(CPT_ERR_INVALID, "clip %d: bad offsets", i);
            if (k.out_offset + k.n_frames > total_frames) return fail(CPT_ERR_INVALID, "clip %d: outputs exceed total_frames", i);
            sp.in_lo = std::min({sp.in_lo, k.frame_offset, k.init_offset});
            sp.in_hi = std::max({sp.in_hi, k.frame_offset + k.n_frames, k.init_offset + 1});
        }
    }
    const size_t npx = c->g.npx;
    auto upload = [&](int ch, int b) -> int {
        const Chunk &sp = chunks[ch];
        CUDA_TRY(cudaMemcpyAsync(c->stage_frames[b], h_frames + (size_t)sp.in_lo * npx, (size_t)(sp.in_hi - sp.in_lo) * npx * sizeof(uint16_t),
                                 cudaMemcpyHostToDevice, c->copy_stream));
        return CPT_OK;
    };
    return run_host_staged(c, h_clips, chunks, h_regions, h_info, h_filtered, h_labels, upload, nullptr);
}

// Host-staged extraction from PACKED clips: the inflated CPTV frame payloads travel over PCIe (about one byte per pixel
// instead of two), cpt_cptv_decode's kernels rebuild the uint16 frames on the device, the extraction runs on them.
int cpt_extract_batch_cptv_host(cpt_ctx *c, const uint8_t *h_stream, uint64_t stream_bytes, const cpt_cptv_frame *h_table,
                                const int64_t *h_clip_first, const cpt_clip *h_clips, int n_clips, int64_t total_frames,
                                cpt_region *h_regions, cpt_frame_info *h_info, int chunk_clips) {
    if (!c) return fail(CPT_ERR_INVALID, "null ctx");
    if (n_clips < 0 || total_frames < 0) return fail(CPT_ERR_INVALID, "negative sizes");
    if (n_clips == 0) return CPT_OK;
    if (!h_stream || !h_table || !h_clip_first || !h_clips || !h_regions || !h_info) return fail(CPT_ERR_INVALID, "null host buffer");
    CUDA_TRY(cudaSetDevice(c->device));
    if (chunk_clips <= 0) chunk_clips = c->num_sms;
    const size_t npx = c->g.npx;
    std::vector<Chunk> chunks = make_chunks(n_clips, chunk_clips);
    size_t max_rows = 1, max_bytes = 0;
    for (Chunk &sp : chunks) {
        // the chunk's input: the frame table rows of its clips and the payload bytes of those rows
        sp.in_lo = h_clip_first[sp.c0];
        sp.in_hi = h_clip_first[sp.c1];
        if (sp.in_lo < 0 || sp.in_hi < sp.in_lo) return fail(CPT_ERR_INVALID, "clip table rows must ascend");
        sp.byte_lo = UINT64_MAX;
        for (int64_t r = sp.in_lo; r < sp.in_hi; ++r) {
            // every payload must lie inside the stream (a malformed file must not make the device read out of bounds)
            const cpt_cptv_frame &f = h_table[r];
            if (f.bit_width < 1 || f.bit_width > 24) return fail(CPT_ERR_INVALID, "frame %lld: unsupported bit width %d", (long long)r, f.bit_width);
            const uint64_t size = 4 + ((uint64_t)(npx - 1) * (uint64_t)f.bit_width + 7) / 8;
            if (f.payload_offset > stream_bytes || size > stream_bytes - f.payload_offset)
                return fail(CPT_ERR_INVALID, "frame %lld: payload outside the stream", (long long)r);
            sp.byte_lo = std::min(sp.byte_lo, f.payload_offset);
            sp.byte_hi = std::max(sp.byte_hi, f.payload_offset + size);
        }
        if (sp.in_hi == sp.in_lo) sp.byte_lo = 0;
        for (int i = sp.c0; i < sp.c1; ++i) {
            const cpt_clip &k = h_clips[i];
            if (k.flags & CPT_CLIP_RESUME) return fail(CPT_ERR_UNSUPPORTED, "clip %d: CPT_CLIP_RESUME is not supported by the host-staged calls", i);
            if (k.n_frames < 0 || k.out_offset < 0 || k.ring_frames != 0) return fail(CPT_ERR_INVALID, "clip %d: bad offsets", i);
            if (k.frame_offset < h_clip_first[i] || k.frame_offset + k.n_frames > h_clip_first[i + 1] || k.init_offset < h_clip_first[i] ||
                k.init_offset >= std::max(h_clip_first[i + 1], h_clip_first[i] + 1))
                return fail(CPT_ERR_INVALID, "clip %d: frames outside the clip's rows of the frame table", i);
            if (k.out_offset + k.n_frames > total_frames) return fail(CPT_ERR_INVALID, "clip %d: outputs exceed total_frames", i);
        }
        max_rows = std::max(max_rows, (size_t)(sp.in_hi - sp.in_lo));
        max_bytes = std::max(max_bytes, (size_t)(sp.byte_hi - sp.byte_lo));
    }
    // packed staging: payload bytes (+4: the unpacker's 32-bit window may read past the last payload), frame table rows,
    // the clips' first rows; the decoder's int32 change images
    for (int b = 0; b < 2; ++b) {
        CUDA_TRY(c->pk_stream[b].ensure(max_bytes + 4));
        CUDA_TRY(c->pk_table[b].ensure(max_rows));
        CUDA_TRY(c->pk_h_table[b].ensure(max_rows));
        CUDA_TRY(c->pk_first[b].ensure((size_t)chunk_clips + 1));
        CUDA_TRY(c->pk_h_first[b].ensure((size_t)chunk_clips + 1));
    }
    CUDA_TRY(c->pk_change.ensure(max_rows * npx));
    auto upload = [&](int ch, int b) -> int {
        const Chunk &sp = chunks[ch];
        const int rows = (int)(sp.in_hi - sp.in_lo);
        // the host tables of buffers b are rewritten here: the copies of chunk ch-2 out of them must have run
        if (ch >= 2) CUDA_TRY(cudaEventSynchronize(c->ev_compute[b]));
        for (int r = 0; r < rows; ++r) {
            c->pk_h_table[b][r] = h_table[sp.in_lo + r];
            c->pk_h_table[b][r].payload_offset -= sp.byte_lo;
        }
        for (int i = sp.c0; i <= sp.c1; ++i) c->pk_h_first[b][i - sp.c0] = (int32_t)(h_clip_first[i] - sp.in_lo);
        if (rows > 0) {
            CUDA_TRY(cudaMemcpyAsync(c->pk_stream[b], h_stream + sp.byte_lo, (size_t)(sp.byte_hi - sp.byte_lo), cudaMemcpyHostToDevice, c->copy_stream));
            CUDA_TRY(cudaMemcpyAsync(c->pk_table[b], c->pk_h_table[b], (size_t)rows * sizeof(cpt_cptv_frame), cudaMemcpyHostToDevice, c->copy_stream));
        }
        CUDA_TRY(cudaMemcpyAsync(c->pk_first[b], c->pk_h_first[b], (size_t)(sp.c1 - sp.c0 + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, c->copy_stream));
        return CPT_OK;
    };
    auto decode = [&](int ch, int b) -> int {
        const Chunk &sp = chunks[ch];
        const int rows = (int)(sp.in_hi - sp.in_lo);
        if (rows == 0) return CPT_OK;
        return cpt::cptv_decode_launch(c, c->pk_stream[b], c->pk_table[b], rows, c->pk_first[b], sp.c1 - sp.c0, c->stage_frames[b],
                                       c->pk_change, c->stream);
    };
    return run_host_staged(c, h_clips, chunks, h_regions, h_info, nullptr, nullptr, upload, decode);
}

int cpt_background_process(cpt_ctx *c, void *d_state, const int32_t *d_record_index, int n_records,
                           const int32_t *d_frames, int weight_slot) {
    if (!c || !d_state || !d_frames) return fail(CPT_ERR_INVALID, "null argument");
    if (n_records < 0) return fail(CPT_ERR_INVALID, "n_records < 0");
    if (weight_slot < 0 || weight_slot >= 4 || !c->tables[weight_slot].d_thr)
        return fail(CPT_ERR_INVALID, "weight table slot %d is not set (cpt_set_weight_table)", weight_slot);
    if (n_records == 0) return CPT_OK;
    CUDA_TRY(cudaSetDevice(c->device));
    cpt::WeightTable wt = c->tables[weight_slot].device();
    cpt::background_step_kernel<<<n_records, 1024, 0, c->stream>>>(c->g, (uint8_t *)d_state, d_frames, d_record_index, wt);
    CUDA_TRY(cudaGetLastError());
    return CPT_OK;
}

int cpt_frame_medians(cpt_ctx *c, const uint16_t *d_frames, int64_t n_frames, float *d_medians) {
    if (!c || !d_frames || !d_medians) return fail(CPT_ERR_INVALID, "null argument");
    if (n_frames < 0 || n_frames > 0x7fffffff) return fail(CPT_ERR_INVALID, "bad n_frames");
    if (n_frames == 0) return CPT_OK;
    CUDA_TRY(cudaSetDevice(c->device));
    const size_t smem = (((size_t)c->g.npx * sizeof(uint16_t) + 15) & ~(size_t)15) + 2048 * sizeof(uint32_t);  // median.cuh bins
    cpt::frame_median_kernel<<<(unsigned)n_frames, 256, smem, c->stream>>>(d_frames, c->g.npx, d_medians);
    CUDA_TRY(cudaGetLastError());
    return CPT_OK;
}

int cpt_state_read(cpt_ctx *c, const void *d_state, int clip_index, int32_t *h_background, uint16_t *h_weight_count,
                   double *h_average, uint32_t *h_sliding_sum, int32_t *h_frames_seen) {
    if (!c || !d_state || clip_index < 0) return fail(CPT_ERR_INVALID, "bad argument");
    CUDA_TRY(cudaSetDevice(c->device));
    const cpt::Geometry &g = c->g;
    size_t sb = cpt::state_bytes(g.npx);
    std::vector<uint8_t> buf(sb);
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    CUDA_TRY(cudaMemcpy(buf.data(), (const uint8_t *)d_state + sb * clip_index, sb, cudaMemcpyDeviceToHost));
    const cpt::StateHeader *h = (const cpt::StateHeader *)buf.data();
    const uint16_t *B = (const uint16_t *)(buf.data() + sizeof(cpt::StateHeader));
    const uint16_t *K = B + g.npx;
    const uint32_t *S = (const uint32_t *)(K + g.npx);
    if (h_background)
        for (int i = 0; i < g.npx; ++i) h_background[i] = B[i];
    if (h_weight_count)
        for (int y = 0; y < g.crop_h; ++y)
            for (int x = 0; x < g.crop_w; ++x) h_weight_count[y * g.crop_w + x] = K[(y + g.edge) * g.W + x + g.edge];
    if (h_average) *h_average = h->average;
    if (h_sliding_sum) memcpy(h_sliding_sum, S, sizeof(uint32_t) * g.npx);
    if (h_frames_seen) *h_frames_seen = h->frames_seen;
    return CPT_OK;
}

int cpt_state_write(cpt_ctx *c, void *d_state, int clip_index, const int32_t *h_background,
                    const uint16_t *h_weight_count, double average) {
    if (!c || !d_state || clip_index < 0 || !h_background) return fail(CPT_ERR_INVALID, "bad argument");
    CUDA_TRY(cudaSetDevice(c->device));
    const cpt::Geometry &g = c->g;
    size_t sb = cpt::state_bytes(g.npx);
    std::vector<uint8_t> buf(sb, 0);
    cpt::StateHeader *h = (cpt::StateHeader *)buf.data();
    uint16_t *B = (uint16_t *)(buf.data() + sizeof(cpt::StateHeader));
    uint16_t *K = B + g.npx;
    for (int i = 0; i < g.npx; ++i) {
        if (h_background[i] < 0 || h_background[i] > 65535) return fail(CPT_ERR_INVALID, "background value out of uint16 range");
        B[i] = (uint16_t)h_background[i];
    }
    if (h_weight_count)
        for (int y = 0; y < g.crop_h; ++y)
            for (int x = 0; x < g.crop_w; ++x) K[(y + g.edge) * g.W + x + g.edge] = h_weight_count[y * g.crop_w + x];
    h->average = average;
    h->initialised = 1;
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    CUDA_TRY(cudaMemcpy((uint8_t *)d_state + sb * clip_index, buf.data(), sb, cudaMemcpyHostToDevice));
    return CPT_OK;
}

}  // extern "C"
