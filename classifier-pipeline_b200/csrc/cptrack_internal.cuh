// cptrack_internal.cuh -- what the translation units behind the C ABI share: the context record,
// error reporting and the CUDA_TRY macro.  Not part of the public interface (include/cptrack.h).
#pragma once
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <vector>

#include "cptrack_kernels.cuh"

namespace cpt {

char *error_buffer();  // thread local, 512 bytes (cptrack.cu)

inline int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(error_buffer(), 512, fmt, ap);
    va_end(ap);
    return code;
}

struct HostWeightTable {
    std::vector<double> w;
    uint32_t *d_thr = nullptr;
    int max_count = 0;
    int has_bounds = 0;
    int max_bound = 0;
    int linear_upto = 0;
    cpt::WeightTable device() const { return cpt::WeightTable{d_thr, max_count, has_bounds, max_bound, linear_upto}; }
};

}  // namespace cpt

#define CUDA_TRY(expr)                                                                               \
    do {                                                                                             \
        cudaError_t e_ = (expr);                                                                     \
        if (e_ != cudaSuccess) return cpt::fail(CPT_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(e_)); \
    } while (0)

namespace cpt {

// Grow-only owner of an array of T in device memory, or in pinned host memory when Pinned.  ensure(count) reallocates
// only when the capacity is too small.  It synchronises the whole device before it frees: the old memory may still be in
// use on the copy streams or on a caller's stream, not only on the context's stream.  The capacity is set only once the
// new allocation has succeeded: a failed ensure leaves no memory and a capacity of 0.
template <class T, bool Pinned = false>
class Grow {
  public:
    Grow() = default;
    Grow(const Grow &) = delete;
    Grow &operator=(const Grow &) = delete;
    ~Grow() { release(); }

    cudaError_t ensure(size_t count) {
        if (count <= cap_) return cudaSuccess;
        if (p_) {
            const cudaError_t e = cudaDeviceSynchronize();
            if (e != cudaSuccess) return e;
            release();
        }
        void *p = nullptr;
        const cudaError_t e = Pinned ? cudaHostAlloc(&p, count * sizeof(T), cudaHostAllocDefault) : cudaMalloc(&p, count * sizeof(T));
        if (e != cudaSuccess) return e;
        p_ = static_cast<T *>(p);
        cap_ = count;
        return cudaSuccess;
    }
    operator T *() const { return p_; }

  private:
    void release() {
        if (Pinned) cudaFreeHost(p_);
        else cudaFree(p_);
        p_ = nullptr;
        cap_ = 0;
    }
    T *p_ = nullptr;
    size_t cap_ = 0;
};

}  // namespace cpt

struct cpt_ctx {
    int device = 0;
    cpt::Geometry g{};
    cudaStream_t stream = nullptr;
    cudaStream_t own_stream = nullptr;
    cudaStream_t copy_stream = nullptr, d2h_stream = nullptr;
    int num_sms = 0;
    cpt::HostWeightTable tables[4];
    bool force_single = false;  // cpt_debug_force_single_kernel
    bool time_kernels = false;  // cpt_debug_kernel_times_ex
    bool timed_valid = false;
    cudaEvent_t ev_k[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    int *work_counter = nullptr;
    uint16_t *zero_frame = nullptr;
    long long *debug = nullptr;
    cudaEvent_t ev_h2d[2], ev_compute[2], ev_d2h[2];
    bool events = false;
    bool nlm_table_ready = false;  // cpt_nlm_denoise_u8 uploaded its weight table (constant memory of this device)

    // scratch and staging, grown on demand
    cpt::Grow<float> scratch;  // per-CTA images of regions-only launches of the single persistent kernel
    cpt::Grow<int8_t> qbytes;  // split plan: quad bytes
    cpt::Grow<cpt::StripRec> prec;  // split plan: strip pass records
    cpt::Grow<cpt::FrameHdr> fhdr;  // split plan: per-frame headers
    cpt::Grow<uint32_t> maskbits;  // split plan: thresholded masks between frame_regions_kernel and frame_components_kernel
    cpt::Grow<int> fallback;  // split plan: count, then the frames left to frame_components_kernel
    cpt::Grow<uint8_t> u8_frames[2];  // denoise passes: normalised / denoised images
    cpt::Grow<uint16_t> stage_frames[2];  // host-staged calls: input frames per buffer
    cpt::Grow<cpt_region> stage_regions[2];  // host-staged calls: region lists per buffer
    cpt::Grow<cpt_frame_info> stage_info[2];  // host-staged calls: frame records per buffer
    cpt::Grow<float> stage_filtered[2];  // host-staged calls that return the filtered images
    cpt::Grow<uint8_t> stage_labels[2];  // host-staged calls that return the label images
    cpt::Grow<float> scratch_filtered;  // filtered images of host-staged calls that do not return them
    cpt::Grow<cpt_clip> d_clips;  // host-staged calls: clip records rebased to their chunk
    cpt::Grow<uint8_t> pk_stream[2];  // packed host-staged call: payload bytes per buffer
    cpt::Grow<cpt_cptv_frame> pk_table[2];  // packed host-staged call: frame table rows per buffer
    cpt::Grow<cpt_cptv_frame, true> pk_h_table[2];  // packed host-staged call: the same rows, rebased on the host
    cpt::Grow<int32_t> pk_first[2];  // packed host-staged call: first row of each clip of the chunk
    cpt::Grow<int32_t, true> pk_h_first[2];  // packed host-staged call: the same, on the host
    cpt::Grow<int32_t> pk_change;  // packed host-staged call: the decoder's change images
    cpt::Grow<int32_t> cptv_scratch;  // cpt_cptv_decode: the decoder's change images
    cpt::Grow<uint8_t> detect_scratch;  // cpt_detect_objects / _batch: images, masks, union-find and component tables
    cpt::Grow<int> merge_order;  // cpt_ir_merge_components: list order of every frame of a launch
    cpt::Grow<uint8_t> motion_scratch;  // cpt_motion_clips: detector records, steps, mean rows, results, ring copies
    cpt::Grow<uint8_t> ir_clips_scratch;  // cpt_ir_motion_clips: clip records, flags, steps, results, staged host frames
};

