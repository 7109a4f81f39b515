// motion_kernels.cu -- CPTVMotionDetector.process_frame (piclassifier/cptvmotiondetector.py:74-205) as ONE launch
// per frame (M1 of SURVEY.md section 8a): batch-1 latency is the metric, so the running mean, the weighted
// background update and the motion count are fused into a single 1024-thread CTA and the host reads back one
// 32-byte result record.  motion_step_kernel (per frame) and motion_clips_kernel (recordings) both run motion_step:
//   phase 1  RunningMean.add (motiondetector.py:160-175): uint32 sum += new - oldest-in-ring (modular, as numpy)
//   phase 2  WeightedBackground.process_frame(sum / n) (motiondetector.py:197-244) unless FFC affected
//   phase 3  detect(): count(clip(cur, T) - clip(oldest_nonffc, T) > delta_thresh), T = background average
//            (cptvmotiondetector.py:74-120), with the optional second delta ring (one_diff_only False)
// The frame ring, the sum and the delta ring live in HBM for the life of the detector.
#include <algorithm>
#include <cstring>
#include <vector>

#include "background_step.cuh"
#include "cptrack_internal.cuh"

struct cpt_motion {
    cpt_ctx *ctx = nullptr;
    int ring_frames = 0, mean_frames = 0, diff_frames = 0, weight_slot = 0;
    uint16_t *d_ring = nullptr;     // [ring_frames][H][W]
    uint32_t *d_sum = nullptr;      // [H][W]
    double *d_diff = nullptr;       // [diff_frames][crop_h][crop_w]
    int32_t *d_mean_count = nullptr;
    cpt_motion_result *d_result = nullptr;
    cpt_motion_result *h_result = nullptr;  // pinned
    uint16_t *h_stage = nullptr;            // pinned frame
};

namespace cpt {

struct MotionShared {
    unsigned long long red_sum[32];
    int red_changed;
    int red_count[32];
    int error;
};

// One process_frame on the device: the three phases of the file comment for one frame.  `cur`, `old` (the ring's
// oldest frame, read when the running mean is full) and `nonffc` (the oldest non-FFC frame, read with
// CPT_MOTION_DETECT) may come from the ring or from a staged frame array.  `n` is RunningMean.running_mean_frames
// before the step; the new count is returned to every thread.  Every thread of the CTA must call; thread 0 writes
// *result.  Ends with a barrier, so a CTA may run steps back to back.
__device__ __forceinline__ int motion_phases(const Geometry &g, const uint16_t *cur, const uint16_t *old, const uint16_t *nonffc,
                                             uint32_t *sum, int n, int mean_frames, double *diff, int diff_slot_new,
                                             int diff_slot_old, uint8_t *bg_state, const WeightTable &wt, uint32_t flags,
                                             int delta_thresh, double init_average, MotionShared &sh,
                                             cpt_motion_result *result) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) sh.error = 0;
    __syncthreads();

    // ---- phase 1: running mean
    if (flags & CPT_MOTION_MEAN) {
        const bool restart = (flags & CPT_MOTION_MEAN_RESTART) || n == 0;
        const bool full = !restart && n == mean_frames;
        for (int i = tid; i < g.npx / 2; i += blockDim.x) {
            const uint32_t c2 = reinterpret_cast<const uint32_t *>(cur)[i];
            uint2 s = reinterpret_cast<uint2 *>(sum)[i];
            if (restart) {
                s.x = c2 & 0xffffu;
                s.y = c2 >> 16;
            } else {
                if (full) {  // `running_mean -= oldest; running_mean += new`, uint32 modular
                    const uint32_t o2 = reinterpret_cast<const uint32_t *>(old)[i];
                    s.x -= o2 & 0xffffu;
                    s.y -= o2 >> 16;
                }
                s.x += c2 & 0xffffu;
                s.y += c2 >> 16;
            }
            reinterpret_cast<uint2 *>(sum)[i] = s;
        }
        n = restart ? 1 : (full ? n : n + 1);
    }
    __syncthreads();

    // ---- phase 2: background from the running mean (np.int32(sum / n): truncation == floor division here)
    if ((flags & CPT_MOTION_BACKGROUND) && n > 0) {
        const uint32_t *S = sum;
        const uint32_t un = (uint32_t)n;
        int *err = &sh.error;
        background_step(g, bg_state, [S, un, err](int p) {
            const uint32_t v = S[p] / un;
            if (v > 65535u) { *err = 1; return 65535; }
            return (int)v;
        }, wt, sh.red_sum, &sh.red_changed);
    }

    // ---- phase 3: motion count against the oldest non-FFC frame
    int count = 0;
    const StateHeader *bg_hdr = reinterpret_cast<const StateHeader *>(bg_state);
    const double T = bg_hdr->initialised ? bg_hdr->average : init_average;
    if (flags & CPT_MOTION_DETECT) {
        const double dt = (double)delta_thresh;
        const bool warmer = flags & CPT_MOTION_WARMER_ONLY, one = flags & CPT_MOTION_ONE_DIFF;
        double *dnew = diff ? diff + (size_t)diff_slot_new * g.ncrop : nullptr;
        const double *dold = (diff && diff_slot_old >= 0) ? diff + (size_t)diff_slot_old * g.ncrop : nullptr;
        for (int i = tid; i < g.ncrop; i += blockDim.x) {
            const int y = i / g.crop_w + g.edge, x = i - (y - g.edge) * g.crop_w + g.edge;
            const int p = y * g.W + x;
            double d = fmax((double)cur[p], T) - fmax((double)nonffc[p], T);
            if (!warmer) d = fabs(d);
            if (one) {
                count += d > dt;
            } else {
                if (d >= dt) d = dt;
                if (dold) count += (dold[i] + d == 2.0 * dt);
                dnew[i] = d;
            }
        }
    }
    count = __reduce_add_sync(0xffffffffu, count);
    if (lane == 0) sh.red_count[warp] = count;
    __syncthreads();
    if (tid == 0) {
        int total = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) total += sh.red_count[w];
        cpt_motion_result r;
        r.average = T;
        r.diff = total;
        r.error = sh.error;
        r.mean_frames = n;
        r.reserved = 0;
        *result = r;
    }
    __syncthreads();
    return n;
}

// Per detector of a cpt_motion_clips launch, and the detector of a cpt_motion_step launch.
struct MotionClipArgs {
    uint16_t *ring;
    uint32_t *sum;
    double *diff;
    int32_t *mean_count;
    uint8_t *bg_state;
    WeightTable wt;
    double init_average;
    int delta_thresh, mean_frames, first_step, n_steps;
};

// A frame reference of cpt_motion_clip_step: row r >= 0 of the staged frames, or ring slot -1 - r as it stood before
// the launch (the ring is refreshed only after this kernel, by motion_ring_gather_kernel).
__device__ __forceinline__ const uint16_t *motion_frame(const uint16_t *frames, const uint16_t *ring, int npx, int ref) {
    return ref >= 0 ? frames + (size_t)ref * npx : ring + (size_t)(-1 - ref) * npx;
}

// One step of a detector, the one copy for both entry points: the RunningMean(frames, window) start from the step's mean
// rows (motiondetector.py:161-164) when it has any, then motion_phases.  `n` is the mean count before the step; returns
// the count after it.  Every thread of the CTA must call.
__device__ __forceinline__ int motion_step(const Geometry &g, const MotionClipArgs &c, const cpt_motion_clip_step &st,
                                           const int32_t *mean_rows, const uint16_t *frames, int n, MotionShared &sh,
                                           cpt_motion_result *result) {
    if (st.mean_count > 0) {
        for (int i = threadIdx.x; i < g.npx; i += blockDim.x) {
            uint32_t v = 0;
            for (int k = 0; k < st.mean_count; ++k) v += motion_frame(frames, c.ring, g.npx, mean_rows[st.mean_first + k])[i];
            c.sum[i] = v;
        }
        n = st.mean_count;
        __syncthreads();
    }
    return motion_phases(g, motion_frame(frames, c.ring, g.npx, st.frame), motion_frame(frames, c.ring, g.npx, st.oldest),
                         (st.flags & CPT_MOTION_DETECT) ? motion_frame(frames, c.ring, g.npx, st.nonffc) : nullptr, c.sum, n, c.mean_frames, c.diff, st.diff_slot_new,
                         st.diff_slot_old, c.bg_state, c.wt, st.flags, c.delta_thresh, c.init_average, sh, result);
}

// cpt_motion_clips: one CTA per detector walks that detector's steps in order, one cpt_motion_result per step.
__global__ void __launch_bounds__(1024, 1) motion_clips_kernel(const Geometry g, const MotionClipArgs *clips,
                                                               const cpt_motion_clip_step *steps, const int32_t *mean_rows,
                                                               const uint16_t *frames, cpt_motion_result *results) {
    __shared__ MotionShared sh;
    const MotionClipArgs c = clips[blockIdx.x];
    int n = *c.mean_count;
    for (int s = c.first_step; s < c.first_step + c.n_steps; ++s)  // each step record read once, into registers
        n = motion_step(g, c, cpt_motion_clip_step(steps[s]), mean_rows, frames, n, sh, results + s);
    if (threadIdx.x == 0) *c.mean_count = n;
}

// cpt_motion_step's records, passed by value: no upload besides the frame.  Every frame reference is a ring slot.
constexpr int kMotionStepMeanRows = 64;
struct MotionMeanRows { int32_t row[kMotionStepMeanRows]; };

__global__ void __launch_bounds__(1024, 1) motion_step_kernel(const Geometry g, const MotionClipArgs c, const cpt_motion_clip_step st,
                                                              const __grid_constant__ MotionMeanRows mean, cpt_motion_result *result) {
    __shared__ MotionShared sh;
    const int n = motion_step(g, c, st, mean.row, nullptr, *c.mean_count, sh, result);
    if (threadIdx.x == 0) *c.mean_count = n;
}

struct RingCopy {
    uint16_t *dst;
    int64_t row;
};

// After motion_clips_kernel: each listed ring slot takes the staged frame the per-frame loop would have left there.
__global__ void __launch_bounds__(256) motion_ring_gather_kernel(const RingCopy *copies, const uint16_t *frames, int npx) {
    const RingCopy c = copies[blockIdx.x];
    const uint32_t *src = reinterpret_cast<const uint32_t *>(frames + c.row * npx);
    uint32_t *dst = reinterpret_cast<uint32_t *>(c.dst);
    for (int i = threadIdx.x; i < npx / 2; i += blockDim.x) dst[i] = src[i];
}

}  // namespace cpt

using cpt::fail;

// The detector record of a step of either entry point: its handle on ctx c, its state record and its weight table.
static int motion_clip_args(cpt_ctx *c, const cpt_motion_clip &k, int d, cpt::MotionClipArgs &a) {
    const cpt_motion *m = k.m;
    if (!m || m->ctx != c) return fail(CPT_ERR_INVALID, "detector %d does not belong to this context", d);
    if (!k.d_background_state) return fail(CPT_ERR_INVALID, "detector %d has no background state", d);
    if (!c->tables[m->weight_slot].d_thr) return fail(CPT_ERR_INVALID, "weight table slot %d is not set", m->weight_slot);
    a = cpt::MotionClipArgs{m->d_ring, m->d_sum, m->d_diff, m->d_mean_count, (uint8_t *)k.d_background_state, c->tables[m->weight_slot].device(),
                            k.init_average, k.delta_thresh, m->mean_frames, k.first_step, k.n_steps};
    return CPT_OK;
}

// Step i of detector m, checked before anything runs: its frame references (r >= 0 a row of the call's n_frames frames,
// r < 0 ring slot -1 - r), delta-ring slots and the delta ring itself, and its mean rows in h_mean_rows[0 .. n_mean_rows).
static int motion_check_step(const cpt_motion *m, const cpt_motion_clip_step &st, int64_t n_frames, const int32_t *h_mean_rows,
                             int n_mean_rows, int i) {
    auto ref_ok = [&](int32_t r) { return r >= 0 ? r < n_frames : -1 - (int64_t)r < m->ring_frames; };
    if (!ref_ok(st.frame) || !ref_ok(st.oldest)) return fail(CPT_ERR_INVALID, "step %d: frame reference out of range", i);
    if (st.flags & CPT_MOTION_DETECT) {
        if (!ref_ok(st.nonffc)) return fail(CPT_ERR_INVALID, "step %d: oldest non-FFC reference out of range", i);
        if (!(st.flags & CPT_MOTION_ONE_DIFF)) {
            if (!m->d_diff) return fail(CPT_ERR_INVALID, "step %d: the detector was opened without a delta ring", i);
            if (st.diff_slot_new < 0 || st.diff_slot_new >= m->diff_frames || st.diff_slot_old >= m->diff_frames)
                return fail(CPT_ERR_INVALID, "step %d: delta ring slot out of range", i);
        }
    }
    if (st.mean_count < 0 || st.mean_count > m->mean_frames || st.mean_first < 0 || st.mean_count > n_mean_rows - st.mean_first)
        return fail(CPT_ERR_INVALID, "step %d: mean rows out of range", i);
    for (int j = 0; j < st.mean_count; ++j)
        if (!ref_ok(h_mean_rows[st.mean_first + j])) return fail(CPT_ERR_INVALID, "step %d: mean frame reference out of range", i);
    return CPT_OK;
}

extern "C" {

cpt_motion *cpt_motion_open(cpt_ctx *c, int ring_frames, int mean_frames, int diff_frames, int weight_slot) {
    if (!c || ring_frames < 1 || mean_frames < 1 || diff_frames < 0 || weight_slot < 0 || weight_slot >= 4) {
        fail(CPT_ERR_INVALID, "cpt_motion_open: bad argument");
        return nullptr;
    }
    if (!c->tables[weight_slot].d_thr) {
        fail(CPT_ERR_INVALID, "weight table slot %d is not set (cpt_set_weight_table)", weight_slot);
        return nullptr;
    }
    if (cudaSetDevice(c->device) != cudaSuccess) {
        fail(CPT_ERR_CUDA, "cudaSetDevice failed");
        return nullptr;
    }
    cpt_motion *m = new cpt_motion();
    m->ctx = c;
    m->ring_frames = ring_frames; m->mean_frames = mean_frames; m->diff_frames = diff_frames; m->weight_slot = weight_slot;
    const size_t npx = c->g.npx;
    bool ok = cudaMalloc(&m->d_ring, (size_t)ring_frames * npx * sizeof(uint16_t)) == cudaSuccess &&
              cudaMalloc(&m->d_sum, npx * sizeof(uint32_t)) == cudaSuccess &&
              cudaMalloc(&m->d_mean_count, sizeof(int32_t)) == cudaSuccess &&
              cudaMalloc(&m->d_result, sizeof(cpt_motion_result)) == cudaSuccess &&
              cudaHostAlloc(&m->h_result, sizeof(cpt_motion_result), cudaHostAllocDefault) == cudaSuccess &&
              cudaHostAlloc(&m->h_stage, npx * sizeof(uint16_t), cudaHostAllocDefault) == cudaSuccess;
    if (ok && diff_frames > 0) ok = cudaMalloc(&m->d_diff, (size_t)diff_frames * c->g.ncrop * sizeof(double)) == cudaSuccess;
    if (ok) {
        ok = cudaMemset(m->d_ring, 0, (size_t)ring_frames * npx * sizeof(uint16_t)) == cudaSuccess &&
             cudaMemset(m->d_sum, 0, npx * sizeof(uint32_t)) == cudaSuccess &&
             cudaMemset(m->d_mean_count, 0, sizeof(int32_t)) == cudaSuccess;
        if (ok && m->d_diff) ok = cudaMemset(m->d_diff, 0, (size_t)diff_frames * c->g.ncrop * sizeof(double)) == cudaSuccess;
    }
    if (!ok) {
        fail(CPT_ERR_NOMEM, "cpt_motion_open: allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
        cpt_motion_close(m);
        return nullptr;
    }
    return m;
}

void cpt_motion_close(cpt_motion *m) {
    if (!m) return;
    cudaSetDevice(m->ctx->device);
    cudaStreamSynchronize(m->ctx->stream);
    cudaFree(m->d_ring);
    cudaFree(m->d_sum);
    cudaFree(m->d_diff);
    cudaFree(m->d_mean_count);
    cudaFree(m->d_result);
    cudaFreeHost(m->h_result);
    cudaFreeHost(m->h_stage);
    delete m;
}

int cpt_motion_store(cpt_motion *m, const uint16_t *h_pix, int slot) {
    if (!m || !h_pix) return fail(CPT_ERR_INVALID, "null argument");
    if (slot < 0 || slot >= m->ring_frames) return fail(CPT_ERR_INVALID, "ring slot %d out of range", slot);
    cpt_ctx *c = m->ctx;
    CUDA_TRY(cudaSetDevice(c->device));
    const size_t bytes = (size_t)c->g.npx * sizeof(uint16_t);
    CUDA_TRY(cudaStreamSynchronize(c->stream));  // the staging buffer is free again
    memcpy(m->h_stage, h_pix, bytes);
    CUDA_TRY(cudaMemcpyAsync(m->d_ring + (size_t)slot * c->g.npx, m->h_stage, bytes, cudaMemcpyHostToDevice, c->stream));
    return CPT_OK;
}

int cpt_motion_step(const cpt_motion_clip *h_clip, const uint16_t *h_pix, const cpt_motion_clip_step *h_step, const int32_t *h_mean_rows,
                    int n_mean_rows, cpt_motion_result *h_result) {
    if (!h_clip || !h_clip->m || !h_pix || !h_step || !h_result || (n_mean_rows > 0 && !h_mean_rows))
        return fail(CPT_ERR_INVALID, "null argument");
    if (n_mean_rows < 0 || n_mean_rows > cpt::kMotionStepMeanRows) return fail(CPT_ERR_INVALID, "bad mean row count %d", n_mean_rows);
    cpt_motion *m = h_clip->m;
    cpt_ctx *c = m->ctx;
    cpt::MotionClipArgs a;
    int rc = motion_clip_args(c, *h_clip, 0, a);
    if (!rc) rc = motion_check_step(m, *h_step, 0, h_mean_rows, n_mean_rows, 0);
    if (!rc) rc = cpt_motion_store(m, h_pix, -1 - h_step->frame);
    if (rc) return rc;
    cpt::MotionMeanRows mean{};
    std::copy(h_mean_rows, h_mean_rows + n_mean_rows, mean.row);
    cpt::motion_step_kernel<<<1, 1024, 0, c->stream>>>(c->g, a, *h_step, mean, m->d_result);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(m->h_result, m->d_result, sizeof(cpt_motion_result), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    *h_result = *m->h_result;
    if (h_result->error) return fail(CPT_ERR_INVALID, "running mean left the uint16 range (inconsistent ring / mean window)");
    return CPT_OK;
}

int cpt_motion_clips(cpt_ctx *c, const cpt_motion_clip *h_clips, int n, const uint16_t *d_frames, int64_t n_frames,
                     const cpt_motion_clip_step *h_steps, int n_steps, const int32_t *h_mean_rows, int n_mean_rows,
                     cpt_motion_result *h_results) {
    if (!c || n < 0 || n_frames < 0 || n_steps < 0 || n_mean_rows < 0) return fail(CPT_ERR_INVALID, "cpt_motion_clips: bad argument");
    if ((n && !h_clips) || (n_frames && !d_frames) || (n_steps && (!h_steps || !h_results)) || (n_mean_rows && !h_mean_rows))
        return fail(CPT_ERR_INVALID, "cpt_motion_clips: null argument");
    std::vector<cpt::MotionClipArgs> args(n);
    std::vector<cpt::RingCopy> copies;
    for (int d = 0; d < n; ++d) {
        const cpt_motion_clip &k = h_clips[d];
        int rc = motion_clip_args(c, k, d, args[d]);
        if (rc) return rc;
        const cpt_motion *m = k.m;
        for (int e = 0; e < d; ++e)
            if (h_clips[e].m == m || h_clips[e].d_background_state == k.d_background_state)
                return fail(CPT_ERR_INVALID, "cpt_motion_clips: detectors %d and %d share a handle or a state record", e, d);
        if (k.first_step < 0 || k.n_steps < 0 || k.n_steps > n_steps - k.first_step)
            return fail(CPT_ERR_INVALID, "cpt_motion_clips: detector %d: steps out of range", d);
        for (int i = k.first_step; i < k.first_step + k.n_steps; ++i)
            if ((rc = motion_check_step(m, h_steps[i], n_frames, h_mean_rows, n_mean_rows, i))) return rc;
        for (int s = 0; k.ring_rows && s < m->ring_frames; ++s) {
            const int32_t r = k.ring_rows[s];
            if (r < -1 || r >= n_frames) return fail(CPT_ERR_INVALID, "detector %d: ring row out of range", d);
            if (r >= 0) copies.push_back({m->d_ring + (size_t)s * c->g.npx, r});
        }
    }
    if (n == 0) return CPT_OK;
    CUDA_TRY(cudaSetDevice(c->device));
    // one scratch block: detector records | steps | mean rows | results | ring copies, each 256-byte aligned
    auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t o_steps = up(sizeof(cpt::MotionClipArgs) * n), o_mean = o_steps + up(sizeof(cpt_motion_clip_step) * n_steps),
                 o_res = o_mean + up(sizeof(int32_t) * n_mean_rows), o_copy = o_res + up(sizeof(cpt_motion_result) * n_steps),
                 total = o_copy + up(sizeof(cpt::RingCopy) * copies.size());
    CUDA_TRY(c->motion_scratch.ensure(total));
    uint8_t *base = c->motion_scratch;
    auto *d_args = reinterpret_cast<cpt::MotionClipArgs *>(base);
    auto *d_steps = reinterpret_cast<cpt_motion_clip_step *>(base + o_steps);
    auto *d_mean = reinterpret_cast<int32_t *>(base + o_mean);
    auto *d_res = reinterpret_cast<cpt_motion_result *>(base + o_res);
    auto *d_copy = reinterpret_cast<cpt::RingCopy *>(base + o_copy);
    CUDA_TRY(cudaMemcpyAsync(d_args, args.data(), sizeof(cpt::MotionClipArgs) * n, cudaMemcpyHostToDevice, c->stream));
    if (n_steps) CUDA_TRY(cudaMemcpyAsync(d_steps, h_steps, sizeof(cpt_motion_clip_step) * n_steps, cudaMemcpyHostToDevice, c->stream));
    if (n_mean_rows) CUDA_TRY(cudaMemcpyAsync(d_mean, h_mean_rows, sizeof(int32_t) * n_mean_rows, cudaMemcpyHostToDevice, c->stream));
    if (!copies.empty())
        CUDA_TRY(cudaMemcpyAsync(d_copy, copies.data(), sizeof(cpt::RingCopy) * copies.size(), cudaMemcpyHostToDevice, c->stream));
    cpt::motion_clips_kernel<<<n, 1024, 0, c->stream>>>(c->g, d_args, d_steps, d_mean, d_frames, d_res);
    CUDA_TRY(cudaGetLastError());
    if (!copies.empty()) {  // stream order: the ring changes only after every step has read it
        cpt::motion_ring_gather_kernel<<<(unsigned)copies.size(), 256, 0, c->stream>>>(d_copy, d_frames, c->g.npx);
        CUDA_TRY(cudaGetLastError());
    }
    if (n_steps) CUDA_TRY(cudaMemcpyAsync(h_results, d_res, sizeof(cpt_motion_result) * n_steps, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));  // the host vectors above and the scratch block are free again
    return CPT_OK;
}

}  // extern "C"
