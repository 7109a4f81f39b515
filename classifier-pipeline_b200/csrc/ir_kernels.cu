// ir_kernels.cu -- the device half of IRMotionDetector.process_frame (piclassifier/irmotiondetector.py:103-153) for
// 640x480 BGR frames: grey conversion, |oldest - current| > 12, erosion with a k x k box and the count of surviving pixels
// (for the frame difference and for the foreground mask of the background model), per frame and for whole clips.
//   bgr_to_gray_kernel   cv2.cvtColor(BGR2GRAY) in OpenCV's 8-bit fixed point
//   ir_pack_kernel       cv2.absdiff + cv2.threshold(THRESH_BINARY) and the foreground mask, as bit planes (one warp per
//                        32-pixel word)
//   ir_frame_kernel      whole clips, one step of every clip: grey into the ring, the difference bit, the MOG2 update
//                        (mog2.cuh) with the rate the clip's movement flag selects, the mask byte and its bit
//   ir_erode_kernel      erosion with a k x k box (anchor k / 2, pixels outside the image count as set) and the count of
//                        surviving pixels of both bit planes; its last CTA per clip applies the trigger rule
// and the rectangle merging of the IR tracker's detection half for a batch of frames:
//   ir_merge_kernel      track/irtrackextractor.py merge_components on every frame's stats rows, one warp per frame
#include <algorithm>
#include <vector>

#include "mog2.cuh"

namespace cpt {

constexpr int kErodeBand = 32;    // output rows per CTA of ir_erode_kernel (8 warps x 4 rows)
constexpr int kErodeWords = 32;   // 32-pixel words per CTA row: one per lane
constexpr int kErodeMaxK = 64;    // largest erosion box

// One clip of an ir_frame_kernel / ir_erode_kernel launch, constant during the call.
struct IrClipArgs {
    uint8_t *ring;    // [ring_frames][H][W] grey
    float *state;     // the MOG2 state (mog2.cuh)
    uint8_t *mask;    // [H][W] foreground mask, 0 / 255
    uint32_t *bits;   // [2][H][words per row]: difference and foreground bit planes
    Mog2Consts c;
    int first_step, n_steps;
};
// What a clip carries from step to step: the decision state and the erosion kernel's accumulators and ticket.
struct IrClipFlag {
    int movement, triggered;
    int diff, mask;
    unsigned ticket;
    int reserved[3];
};
// One step on the device: alpha / prune [0] with learning rate -1, [1] with learning rate 0 (the clip is recording).
struct IrStep {
    const uint8_t *bgr;
    int slot_new, slot_oldest, detect, fresh;
    float alpha[2], prune[2];
};
struct IrRule {
    int threshold, trigger_frames, max_triggered, erode_idle, erode_recording;
    int decide;  // 0: counts only (cpt_ir_motion_detect)
};

__device__ __forceinline__ uint8_t bgr_to_gray(const uint8_t *p) {
    return (uint8_t)((p[0] * 3735 + p[1] * 19235 + p[2] * 9798 + (1 << 14)) >> 15);
}

__device__ __forceinline__ bool ir_changed(int oldest, int gray, int threshold) { return abs(oldest - gray) > threshold; }

__global__ void __launch_bounds__(256) bgr_to_gray_kernel(const uint8_t *bgr, int n, uint8_t *gray) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) gray[i] = bgr_to_gray(bgr + 3 * i);
}

// Bit planes: word w of row y holds columns 32w .. 32w + 31 (bit i = column 32w + i); columns right of the image are set.
__global__ void __launch_bounds__(256) ir_pack_kernel(const uint8_t *__restrict__ oldest, const uint8_t *__restrict__ gray,
                                                      const uint8_t *__restrict__ mask, int W, int H, int wpr, int threshold,
                                                      uint32_t *__restrict__ bits) {
    const int word = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (word >= H * wpr) return;  // whole warps
    const int y = word / wpr, x = (word - y * wpr) * 32 + lane;
    bool changed = true, fg = true;
    if (x < W) {
        const int64_t p = (int64_t)y * W + x;
        changed = ir_changed(oldest[p], gray[p], threshold);
        fg = mask && mask[p] != 0;
    }
    const unsigned dw = __ballot_sync(0xffffffffu, changed), mw = __ballot_sync(0xffffffffu, fg);
    if (lane == 0) {
        bits[word] = dw;
        if (mask) bits[(size_t)H * wpr + word] = mw;
    }
}

// One step of every clip c0 + blockIdx.y that has a step j: one thread per pixel, one warp per 32-pixel word.
__global__ void __launch_bounds__(256) ir_frame_kernel(const IrClipArgs *__restrict__ clips, const IrClipFlag *__restrict__ flags,
                                                       const IrStep *__restrict__ steps, int j, int c0, int W, int H, int wpr,
                                                       int threshold) {
    const int ci = c0 + blockIdx.y;
    const IrClipArgs &k = clips[ci];
    if (j >= k.n_steps) return;
    const IrStep &s = steps[k.first_step + j];
    const int word = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (word >= H * wpr) return;  // whole warps
    const int y = word / wpr, x = (word - y * wpr) * 32 + lane;
    const int64_t npx = (int64_t)W * H;
    bool changed = true, fg = true;  // columns right of the image count as set, as cv2.erode's border
    if (x < W) {
        const int64_t p = (int64_t)y * W + x;
        const uint8_t g = bgr_to_gray(s.bgr + 3 * p);
        // a ring of one frame compares the new grey frame with itself, as the per-frame calls do
        const uint8_t old = s.slot_oldest == s.slot_new ? g : k.ring[s.slot_oldest * npx + p];
        k.ring[s.slot_new * npx + p] = g;
        changed = ir_changed(old, g, threshold);
        const int rec = flags[ci].movement != 0;
        float w[kMog2Modes], v[kMog2Modes], m[kMog2Modes];
        int nmodes;
        mog2_load(k.state, npx, p, s.fresh, w, v, m, nmodes);
        const int bg = mog2_pixel(w, v, m, nmodes, (float)g, s.alpha[rec], s.prune[rec], k.c);
        mog2_store(k.state, npx, p, w, v, m, nmodes);
        k.mask[p] = bg ? 0 : 255;
        fg = !bg;
    }
    const unsigned dw = __ballot_sync(0xffffffffu, changed), mw = __ballot_sync(0xffffffffu, fg);
    if (s.detect && lane == 0) {
        k.bits[word] = dw;
        k.bits[(size_t)H * wpr + word] = mw;
    }
}

// Word w of a row eroded horizontally: bit i is set iff input columns 32w + i - a .. 32w + i - a + ek - 1 are all set.
// Words outside the row count as set.  The window of the word spans at most four input words (ek <= 64).
__device__ __forceinline__ uint32_t erode_row_word(const uint32_t *__restrict__ row, int wpr, int w, int ek, int a) {
    const int p0 = 32 * w - a, q0 = p0 >> 5;  // floor
    uint32_t in0, in1, in2, in3;
    {
        const int q = q0;
        in0 = q < 0 || q >= wpr ? ~0u : row[q];
        in1 = q + 1 < 0 || q + 1 >= wpr ? ~0u : row[q + 1];
        in2 = q + 2 < 0 || q + 2 >= wpr ? ~0u : row[q + 2];
        in3 = q + 3 < 0 || q + 3 >= wpr ? ~0u : row[q + 3];
    }
    uint32_t out = ~0u;
    for (int d = 0; d < ek; ++d) {
        const int p = p0 + d, rel = (p >> 5) - q0;
        const uint32_t lo = rel == 0 ? in0 : rel == 1 ? in1 : in2;
        const uint32_t hi = rel == 0 ? in1 : rel == 1 ? in2 : in3;
        out &= __funnelshift_r(lo, hi, p & 31);
    }
    return out;
}

// Erosion and count of the bit planes of every clip c0 + blockIdx.y that has a step j; a CTA takes kErodeBand rows and
// kErodeWords words of them, plus ek - 1 halo rows.  The box is erode_recording while the clip's movement flag is set,
// erode_idle otherwise.  The counts add up in the clip's IrClipFlag; the CTA that takes the clip's last ticket writes the
// step's result and, with rule.decide, applies the trigger rule to the clip's flag (irmotiondetector.py:120-139).  A step
// without detect gets its result from the first CTA and changes nothing.
__global__ void __launch_bounds__(256) ir_erode_kernel(const IrClipArgs *__restrict__ clips, IrClipFlag *flags,
                                                       const IrStep *__restrict__ steps, int j, int c0, int W, int H, int wpr,
                                                       int n_planes, IrRule rule, cpt_ir_motion_clip_result *__restrict__ results) {
    const int ci = c0 + blockIdx.y;
    const IrClipArgs &k = clips[ci];
    if (j >= k.n_steps) return;
    IrClipFlag &f = flags[ci];
    cpt_ir_motion_clip_result *res = results + k.first_step + j;
    const int rec = *(volatile int *)&f.movement;
    if (!steps[k.first_step + j].detect) {
        if (blockIdx.x == 0 && threadIdx.x == 0) *res = cpt_ir_motion_clip_result{rec, f.triggered, -1, -1};
        return;
    }
    __shared__ uint32_t rows[2][kErodeBand + kErodeMaxK - 1][kErodeWords];
    __shared__ int block_count[2];
    const int ek = rec ? rule.erode_recording : rule.erode_idle, a = ek / 2;
    const int tiles_x = (wpr + kErodeWords - 1) / kErodeWords;
    const int y0 = (blockIdx.x / tiles_x) * kErodeBand, lane = threadIdx.x & 31, tr = threadIdx.x >> 5;
    const int w = (blockIdx.x % tiles_x) * kErodeWords + lane;
    if (threadIdx.x < 2) block_count[threadIdx.x] = 0;
#pragma unroll
    for (int pl = 0; pl < 2; ++pl) {
        if (pl >= n_planes) break;
        const uint32_t *plane = k.bits + (size_t)pl * H * wpr;
        for (int r = tr; r < kErodeBand + ek - 1; r += 8) {
            const int y = y0 - a + r;
            rows[pl][r][lane] = y < 0 || y >= H || w >= wpr ? ~0u : erode_row_word(plane + (size_t)y * wpr, wpr, w, ek, a);
        }
    }
    __syncthreads();
    int count[2] = {0, 0};
    if (w < wpr) {
        const uint32_t valid = 32 * (w + 1) <= W ? ~0u : (1u << (W - 32 * w)) - 1u;
        for (int r = tr; r < kErodeBand && y0 + r < H; r += 8) {
#pragma unroll
            for (int pl = 0; pl < 2; ++pl) {
                if (pl >= n_planes) break;
                uint32_t v = ~0u;
                for (int d = 0; d < ek; ++d) v &= rows[pl][r + d][lane];
                count[pl] += __popc(v & valid);
            }
        }
    }
#pragma unroll
    for (int pl = 0; pl < 2; ++pl) {
        const int s = __reduce_add_sync(0xffffffffu, count[pl]);
        if (lane == 0 && s) atomicAdd(&block_count[pl], s);
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    if (block_count[0]) atomicAdd(&f.diff, block_count[0]);
    if (block_count[1]) atomicAdd(&f.mask, block_count[1]);
    __threadfence();
    if (atomicAdd(&f.ticket, 1u) != gridDim.x - 1) return;
    // the last CTA of the clip: every other CTA's counts are in
    __threadfence();
    const int diff = atomicExch(&f.diff, 0), mask = atomicExch(&f.mask, 0);
    f.ticket = 0;
    int trig = f.triggered, mov = rec;
    if (rule.decide) {
        // with the background frozen while motion lasts, the frame difference bounds the mask count
        const int m = rec ? min(diff, mask) : mask;
        trig = m > 0 ? min(trig + 1, rule.max_triggered) : max(trig - 1, 0);
        if (!rec && trig >= rule.trigger_frames) mov = 1;
        else if (rec && trig <= 0) mov = 0;
        f.triggered = trig;
        f.movement = mov;
    }
    *res = cpt_ir_motion_clip_result{mov, trig, diff, mask};
}

// CTAs per clip of ir_erode_kernel
inline int erode_ctas(int H, int wpr) { return ((H + kErodeBand - 1) / kErodeBand) * ((wpr + kErodeWords - 1) / kErodeWords); }

// merge_components' pair test (track/irtrackextractor.py): rect a = the scanning rectangle, b = the other one.  The squared
// distance wraps in 32 bits as numpy's int32 arithmetic on the stats rows does.
__device__ __forceinline__ bool ir_rects_merge(int ax, int ay, int aw, int ah, int bx, int by, int bw, int bh, double max_gap) {
    bool within = false;
    if (bw + aw > max(bx + bw, aw + ax) - min(bx, ax)) within = bh + ah > max(by + bh, ay + ah) - min(by, ay);
    int x1 = 0, x2 = 0, y1 = 0, y2 = 0;
    if (aw + bw > max(ax + aw, bw + bx) - min(ax, bx)) {
    } else if (ax < bx) {
        x1 = ax + aw; x2 = bx;
    } else {
        x1 = bx + bw; x2 = ax;
    }
    if (ah + bh > max(ay + ah, by + bh) - min(ay, by)) {
    } else if (ay < by) {
        y1 = ay + ah; y2 = by;
    } else {
        y1 = by + bh; y2 = ay;
    }
    const unsigned dx = (unsigned)(x1 - x2), dy = (unsigned)(y1 - y2);
    const int d2 = (int)(dx * dx + dy * dy);
    return sqrt((double)d2) < max_gap || within;
}

// One warp per frame.  stats [frame][max_components + 1][5] with row 0 the background, counts = cv2's label count.  The
// list lives in the frame's output rows (merged, [max_components][5]) and in order[max_components] (the label of each list
// position; negative once deleted), so no list length is too long: every step is a warp-wide pass over the list, 32
// positions at a time.  A deletion only marks the position, which keeps the survivors in the order the Python list keeps
// them.
__global__ void __launch_bounds__(128) ir_merge_kernel(const int32_t *stats, const int32_t *counts, int n_frames, int max_components,
                                                       int min_mass, int min_size, double max_gap, int *order, int32_t *merged,
                                                       int32_t *merged_counts) {
    const int f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (f >= n_frames) return;  // whole warps
    const unsigned below = (1u << lane) - 1u;
    const int n = counts[f];
    if (n < 1 || n - 1 > max_components) {  // overflowed: the list is truncated, never merge it
        if (lane == 0) merged_counts[f] = -1;
        return;
    }
    stats += (size_t)f * ((size_t)max_components + 1) * 5;
    merged += (size_t)f * (size_t)max_components * 5;
    int *ord = order + (size_t)f * max_components;
    // filter, in label order
    int m = 0;
    for (int b = 0; b < n - 1; b += 32) {
        const int l = b + lane + 1;
        bool keep = false;
        if (l < n) {
            const int32_t *r = stats + l * 5;
            keep = r[4] > min_mass || (r[2] > min_size && r[3] > min_size);
        }
        const unsigned k = __ballot_sync(0xffffffffu, keep);
        if (keep) ord[m + __popc(k & below)] = l;
        m += __popc(k);
    }
    __syncwarp();
    // stable sort by area, descending: the rank counts larger areas and equal areas earlier in the list
    for (int b = 0; b < m; b += 32) {
        const int i = b + lane;
        if (i < m) {
            const int li = ord[i], ai = stats[li * 5 + 4];
            int rank = 0;
            for (int j = 0; j < m; ++j) {
                const int aj = stats[ord[j] * 5 + 4];
                rank += aj > ai || (aj == ai && j < i);
            }
            merged[rank * 5] = li;
        }
    }
    __syncwarp();
    for (int p = lane; p < m; p += 32) {
        const int l = merged[p * 5];
        ord[p] = l;
        for (int k = 0; k < 5; ++k) merged[p * 5 + k] = stats[l * 5 + k];
    }
    __syncwarp();
    // the scan: the current rectangle's original against every live original; merges fold in list order
    int cur = 0;
    while (cur < m) {
        const int32_t *rc = stats + ord[cur] * 5;
        const int rx = rc[0], ry = rc[1], rw = rc[2], rh = rc[3];
        int mx = merged[cur * 5], my = merged[cur * 5 + 1], mw = merged[cur * 5 + 2], mh = merged[cur * 5 + 3], ma = merged[cur * 5 + 4];
        bool any = false;
        for (int b = 0; b < m; b += 32) {
            const int p = b + lane;
            const int l = p < m ? ord[p] : 0;
            int x2 = 0, y2 = 0, w2 = 0, h2 = 0, a2 = 0;
            bool hit = false;
            if (l > 0) {
                const int32_t *r2 = stats + l * 5;
                x2 = r2[0]; y2 = r2[1]; w2 = r2[2]; h2 = r2[3]; a2 = r2[4];
                hit = x2 != rx && ir_rects_merge(rx, ry, rw, rh, x2, y2, w2, h2, max_gap);
            }
            unsigned hits = __ballot_sync(0xffffffffu, hit);
            any |= hits != 0;
            if (hit) ord[p] = -l;
            while (hits) {
                const int k = __ffs(hits) - 1;
                hits &= hits - 1;
                const int X = __shfl_sync(0xffffffffu, x2, k), Y = __shfl_sync(0xffffffffu, y2, k);
                const int W2 = __shfl_sync(0xffffffffu, w2, k), H2 = __shfl_sync(0xffffffffu, h2, k), A2 = __shfl_sync(0xffffffffu, a2, k);
                const int cur_right = mx + mw;
                mx = min(mx, X);
                my = min(my, Y);
                mw = max(cur_right, X + W2) - mx;
                mh = max(my + mh, Y + H2) - my;  // the bottom edge from the updated y, as the reference writes it
                ma += A2;
            }
        }
        if (any && lane == 0) {
            merged[cur * 5] = mx; merged[cur * 5 + 1] = my; merged[cur * 5 + 2] = mw; merged[cur * 5 + 3] = mh; merged[cur * 5 + 4] = ma;
        }
        __syncwarp();
        // a merge restarts the scan at the first live rectangle, otherwise it moves to the next live one
        const int start = any ? 0 : cur + 1;
        cur = m;
        for (int b = start; b < m; b += 32) {
            const int p = b + lane;
            const unsigned live = __ballot_sync(0xffffffffu, p < m && ord[p] > 0);
            if (live) {
                cur = b + __ffs(live) - 1;
                break;
            }
        }
    }
    // compact the live rows in place (a row only moves down, and a chunk is read before it is written)
    int out = 0;
    for (int b = 0; b < m; b += 32) {
        const int p = b + lane;
        const bool live = p < m && ord[p] > 0;
        int row[5];
        if (live)
            for (int k = 0; k < 5; ++k) row[k] = merged[p * 5 + k];
        const unsigned lv = __ballot_sync(0xffffffffu, live);
        __syncwarp();
        if (live)
            for (int k = 0; k < 5; ++k) merged[(out + __popc(lv & below)) * 5 + k] = row[k];
        out += __popc(lv);
        __syncwarp();
    }
    if (lane == 0) merged_counts[f] = out;
}

}  // namespace cpt

using cpt::fail;

// The leading members (ctx, W, H, ring_frames, d_ring) are read through the handle's address (native.py, _IrMotionHead);
// keep their order.
struct cpt_ir_motion {
    cpt_ctx *ctx;
    int W, H, ring_frames;
    uint8_t *d_ring;   // [ring_frames][H][W] grey
    uint8_t *d_bgr;    // [H][W][3] BGR, then at ir_records_offset cpt_ir_motion_step's IrStepRecords and cpt_ir_motion_detect's
    uint8_t *d_in_mask;
    uint32_t *d_bits;  // [2][H][words per row]: bit planes of the difference and of the foreground mask
    struct IrStepRecords *d_detect;  // the one-clip, one-step records of cpt_ir_motion_detect's ir_erode_kernel, set at open
    uint8_t *h_pin;  // pinned staging laid out as d_bgr: BGR and records in; grey, counts and records out
};

// A one-clip, one-step launch's records (cpt_ir_motion_step's go up with the frame; flag and result come back together).
struct IrStepRecords {
    cpt::IrClipArgs args;
    cpt::IrStep step;
    cpt::IrClipFlag flag;
    cpt_ir_motion_clip_result result;
};
static_assert(offsetof(IrStepRecords, result) == offsetof(IrStepRecords, flag) + sizeof(cpt::IrClipFlag), "flag, then result");
static size_t ir_records_offset(size_t npx) { return (3 * npx + 255) & ~(size_t)255; }

static int ir_check_params(const cpt_ir_motion_clip_params *p) {
    if (p->erode_idle < 1 || p->erode_idle > cpt::kErodeMaxK || p->erode_recording < 1 || p->erode_recording > cpt::kErodeMaxK)
        return fail(CPT_ERR_INVALID, "erosion boxes must be 1..64 pixels");
    return CPT_OK;
}

// Clip d: both handles on ctx c, of the call's W x H geometry (W == 0: clip d sets it), and a mask buffer.
static int ir_check_clip(cpt_ctx *c, const cpt_ir_motion_clip &k, int d, int &W, int &H) {
    const cpt_ir_motion *m = k.m;
    const cpt_mog2 *g = k.mog2;
    if (!m || !g || m->ctx != c || g->ctx != c) return fail(CPT_ERR_INVALID, "clip %d: a handle is missing or belongs to another context", d);
    if (W == 0) { W = m->W; H = m->H; }
    if (m->W != W || m->H != H || g->W != W || g->H != H)
        return fail(CPT_ERR_INVALID, "clip %d: the handles do not share one %d x %d geometry", d, W, H);
    if (!k.d_mask) return fail(CPT_ERR_INVALID, "clip %d has no mask buffer", d);
    return CPT_OK;
}

static int ir_check_slots(const cpt_ir_motion *m, const cpt_ir_motion_clip_step &st, int i) {
    if (st.slot_new < 0 || st.slot_new >= m->ring_frames || st.slot_oldest < 0 || st.slot_oldest >= m->ring_frames)
        return fail(CPT_ERR_INVALID, "step %d: ring slot out of range", i);
    return CPT_OK;
}

// The device records of clip k and of its steps h_steps[k.first_step .. + k.n_steps), all but each step's frame address:
// each step's rate pair of both learning rates it may take, from cv2's rule (mog2.cuh), with the model's frame count
// advanced once per step.
static void ir_clip_records(const cpt_ir_motion_clip &k, const cpt_ir_motion_clip_step *h_steps, cpt::IrClipArgs &args,
                            cpt::IrClipFlag &flag, cpt::IrStep *steps) {
    args = cpt::IrClipArgs{k.m->d_ring, k.mog2->d_state, k.d_mask, k.m->d_bits, k.mog2->c, k.first_step, k.n_steps};
    flag = cpt::IrClipFlag{k.movement != 0, k.triggered, 0, 0, 0u, {0, 0, 0}};
    for (int i = k.first_step; i < k.first_step + k.n_steps; ++i) {
        const cpt_ir_motion_clip_step &st = h_steps[i];
        cpt::IrStep &s = steps[i];
        s.slot_new = st.slot_new; s.slot_oldest = st.slot_oldest; s.detect = st.detect != 0;
        s.fresh = cpt::mog2_reinitialises(k.mog2->nframes, -1.0);
        int frozen = k.mog2->nframes;
        cpt::mog2_next_rate(*k.mog2, frozen, 0.0, s.alpha[1], s.prune[1]);
        cpt::mog2_next_rate(*k.mog2, k.mog2->nframes, -1.0, s.alpha[0], s.prune[0]);
    }
}

extern "C" {

cpt_ir_motion *cpt_ir_motion_open(cpt_ctx *c, int width, int height, int ring_frames) {
    if (!c || width < 1 || height < 1 || ring_frames < 1 || (long long)width * height > (1ll << 24)) {
        fail(CPT_ERR_INVALID, "bad IR motion detector geometry");
        return nullptr;
    }
    if (cudaSetDevice(c->device) != cudaSuccess) {
        fail(CPT_ERR_CUDA, "cudaSetDevice failed");
        return nullptr;
    }
    cpt_ir_motion *m = new cpt_ir_motion();
    m->ctx = c; m->W = width; m->H = height; m->ring_frames = ring_frames;
    const size_t n = (size_t)width * height, wpr = (width + 31) / 32;
    const size_t stage = ir_records_offset(n) + sizeof(IrStepRecords);
    if (cudaMalloc(&m->d_bgr, stage + sizeof(IrStepRecords)) != cudaSuccess || cudaMalloc(&m->d_ring, n * ring_frames) != cudaSuccess ||
        cudaMalloc(&m->d_in_mask, n) != cudaSuccess || cudaMalloc(&m->d_bits, 2 * height * wpr * sizeof(uint32_t)) != cudaSuccess ||
        cudaHostAlloc((void **)&m->h_pin, stage, cudaHostAllocDefault) != cudaSuccess) {
        fail(CPT_ERR_NOMEM, "IR motion detector allocation failed");
        cpt_ir_motion_close(m);
        return nullptr;
    }
    m->d_detect = reinterpret_cast<IrStepRecords *>(m->d_bgr + stage);
    IrStepRecords detect{};
    detect.args.bits = m->d_bits;
    detect.args.n_steps = 1;
    detect.step.detect = 1;
    if (cudaMemset(m->d_ring, 0, n * ring_frames) != cudaSuccess ||
        cudaMemcpy(m->d_detect, &detect, sizeof(detect), cudaMemcpyHostToDevice) != cudaSuccess) {
        fail(CPT_ERR_CUDA, "IR motion detector initialisation failed");
        cpt_ir_motion_close(m);
        return nullptr;
    }
    return m;
}

void cpt_ir_motion_close(cpt_ir_motion *m) {
    if (!m) return;
    cudaSetDevice(m->ctx->device);
    cudaStreamSynchronize(m->ctx->stream);
    cudaFree(m->d_bgr); cudaFree(m->d_ring); cudaFree(m->d_in_mask); cudaFree(m->d_bits);
    cudaFreeHost(m->h_pin);
    delete m;
}

int cpt_ir_motion_gray(cpt_ir_motion *m, const uint8_t *h_bgr, int slot_new, uint8_t *h_gray_out) {
    if (!m || !h_bgr) return fail(CPT_ERR_INVALID, "null argument");
    if (slot_new < 0 || slot_new >= m->ring_frames) return fail(CPT_ERR_INVALID, "ring slot out of range");
    cpt_ctx *c = m->ctx;
    CUDA_TRY(cudaSetDevice(c->device));
    const int n = m->W * m->H;
    CUDA_TRY(cudaStreamSynchronize(c->stream));  // without h_gray_out the previous frame's copy from h_pin may still run
    memcpy(m->h_pin, h_bgr, 3 * (size_t)n);
    CUDA_TRY(cudaMemcpyAsync(m->d_bgr, m->h_pin, 3 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    uint8_t *gray = m->d_ring + (size_t)slot_new * n;
    cpt::bgr_to_gray_kernel<<<(n + 255) / 256, 256, 0, c->stream>>>(m->d_bgr, n, gray);
    CUDA_TRY(cudaGetLastError());
    if (h_gray_out) {
        CUDA_TRY(cudaMemcpyAsync(m->h_pin, gray, n, cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(cudaStreamSynchronize(c->stream));
        memcpy(h_gray_out, m->h_pin, n);
    }
    return CPT_OK;
}

int cpt_ir_motion_detect(cpt_ir_motion *m, int slot_new, int slot_oldest, int threshold, int erode_k, const uint8_t *h_mask,
                         int32_t *h_diff_pixels, int32_t *h_mask_pixels) {
    if (!m || !h_diff_pixels) return fail(CPT_ERR_INVALID, "null argument");
    if (slot_new < 0 || slot_new >= m->ring_frames || slot_oldest < 0 || slot_oldest >= m->ring_frames)
        return fail(CPT_ERR_INVALID, "ring slot out of range");
    if (erode_k < 1 || erode_k > cpt::kErodeMaxK) return fail(CPT_ERR_INVALID, "erosion box must be 1..64 pixels");
    if (h_mask && !h_mask_pixels) return fail(CPT_ERR_INVALID, "h_mask_pixels is required with h_mask");
    cpt_ctx *c = m->ctx;
    CUDA_TRY(cudaSetDevice(c->device));
    const int W = m->W, H = m->H, wpr = (W + 31) / 32;
    const size_t n = (size_t)W * H;
    cudaStream_t st = c->stream;
    if (h_mask) {
        // the host mask goes through pinned staging into the detector's own device buffer
        CUDA_TRY(cudaStreamSynchronize(st));  // h_pin may still be the source of an earlier copy
        memcpy(m->h_pin, h_mask, n);
        CUDA_TRY(cudaMemcpyAsync(m->d_in_mask, m->h_pin, n, cudaMemcpyHostToDevice, st));
    }
    const uint8_t *d_mask = h_mask ? m->d_in_mask : nullptr;
    cpt::ir_pack_kernel<<<(H * wpr + 7) / 8, 256, 0, st>>>(m->d_ring + slot_oldest * n, m->d_ring + slot_new * n, d_mask, W, H, wpr,
                                                           threshold, m->d_bits);
    const cpt::IrRule rule{threshold, 0, 0, erode_k, erode_k, 0};
    IrStepRecords *d = m->d_detect;
    cpt::ir_erode_kernel<<<dim3(cpt::erode_ctas(H, wpr), 1), 256, 0, st>>>(&d->args, &d->flag, &d->step, 0, 0, W, H, wpr,
                                                                          d_mask ? 2 : 1, rule, &d->result);
    CUDA_TRY(cudaGetLastError());
    auto *h_result = reinterpret_cast<cpt_ir_motion_clip_result *>(m->h_pin + 3 * n);
    CUDA_TRY(cudaMemcpyAsync(h_result, &d->result, sizeof(*h_result), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    *h_diff_pixels = h_result->diff_pixels;
    if (h_mask_pixels) *h_mask_pixels = d_mask ? h_result->mask_pixels : 0;
    return CPT_OK;
}

int cpt_ir_motion_step(cpt_ir_motion_clip *h_clip, const uint8_t *h_bgr, const cpt_ir_motion_clip_step *h_step,
                       const cpt_ir_motion_clip_params *p, cpt_ir_motion_clip_result *h_result) {
    if (!h_clip || !h_bgr || !h_step || !p || !h_result) return fail(CPT_ERR_INVALID, "null argument");
    cpt_ir_motion_clip k = *h_clip;
    k.first_step = 0; k.n_steps = 1;
    int W = 0, H = 0, rc = ir_check_params(p);
    if (!rc) rc = ir_check_clip(k.m ? k.m->ctx : nullptr, k, 0, W, H);
    if (!rc) rc = ir_check_slots(k.m, *h_step, 0);
    if (rc) return rc;
    cpt_ir_motion *m = k.m;
    CUDA_TRY(cudaSetDevice(m->ctx->device));
    cudaStream_t st = m->ctx->stream;
    CUDA_TRY(cudaStreamSynchronize(st));  // h_pin may still be the source of an earlier copy
    const size_t n = (size_t)W * H, off = ir_records_offset(n);
    auto *h = reinterpret_cast<IrStepRecords *>(m->h_pin + off), *d = reinterpret_cast<IrStepRecords *>(m->d_bgr + off);
    ir_clip_records(k, h_step, h->args, h->flag, &h->step);
    h->step.bgr = m->d_bgr;
    // frame and records go up in four slices, each copy overlapping the memcpy of the next slice into the pinned buffer
    const size_t total = off + sizeof(IrStepRecords), slice = (total + 3) / 4;
    for (size_t o = 0; o < total; o += slice) {
        if (o < 3 * n) memcpy(m->h_pin + o, h_bgr + o, std::min(slice, 3 * n - o));
        CUDA_TRY(cudaMemcpyAsync(m->d_bgr + o, m->h_pin + o, std::min(slice, total - o), cudaMemcpyHostToDevice, st));
    }
    const int wpr = (W + 31) / 32;
    const cpt::IrRule rule{p->threshold, p->trigger_frames, p->max_triggered, p->erode_idle, p->erode_recording, 1};
    cpt::ir_frame_kernel<<<dim3((H * wpr + 7) / 8, 1), 256, 0, st>>>(&d->args, &d->flag, &d->step, 0, 0, W, H, wpr, p->threshold);
    cpt::ir_erode_kernel<<<dim3(cpt::erode_ctas(H, wpr), 1), 256, 0, st>>>(&d->args, &d->flag, &d->step, 0, 0, W, H, wpr, 2, rule, &d->result);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(&h->flag, &d->flag, sizeof(h->flag) + sizeof(h->result), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    h_clip->movement = h->flag.movement;
    h_clip->triggered = h->flag.triggered;
    *h_result = h->result;
    return CPT_OK;
}

int cpt_ir_motion_clips(cpt_ctx *c, cpt_ir_motion_clip *h_clips, int n, const uint8_t *const *h_frames, int64_t n_frames,
                        const cpt_ir_motion_clip_step *h_steps, int n_steps, const cpt_ir_motion_clip_params *p,
                        cpt_ir_motion_clip_result *h_results) {
    if (!c || !p || n < 0 || n_frames < 0 || n_steps < 0) return fail(CPT_ERR_INVALID, "cpt_ir_motion_clips: bad argument");
    if ((n && !h_clips) || (n_frames && !h_frames) || (n_steps && (!h_steps || !h_results)))
        return fail(CPT_ERR_INVALID, "cpt_ir_motion_clips: null argument");
    int rc = ir_check_params(p);
    if (rc) return rc;
    // everything is checked before any model's frame count or any device buffer changes
    std::vector<int> owner(n_steps, -1);
    int W = 0, H = 0, max_steps = 0;
    for (int d = 0; d < n; ++d) {
        const cpt_ir_motion_clip &k = h_clips[d];
        if ((rc = ir_check_clip(c, k, d, W, H))) return rc;
        for (int e = 0; e < d; ++e)
            if (h_clips[e].m == k.m || h_clips[e].mog2 == k.mog2 || h_clips[e].d_mask == k.d_mask)
                return fail(CPT_ERR_INVALID, "cpt_ir_motion_clips: clips %d and %d share a handle or a mask buffer", e, d);
        if (k.first_step < 0 || k.n_steps < 0 || k.n_steps > n_steps - k.first_step)
            return fail(CPT_ERR_INVALID, "cpt_ir_motion_clips: clip %d: steps out of range", d);
        for (int i = k.first_step; i < k.first_step + k.n_steps; ++i) {
            if (owner[i] >= 0) return fail(CPT_ERR_INVALID, "cpt_ir_motion_clips: step %d belongs to clips %d and %d", i, owner[i], d);
            owner[i] = d;
            const cpt_ir_motion_clip_step &st = h_steps[i];
            if (st.row < 0 || st.row >= n_frames || !h_frames[st.row])
                return fail(CPT_ERR_INVALID, "cpt_ir_motion_clips: step %d: frame row out of range", i);
            if ((rc = ir_check_slots(k.m, st, i))) return rc;
        }
        max_steps = std::max(max_steps, k.n_steps);
    }
    if (max_steps == 0) return CPT_OK;
    CUDA_TRY(cudaSetDevice(c->device));
    const int wpr = (W + 31) / 32;
    const size_t fb = 3 * (size_t)W * H;
    // Launch units: step j of clips [c0, c1), each unit one ir_frame_kernel and one ir_erode_kernel.  Host frames are
    // staged in chunks of consecutive units whose frames fit in about 256 MB.
    const int64_t cap = p->host_frames ? std::max<int64_t>(1, (256ll << 20) / (int64_t)fb) : INT64_MAX;
    struct Unit { int j, c0, c1; int64_t rows; };
    std::vector<Unit> units;
    for (int j = 0; j < max_steps; ++j) {
        int c0 = 0, last = -1;
        int64_t rows = 0;
        for (int d = 0; d < n; ++d) {
            if (j >= h_clips[d].n_steps) continue;
            if (rows == cap || d - c0 >= 65535) {  // grid.y limit
                units.push_back({j, c0, last + 1, rows});
                c0 = d; rows = 0;
            }
            ++rows;
            last = d;
        }
        if (rows) units.push_back({j, c0, last + 1, rows});
    }
    std::vector<size_t> chunk_end;  // units [chunk_end[i - 1], chunk_end[i])
    for (size_t u = 0, rows = 0; u < units.size(); ++u) {
        if (rows + units[u].rows > (uint64_t)cap) { chunk_end.push_back(u); rows = 0; }
        rows += units[u].rows;
        if (u + 1 == units.size()) chunk_end.push_back(u + 1);
    }
    // one scratch block: clip records | flags | steps | results | staged frames, each 256-byte aligned
    int64_t max_chunk_rows = 0;
    for (size_t i = 0, u = 0; i < chunk_end.size(); ++i) {
        int64_t rows = 0;
        for (; u < chunk_end[i]; ++u) rows += units[u].rows;
        max_chunk_rows = std::max(max_chunk_rows, rows);
    }
    auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t o_flag = up(sizeof(cpt::IrClipArgs) * n), o_step = o_flag + up(sizeof(cpt::IrClipFlag) * n),
                 o_res = o_step + up(sizeof(cpt::IrStep) * n_steps), o_stage = o_res + up(sizeof(cpt_ir_motion_clip_result) * n_steps),
                 total = o_stage + (p->host_frames ? (size_t)max_chunk_rows * fb : 0);
    CUDA_TRY(c->ir_clips_scratch.ensure(total));
    uint8_t *base = c->ir_clips_scratch;
    auto *d_args = reinterpret_cast<cpt::IrClipArgs *>(base);
    auto *d_flags = reinterpret_cast<cpt::IrClipFlag *>(base + o_flag);
    auto *d_steps = reinterpret_cast<cpt::IrStep *>(base + o_step);
    auto *d_res = reinterpret_cast<cpt_ir_motion_clip_result *>(base + o_res);
    uint8_t *d_stage = base + o_stage;
    std::vector<cpt::IrClipArgs> args(n);
    std::vector<cpt::IrClipFlag> flags(n);
    std::vector<cpt::IrStep> steps(n_steps);
    for (int d = 0; d < n; ++d) {
        const cpt_ir_motion_clip &k = h_clips[d];
        ir_clip_records(k, h_steps, args[d], flags[d], steps.data());
        for (int i = k.first_step; i < k.first_step + k.n_steps; ++i) steps[i].bgr = h_frames[h_steps[i].row];
    }
    struct Copy { int64_t row; size_t offset; };
    std::vector<Copy> copies;  // host frames: the staging offset of each step's frame within its chunk
    std::vector<size_t> copies_end;
    if (p->host_frames) {
        for (size_t i = 0, u = 0; i < chunk_end.size(); ++i) {
            size_t slot = 0;
            for (; u < chunk_end[i]; ++u)
                for (int d = units[u].c0; d < units[u].c1; ++d) {
                    const cpt_ir_motion_clip &k = h_clips[d];
                    if (units[u].j >= k.n_steps) continue;
                    const int s = k.first_step + units[u].j;
                    copies.push_back({h_steps[s].row, slot * fb});
                    steps[s].bgr = d_stage + slot * fb;
                    ++slot;
                }
            copies_end.push_back(copies.size());
        }
    }
    cudaStream_t st = c->stream;
    CUDA_TRY(cudaMemcpyAsync(d_args, args.data(), sizeof(cpt::IrClipArgs) * n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_flags, flags.data(), sizeof(cpt::IrClipFlag) * n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_steps, steps.data(), sizeof(cpt::IrStep) * n_steps, cudaMemcpyHostToDevice, st));
    const cpt::IrRule rule{p->threshold, p->trigger_frames, p->max_triggered, p->erode_idle, p->erode_recording, 1};
    const unsigned frame_blocks = (unsigned)((H * wpr + 7) / 8), erode_blocks = (unsigned)cpt::erode_ctas(H, wpr);
    for (size_t i = 0, u = 0; i < chunk_end.size(); ++i) {
        if (p->host_frames)  // stream order: a chunk's frames replace the previous chunk's only after its steps have run
            for (size_t q = i ? copies_end[i - 1] : 0; q < copies_end[i]; ++q)
                CUDA_TRY(cudaMemcpyAsync(d_stage + copies[q].offset, h_frames[copies[q].row], fb, cudaMemcpyHostToDevice, st));
        for (; u < chunk_end[i]; ++u) {
            const Unit &un = units[u];
            const unsigned ny = (unsigned)(un.c1 - un.c0);
            cpt::ir_frame_kernel<<<dim3(frame_blocks, ny), 256, 0, st>>>(d_args, d_flags, d_steps, un.j, un.c0, W, H, wpr, p->threshold);
            cpt::ir_erode_kernel<<<dim3(erode_blocks, ny), 256, 0, st>>>(d_args, d_flags, d_steps, un.j, un.c0, W, H, wpr, 2, rule, d_res);
        }
        CUDA_TRY(cudaGetLastError());
    }
    CUDA_TRY(cudaMemcpyAsync(h_results, d_res, sizeof(cpt_ir_motion_clip_result) * n_steps, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(flags.data(), d_flags, sizeof(cpt::IrClipFlag) * n, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    for (int d = 0; d < n; ++d) {
        h_clips[d].movement = flags[d].movement;
        h_clips[d].triggered = flags[d].triggered;
    }
    return CPT_OK;
}

int cpt_ir_merge_components(cpt_ctx *c, const int32_t *d_stats, const int32_t *d_counts, int n_frames, int max_components, int min_mass,
                            int min_size, double max_gap, int32_t *d_merged, int32_t *d_merged_counts) {
    if (!c || !d_stats || !d_counts || !d_merged || !d_merged_counts) return fail(CPT_ERR_INVALID, "null argument");
    if (n_frames < 0) return fail(CPT_ERR_INVALID, "n_frames < 0");
    if (max_components < 1) return fail(CPT_ERR_INVALID, "max_components < 1");
    if (n_frames == 0) return CPT_OK;
    CUDA_TRY(cudaSetDevice(c->device));
    // frames per launch: the list-order scratch stays near 64 MB whatever the call's length
    const int chunk = (int)std::max<long long>(1, std::min<long long>(n_frames, (16ll << 20) / max_components));
    CUDA_TRY(c->merge_order.ensure((size_t)chunk * max_components));
    const size_t rows = (size_t)max_components + 1;
    for (int f0 = 0; f0 < n_frames; f0 += chunk) {
        const int nf = std::min(chunk, n_frames - f0);
        cpt::ir_merge_kernel<<<(nf + 3) / 4, 128, 0, c->stream>>>(d_stats + (size_t)f0 * rows * 5, d_counts + f0, nf, max_components, min_mass,
                                                                   min_size, max_gap, c->merge_order,
                                                                   d_merged + (size_t)f0 * max_components * 5, d_merged_counts + f0);
    }
    CUDA_TRY(cudaGetLastError());
    return CPT_OK;
}

}  // extern "C"
