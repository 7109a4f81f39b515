// strip_sweep.cu -- the recurrence of the split extraction path (DESIGN.md section 3.1), cut into row strips.
//
// The per-pixel recurrence of the reference (WeightedBackground keep test + 45-frame sliding mean,
// piclassifier/motiondetector.py:197-244, track/cliptrackextractor.py:168-176) never looks at another pixel: only the
// per-frame scalars (mean of the frame, extrema of filtered, mean of the background) couple the pixels of a frame, and
// those are only needed by the later per-frame stages.  So a clip is cut into n_strips bands of whole rows and every
// (clip, strip) pair is an independent work unit of strip_sweep_kernel:
//   * one CTA per unit, 15 consumer warps + a copy warp + a fold warp; a consumer thread owns ONE quad (4 pixels) for the whole
//     clip: background B, weight counter k and sliding sum S of its pixels live in registers from the first frame to the
//     last -- no per-frame state traffic at all;
//   * the strip's rows of the last 45 frames (the window of the sliding mean) plus kLead frames of read-ahead sit in a
//     shared-memory ring filled by the copy warp with one 1-D TMA bulk copy per frame (full mbarriers); the frame
//     leaving the window is read from that ring, so every frame is read from HBM exactly once and never again;
//   * per frame a consumer writes its filtered quad (fp32), the zeroed label bytes and one byte per quad (max filtered
//     relative to a strip reference, for the hot-quad test of the per-frame kernels); the warps' partial sums go through
//     a small shared-memory table to the fold warp, which folds them into the strip's pass record in global memory
//     (done mbarriers release the ring slot to the copy warp and the rows to the fold warp; folded mbarriers hand the
//     table rows and the byte reference back).  Copying and folding were one warp's loop at first: its length, not the
//     read-ahead, bounded the pipeline (26.7 ms without the fold against 29.6 ms with it).
// frame_scalars_kernel (one warp per clip) then folds the strips' records into the per-frame scalars of
// ClipTracker._get_filtered_frame (track/cliptracker.py:93-122): WeightedBackground.average (a running value: scanned over
// the frames with warp ballots), avg_change, the normalisation range, the mapped threshold, the integer normalise
// constants and the per-strip byte thresholds.
#include <type_traits>

#include "cptrack_kernels.cuh"
#include "sm100_primitives.cuh"

namespace cpt {

namespace {

using namespace prim;

constexpr int kLead = 7;                             // frames the copy warp runs ahead of the slowest consumer warp
constexpr int kRingSlots = kMeanFrames + kLead;      // 52 frames of the strip's rows
constexpr int kSlotBytes = kStripPxMax * 2;          // 3840
constexpr int kConsWarps = kStripPxMax / 4 / 32;     // 15
constexpr int kConsThreads = kConsWarps * 32;        // 480
constexpr int kBarRing = 8;                          // full / done barriers and stat rows are reused every kBarRing passes
static_assert(kBarRing > kLead, "a barrier is reused only after every warp has passed its previous use");
static_assert(kStripThreads == kConsThreads + 64, "consumer warps + the copy warp + the fold warp");
constexpr int kStripTable = 4096;                    // first entries of the clip's keep-test table
constexpr int kRefLag = kLead + 1;                    // a frame's quad bytes are stored against the strip minimum kRefLag frames earlier
constexpr int kRefDefault = kQuadRefBias;            // reference of the first kRefLag frames (filtered starts near 0)

struct __align__(128) StripSmem {
    uint8_t ring[kRingSlots][kSlotBytes];
    uint16_t wthr[kStripTable];              // keep-test thresholds of the clip's table (first entries) ...
    uint16_t wbnd[kStripTable];              // ... and their bounds (cptrack_kernels.cuh, WeightTable)
    uint32_t stat[kBarRing][kConsWarps][8];  // per pass and warp: psum, fmin, fmax, nbsum, pmin, pmax, fabs, changed
    int32_t ref_ring[16];                    // byte reference published with pass t, used by pass t + kRefLag
    unsigned long long full[kBarRing], done[kBarRing], folded[kBarRing];
    int32_t unit;
};
static_assert(sizeof(StripSmem) <= 232448, "shared memory budget (227 KB per CTA on sm_100)");

// A thread's pixels.  Everything is kept biased by kBias = 0x4B400000 (the bits of 1.5 * 2^23): nb = kBias - background, so
// that thermal + nb is at once the integer filtered + kBias (ordering, extrema and differences are unaffected) and the bit
// pattern of the float 12582912 + filtered -- one FADD instead of an integer-to-float conversion per pixel.
// kv = the weight counter k -- or, while the keep test is the linear one (thr = k + 1, weight_add == 1), v = nb - k: then
// keep <=> A - B >= k + 1 <=> v > kBias - A, and both outcomes fold into v' = max(v - 1, kBias - A) (kept: k + 1; reset:
// background = A, k = 0).  k = nb - v either way (the same formula converts back).
constexpr int kBias = 0x4B400000;
constexpr float kBiasF = 12582912.0f;
struct QuadState {
    int nb[4], kv[4], f[4];
    uint32_t S[4];
    bool lin;
};

struct StripThread {
    bool active, border_row, first_col, last_col;
    const uint8_t *src, *out;  // the quad inside ring slot 0: the row its state follows / the row it outputs
    int m[4];                  // 1: the pixel counts for the background sum (crop pixel of an owned row)
    int bs0;                   // -(m[0] + .. + m[3]) * kBias
    float *fptr;               // the thread's quad in the clip's first output frame; frame t: + t * npx (t * qstride for the
    uint8_t *lptr;             // quad bytes) -- one wide multiply-add per store instead of three carried 64-bit pointers
    int8_t *qptr;
    uint32_t npx, qstride;
};

// what is uniform over the CTA in one pass of the generic path
struct PassCtx {
    bool update, is_frame, window_full, first_mean;
    uint32_t magic;              // floor(S / cnt) == umulhi(S, magic)
};

struct PassOut {
    uint32_t psum;
    int fmin, fmax, bs, chg, pmin, pmax;   // fmin / fmax biased by kBias
    uint32_t fabs_sum;
};

__device__ __forceinline__ uint2 lds8(const uint8_t *p) { return *reinterpret_cast<const uint2 *>(p); }

// One pass of one quad: [update] WeightedBackground.process_frame for the previous frame (A = floor(S / cnt); keep <=>
// B < A - w_k in the table form of cptrack_kernels.cuh; B' = keep ? B : A, k' = keep ? k + 1 : 0), then [frame] K1 of this
// frame against B' (F = P - B', S += P - P_old) with the frame's sums.  State is unpacked 32-bit integers.
// kTab: 0 thr = k + 1 (weight_add == 1; QuadState::lin form), 1 table in shared memory, 2 table in shared + global memory.
// kSteady: update && frame && window full && cnt == 45 are compile-time facts.
// bmax: largest bound of the table entries a counter can have reached (bounds only matter for backgrounds below them).
// kFull: every consumer thread owns a quad of the strip (12 rows x 40 quads at 160x120): no activity test, no defaults for
// the sums of a thread without one.
template <int kTab, bool kStats, bool kSteady, bool kLabels, bool kFull>
__device__ __forceinline__ void strip_pass(StripSmem &s, const WeightTable &wt, const PassCtx &pc, const StripThread &th,
                                           QuadState &q, PassOut &po, uint32_t cur_off, uint32_t old_off, int refb, int bmax, uint32_t t) {
    const bool is_frame = kSteady || pc.is_frame;
    uint2 pw = make_uint2(0, 0), pv = make_uint2(0, 0), ow = make_uint2(0, 0);
    if (is_frame) {
        pw = lds8(th.src + cur_off);
        pv = th.border_row ? lds8(th.out + cur_off) : pw;
        if (kSteady || pc.window_full) ow = lds8(th.src + old_off);
    }
    int chg = 0;
    if (kSteady || pc.update) {
        int na[4], nn[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) na[i] = kBias - (int)((!kSteady && pc.first_mean) ? q.S[i] : __umulhi(q.S[i], pc.magic));
        if (kTab == 0) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                nn[i] = q.kv[i] > na[i] ? q.nb[i] : na[i];
                q.kv[i] = __viaddmax_s32(q.kv[i], -1, na[i]);
            }
        } else {
            int e[4];
            const bool use_global = kTab == 2;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if (use_global && q.kv[i] >= kStripTable) e[i] = (int)(__ldg(wt.thr + q.kv[i]) & 0xffffu);
                else e[i] = (int)s.wthr[q.kv[i]];
            }
            // bounds (the fp64 rounding of A - w_k depends on the magnitude of B) only matter for backgrounds below the largest
            // bound a counter can have reached: one vote per quad, rarely taken
            const int nbmax = max(max(q.nb[0], q.nb[1]), max(q.nb[2], q.nb[3]));
            if (__any_sync(0xffffffffu, nbmax + bmax > kBias)) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int bound = (use_global && q.kv[i] >= kStripTable) ? (int)(__ldg(wt.thr + q.kv[i]) >> 16) : (int)s.wbnd[q.kv[i]];
                    e[i] -= (q.nb[i] + bound > kBias) ? 1 : 0;   // B < bound
                }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const bool keep = q.nb[i] - na[i] >= e[i];  // A - B >= thr
                nn[i] = keep ? q.nb[i] : na[i];
                q.kv[i] = keep ? q.kv[i] + 1 : 0;
            }
        }
        // crop-border columns copy their neighbour (motiondetector.py:239-244); they were equal before, so they add nothing
        // to `changed` (their own counters only ever feed their own, discarded, keep test)
        if (th.first_col) nn[0] = nn[1];
        if (th.last_col) nn[3] = nn[2];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            chg |= nn[i] ^ q.nb[i];
            q.nb[i] = nn[i];
        }
    }
    // minus the background sum over the crop pixels of owned rows (wrapping arithmetic takes the bias out again)
    po.bs = (int)((uint32_t)q.nb[0] * (uint32_t)th.m[0] +
                  ((uint32_t)q.nb[1] * (uint32_t)th.m[1] +
                   ((uint32_t)q.nb[2] * (uint32_t)th.m[2] + ((uint32_t)q.nb[3] * (uint32_t)th.m[3] + (uint32_t)th.bs0))));
    po.chg = chg;  // (inactive threads follow a real row of the strip: duplicates of real changes)
    po.psum = 0;
    po.fmin = INT32_MAX; po.fmax = INT32_MIN; po.pmin = INT32_MAX; po.pmax = INT32_MIN; po.fabs_sum = 0;
    if (is_frame) {
        int (&f)[4] = q.f;
        f[0] = dp2a_us(pv.x, kLoP, q.nb[0]); f[1] = dp2a_us(pv.x, kHiP, q.nb[1]);
        f[2] = dp2a_us(pv.y, kLoP, q.nb[2]); f[3] = dp2a_us(pv.y, kHiP, q.nb[3]);
        q.S[0] = (uint32_t)dp2a_us(pw.x, kLoP, dp2a_us(ow.x, kLoN, (int)q.S[0]));
        q.S[1] = (uint32_t)dp2a_us(pw.x, kHiP, dp2a_us(ow.x, kHiN, (int)q.S[1]));
        q.S[2] = (uint32_t)dp2a_us(pw.y, kLoP, dp2a_us(ow.y, kLoN, (int)q.S[2]));
        q.S[3] = (uint32_t)dp2a_us(pw.y, kHiP, dp2a_us(ow.y, kHiN, (int)q.S[3]));
        const int lo = min(min(f[0], f[1]), min(f[2], f[3])), hi = max(max(f[0], f[1]), max(f[2], f[3]));
        if (kFull || th.active) {
            po.psum = (uint32_t)dp2a_us(pv.x, kBoth, dp2a_us(pv.y, kBoth, 0));
            po.fmin = lo;
            po.fmax = hi;
            if (kStats) {
                const int p0 = (int)(pv.x & 0xffffu), p1 = (int)(pv.x >> 16), p2 = (int)(pv.y & 0xffffu), p3 = (int)(pv.y >> 16);
                po.pmin = min(min(p0, p1), min(p2, p3));
                po.pmax = max(max(p0, p1), max(p2, p3));
                po.fabs_sum = (uint32_t)(abs(f[0] - kBias) + abs(f[1] - kBias) + abs(f[2] - kBias) + abs(f[3] - kBias));
            }
            *reinterpret_cast<float4 *>(th.fptr + (size_t)t * th.npx) = make_float4(__int_as_float(f[0]) - kBiasF, __int_as_float(f[1]) - kBiasF,
                                                               __int_as_float(f[2]) - kBiasF, __int_as_float(f[3]) - kBiasF);
            if (kLabels) *reinterpret_cast<uint32_t *>(th.lptr + (size_t)t * th.npx) = 0u;
            int b;
            asm("cvt.sat.s8.s32 %0, %1;" : "=r"(b) : "r"(hi - refb));
            th.qptr[(size_t)t * th.qstride] = (int8_t)b;
        }
    }
}

// k <-> v = nb - k (QuadState): the same formula both ways.  Border columns restart from k = 0 (their counters are
// never used; this keeps table indices in range).
__device__ __forceinline__ void quad_state_form(QuadState &q, const StripThread &th, bool lin) {
    if (q.lin == lin) return;
#pragma unroll
    for (int i = 0; i < 4; ++i) q.kv[i] = q.nb[i] - q.kv[i];
    if (!lin) {
        if (th.first_col) q.kv[0] = 0;
        if (th.last_col) q.kv[3] = 0;
    }
    q.lin = lin;
}

// the running positions of a consumer warp: pass t, its ring slots and barriers
struct PassPos {
    int t;
    uint32_t cur_off, old_off;   // ring slots (byte offsets) of frame t and of frame t - 45 (== the slot of frame t + kLead)
    int frames_seen;             // background updates applied so far: no weight counter can exceed it
    int bmax;                    // largest bound among the table entries [0, frames_seen]
};

__device__ __forceinline__ void pass_advance(PassPos &p) {
    ++p.t;
    p.cur_off += kSlotBytes;
    if (p.cur_off == (uint32_t)kRingSlots * kSlotBytes) p.cur_off = 0;
    p.old_off += kSlotBytes;
    if (p.old_off == (uint32_t)kRingSlots * kSlotBytes) p.old_off = 0;
}

// the warp's partial results -> its row of the pass table (the fold warp folds the rows), then the warp's arrival
template <bool kStats>
__device__ __forceinline__ void pass_report(StripSmem &s, const PassOut &po, int bi, int warp, int lane, uint32_t done0) {
    const uint32_t psum = __reduce_add_sync(0xffffffffu, po.psum);
    const int fmin = __reduce_min_sync(0xffffffffu, po.fmin), fmax = __reduce_max_sync(0xffffffffu, po.fmax);
    const int bs = __reduce_add_sync(0xffffffffu, po.bs);
    const bool chg = __any_sync(0xffffffffu, po.chg != 0);
    uint4 *row = reinterpret_cast<uint4 *>(s.stat[bi][warp]);
    if (kStats) {
        const int pmin = __reduce_min_sync(0xffffffffu, po.pmin), pmax = __reduce_max_sync(0xffffffffu, po.pmax);
        const uint32_t fabs_sum = __reduce_add_sync(0xffffffffu, po.fabs_sum);
        if (lane == 0) row[1] = make_uint4((uint32_t)pmin, (uint32_t)pmax, fabs_sum, 0u);
    }
    // (psum < 2^23 for a warp: bit 31 carries `changed`)
    if (lane == 0) row[0] = make_uint4(psum | (chg ? 0x80000000u : 0u), (uint32_t)fmin, (uint32_t)fmax, (uint32_t)bs);
    __syncwarp();
    if (lane == 0) mbar_arrive_addr(done0 + (uint32_t)(bi << 3));  // (release: the ring reads and the row are done)
}

template <bool kStats, bool kLabels, bool kFull>
__device__ void strip_consumer(const KernelArgs &a, StripSmem &s, const cpt_clip &clip, int ci, int y0, int rows, int tid) {
    const Geometry &g = a.g;
    const int W = g.W, H = g.H, e = g.edge, qpr = g.qpr, npx = g.npx;
    const int lane = tid & 31, warp = tid >> 5;
    const WeightTable wt = a.tables[clip.weight_table & 3];
    const bool update_bg = clip.flags & CPT_CLIP_UPDATE_BACKGROUND;
    const bool skip_first = clip.flags & CPT_CLIP_SKIP_FIRST_UPDATE;
    const int n = clip.n_frames;
    StripThread th;
    th.active = tid < rows * qpr;
    const int r = th.active ? tid / qpr : 0, qx = th.active ? tid - r * qpr : 0;
    const int y = y0 + r;
    const int ys = min(max(y, e), H - 1 - e);  // a border row follows the state of the owned row next to it
    th.border_row = ys != y;
    th.first_col = e && qx == 0;
    th.last_col = e && qx == qpr - 1;
    th.src = &s.ring[0][0] + ((ys - y0) * W + 4 * qx) * 2;
    th.out = &s.ring[0][0] + ((y - y0) * W + 4 * qx) * 2;
    {
        const int own = (th.active && !th.border_row) ? 1 : 0;
        th.m[0] = th.first_col ? 0 : own; th.m[1] = own; th.m[2] = own; th.m[3] = th.last_col ? 0 : own;
        th.bs0 = (int)(0u - (uint32_t)(th.m[0] + th.m[1] + th.m[2] + th.m[3]) * (uint32_t)kBias);
    }
    const int pix = y * W + 4 * qx;
    th.fptr = a.filtered + (size_t)clip.out_offset * npx + pix;
    th.lptr = a.labels + (size_t)clip.out_offset * npx + pix;   // (only dereferenced with kLabels)
    th.qptr = a.qbytes + (size_t)clip.out_offset * (H * qpr) + (y * qpr + qx);
    th.npx = (uint32_t)npx;
    th.qstride = (uint32_t)(H * qpr);

    // ---- WeightedBackground first call (motiondetector.py:199-212): background = the initialising frame, edges replicated
    QuadState q;
    q.lin = false;
    {
        const uint16_t *init = a.frames + (size_t)clip.init_offset * npx;
        const uint2 v = th.active ? __ldg(reinterpret_cast<const uint2 *>(init + ys * W + 4 * qx)) : make_uint2(0, 0);
        int b0 = (int)(v.x & 0xffffu), b1 = (int)(v.x >> 16), b2 = (int)(v.y & 0xffffu), b3 = (int)(v.y >> 16);
        if (th.first_col) b0 = b1;
        if (th.last_col) b3 = b2;
        q.nb[0] = kBias - b0; q.nb[1] = kBias - b1; q.nb[2] = kBias - b2; q.nb[3] = kBias - b3;
#pragma unroll
        for (int i = 0; i < 4; ++i) { q.kv[i] = 0; q.S[i] = 0; q.f[i] = kBias; }
    }

    PassPos pp;
    pp.t = 0;
    pp.cur_off = 0;
    pp.old_off = (uint32_t)kLead * kSlotBytes;
    pp.frames_seen = 0;
    pp.bmax = 0;
    constexpr uint32_t kMagic45 = 0xffffffffu / (uint32_t)kMeanFrames + 1u;
    auto table_bound = [&](int k) -> int {  // bound of table entry k
        if (k > wt.max_count) return 0;
        return k < kStripTable ? (int)s.wbnd[k] : (int)(__ldg(wt.thr + k) >> 16);
    };
    const uint32_t full0 = smem_u32(&s.full[0]), done0 = smem_u32(&s.done[0]);
    auto frame_sync = [&](int t, int &refb) {
        // the frame's rows are in the ring; the reference its quad bytes are stored against was published by the fold warp
        // before the copy warp issued this frame (read after the acquire)
        mbar_wait_addr(full0 + (((uint32_t)t & (uint32_t)(kBarRing - 1)) << 3), ((uint32_t)t / (uint32_t)kBarRing) & 1u);
        // (the first kRefLag entries a pass reads hold the default: strip_sweep_kernel fills the ring before a unit starts)
        refb = *(volatile const int32_t *)&s.ref_ring[(t + 16 - kRefLag) & 15] + kBias;
    };

    // ---- generic pass (the first 45 frames, the tail pass, clips that do not update their background)
    auto generic_pass = [&]() {
        const int t = pp.t;
        PassCtx pc;
        pc.is_frame = t < n;
        const int t_abs = clip.first_frame + t;
        // (rawdb.py:84-122: no update follows the frame that initialised the background when it is also the first kept frame)
        pc.update = update_bg && t > 0 && !(skip_first && t_abs == 1);
        // the update belongs to frame t-1: the mean covers min(t_abs, 45) frames
        const uint32_t cnt = (uint32_t)min(max(t_abs, 1), kMeanFrames);
        pc.first_mean = cnt == 1u;
        pc.magic = cnt == 1u ? 0u : 0xffffffffu / cnt + 1u;  // exact for S < 2^22, cnt <= 45
        pc.window_full = t >= kMeanFrames;
        int refb = kRefDefault + kBias;
        if (pc.is_frame) frame_sync(t, refb);
        // (the tail pass enters no frame: its table rows are free once the fold warp has read those of pass t - kBarRing)
        else if (t >= kBarRing) mbar_wait(&s.folded[(t - kBarRing) & (kBarRing - 1)], (uint32_t)((t - kBarRing) / kBarRing) & 1u);
        const bool lin = pp.frames_seen < wt.linear_upto;
        quad_state_form(q, th, lin);
        PassOut po;
        if (lin) strip_pass<0, kStats, false, kLabels, kFull>(s, wt, pc, th, q, po, pp.cur_off, pp.old_off, refb, pp.bmax, (uint32_t)t);
        else strip_pass<2, kStats, false, kLabels, kFull>(s, wt, pc, th, q, po, pp.cur_off, pp.old_off, refb, pp.bmax, (uint32_t)t);
        if (pc.update) {
            ++pp.frames_seen;
            pp.bmax = max(pp.bmax, table_bound(pp.frames_seen));
        }
        pass_report<kStats>(s, po, t & (kBarRing - 1), warp, lane, done0);
        pass_advance(pp);
    };
    // ---- steady passes [pp.t, t_end) with one keep-test form
    auto steady_passes = [&](int t_end, auto tab_tag) {
        constexpr int kTab = decltype(tab_tag)::value;
        quad_state_form(q, th, kTab == 0);
        if (kTab != 0) pp.bmax = max(pp.bmax, table_bound(pp.frames_seen));
        PassCtx pc;
        pc.update = true; pc.is_frame = true; pc.window_full = true; pc.first_mean = false;
        pc.magic = kMagic45;
#pragma unroll 2
        while (pp.t < t_end) {
            int refb;
            frame_sync(pp.t, refb);
            PassOut po;
            strip_pass<kTab, kStats, true, kLabels, kFull>(s, wt, pc, th, q, po, pp.cur_off, pp.old_off, refb, pp.bmax, (uint32_t)pp.t);
            ++pp.frames_seen;
            if (kTab != 0) pp.bmax = max(pp.bmax, table_bound(pp.frames_seen));
            pass_report<kStats>(s, po, pp.t & (kBarRing - 1), warp, lane, done0);
            pass_advance(pp);
        }
    };

    // passes 0 .. n: frames t < n, then the tail pass (the background update that follows the last frame).  A pass is
    // steady once the window is full, i.e. for 45 <= t < n when the clip updates its background from its first frame on.
    const bool can_steady = update_bg && clip.first_frame >= 0;
    while (pp.t < min(n, kMeanFrames)) generic_pass();
    while (pp.t < n) {
        if (!can_steady) { generic_pass(); continue; }
        // the keep-test form changes with the number of updates so far: linear while every reachable entry is k + 1, then the
        // shared-memory table, then shared + global
        const int fs = pp.frames_seen;
        if (fs < wt.linear_upto) steady_passes(min(n, pp.t + (wt.linear_upto - fs)), std::integral_constant<int, 0>{});
        else if (fs < kStripTable) steady_passes(min(n, pp.t + (kStripTable - fs)), std::integral_constant<int, 1>{});
        else steady_passes(n, std::integral_constant<int, 2>{});
    }
    if (update_bg && n > 0 && !(skip_first && clip.first_frame + n == 1)) generic_pass();

    // ---- the clip's state record (cpt_state_bytes): background, counters, sliding sums, last filtered image
    if (a.state && th.active) {
        quad_state_form(q, th, false);
        uint8_t *st_raw = a.state + (size_t)ci * state_bytes(npx);
        uint16_t *st_B = reinterpret_cast<uint16_t *>(st_raw + sizeof(StateHeader));
        uint16_t *st_K = st_B + npx;
        uint32_t *st_S = reinterpret_cast<uint32_t *>(st_K + npx);
        float *st_F = reinterpret_cast<float *>(st_S + npx);
        uint2 bw, kw;
        bw.x = (uint32_t)(kBias - q.nb[0]) | ((uint32_t)(kBias - q.nb[1]) << 16);
        bw.y = (uint32_t)(kBias - q.nb[2]) | ((uint32_t)(kBias - q.nb[3]) << 16);
        // (a border row / column has no counter of its own: zero, as the crop view of cpt_state_read never shows it)
        const int k0 = th.first_col ? 0 : q.kv[0], k3 = th.last_col ? 0 : q.kv[3];
        kw.x = th.border_row ? 0u : ((uint32_t)k0 | ((uint32_t)q.kv[1] << 16));
        kw.y = th.border_row ? 0u : ((uint32_t)q.kv[2] | ((uint32_t)k3 << 16));
        *reinterpret_cast<uint2 *>(st_B + pix) = bw;
        *reinterpret_cast<uint2 *>(st_K + pix) = kw;
        *reinterpret_cast<uint4 *>(st_S + pix) = th.border_row ? make_uint4(0, 0, 0, 0) : make_uint4(q.S[0], q.S[1], q.S[2], q.S[3]);
        if (n > 0)
            *reinterpret_cast<float4 *>(st_F + pix) = make_float4((float)(q.f[0] - kBias), (float)(q.f[1] - kBias), (float)(q.f[2] - kBias),
                                                                  (float)(q.f[3] - kBias));
    }
}

// The copy warp: frame t + kLead goes into the ring slot pass t has just released.  Its loop is the critical path of the
// pipeline (one iteration per pass), so it does nothing else; the records are the fold warp's.
__device__ void strip_copier(const KernelArgs &a, StripSmem &s, const cpt_clip &clip, int y0, int rows, int lane) {
    const Geometry &g = a.g;
    const int n = clip.n_frames;
    const uint32_t bytes = (uint32_t)(rows * g.W) * 2u;
    const unsigned long long policy = l2_policy_evict_first();  // every frame is read exactly once
    const bool linear = clip.ring_frames == 0;
    const uint16_t *lin_src = a.frames + (size_t)clip.frame_offset * g.npx + (size_t)y0 * g.W;  // frame 0 of a linear clip
    if (lane != 0) return;
    auto issue = [&](int fidx) {
        const uint16_t *src = linear ? lin_src + (size_t)fidx * g.npx
                                     : a.frames + (size_t)(clip.frame_offset + (clip.first_frame + fidx) % clip.ring_frames) * g.npx + (size_t)y0 * g.W;
        unsigned long long *bar = &s.full[fidx & (kBarRing - 1)];
        mbar_arrive_expect_tx(bar, bytes);
        bulk_g2s_hint(s.ring[fidx % kRingSlots], src, bytes, bar, policy);
    };
    for (int fidx = 0; fidx < min(kLead, n); ++fidx) issue(fidx);
    for (int t = 0; t + kLead < n; ++t) {
        mbar_wait(&s.done[t & (kBarRing - 1)], (uint32_t)(t / kBarRing) & 1u);  // every consumer warp has finished pass t
        // frame t + kLead lets the consumers into pass t + kLead, whose table rows are those of pass t + kLead - kBarRing and
        // whose byte reference is that of pass t + kLead - kRefLag = t - 1: the fold warp must be done with both
        // (the arrive.expect_tx below releases what it published)
        if (t >= 1) mbar_wait(&s.folded[(t - 1) & (kBarRing - 1)], (uint32_t)((t - 1) / kBarRing) & 1u);
        issue(t + kLead);
    }
}

// The fold warp: the consumer warps' rows of pass t -> the strip's record of pass t in global memory, and the byte
// reference of pass t + kRefLag.
__device__ void strip_folder(const KernelArgs &a, StripSmem &s, const cpt_clip &clip, int ci, int strip, int lane) {
    const Geometry &g = a.g;
    const int n = clip.n_frames, NS = g.n_strips;
    const bool update_bg = clip.flags & CPT_CLIP_UPDATE_BACKGROUND;
    const bool skip_first = clip.flags & CPT_CLIP_SKIP_FIRST_UPDATE;
    const bool want_stats = clip.flags & CPT_CLIP_FRAME_STATS;
    uint4 *rec_frame = reinterpret_cast<uint4 *>(a.prec + (size_t)clip.out_offset * NS + strip);  // pass t: + t * NS records
    uint4 *rec_tail = reinterpret_cast<uint4 *>(a.prec + (size_t)(a.total_frames + ci) * NS + strip);
    const bool in = lane < kConsWarps;
    for (int t = 0; t <= n; ++t) {
        const bool is_frame = t < n;
        const bool update = update_bg && t > 0 && !(skip_first && clip.first_frame + t == 1);
        if (!update && !is_frame) break;
        mbar_wait(&s.done[t & (kBarRing - 1)], (uint32_t)(t / kBarRing) & 1u);  // every consumer warp has finished pass t
        const uint32_t *row = s.stat[t & (kBarRing - 1)][in ? lane : 0];
        const uint4 r0 = *reinterpret_cast<const uint4 *>(row);
        const uint32_t psum = __reduce_add_sync(0xffffffffu, in ? (r0.x & 0x7fffffffu) : 0u);
        // (the consumers' extrema carry the bias of their filtered values; the extrema of a pass without a frame are never read)
        const int fmin = __reduce_min_sync(0xffffffffu, in ? (int)r0.y : INT32_MAX) - kBias;
        const int fmax = __reduce_max_sync(0xffffffffu, in ? (int)r0.z : INT32_MIN) - kBias;
        const int nbsum = __reduce_add_sync(0xffffffffu, in ? (int)r0.w : 0);
        const uint32_t changed = __reduce_or_sync(0xffffffffu, in ? (r0.x >> 31) : 0u);
        int pmin = 0, pmax = 0;
        uint32_t fabs_sum = 0;
        if (want_stats) {
            const uint4 r1 = *reinterpret_cast<const uint4 *>(row + 4);
            pmin = __reduce_min_sync(0xffffffffu, in ? (int)r1.x : INT32_MAX);
            pmax = __reduce_max_sync(0xffffffffu, in ? (int)r1.y : INT32_MIN);
            fabs_sum = __reduce_add_sync(0xffffffffu, in ? r1.z : 0u);
        }
        if (lane == 0) {
            // the reference of pass t + kRefLag: this strip's filtered minimum now, plus the bias (clamped so that it
            // survives the shift below); published first, the record is nobody's critical path
            const int ref = t >= kRefLag ? s.ref_ring[(t - kRefLag) & 15] : kRefDefault;  // what pass t's bytes were stored against
            if (is_frame) s.ref_ring[t & 15] = max(min(fmin, 1 << 20), -(1 << 20)) + kQuadRefBias;
            mbar_arrive(&s.folded[t & (kBarRing - 1)]);  // (release: the rows are read, the reference is written)
            uint4 *dst = is_frame ? rec_frame + (size_t)t * (2 * NS) : rec_tail;
            dst[0] = make_uint4(psum, (uint32_t)fmin, (uint32_t)fmax, (uint32_t)nbsum);
            dst[1] = make_uint4((uint32_t)pmin, (uint32_t)pmax, fabs_sum, ((uint32_t)ref << 1) | (changed & 1u));
        }
        __syncwarp();
    }
}

}  // namespace

// Split path, first launch: the recurrence.  grid = min(units, SMs) persistent CTAs; units = (clip, strip) pairs handed
// out by an atomic counter, clip-major so that the strips of a clip run side by side.
__global__ void __launch_bounds__(kStripThreads, 1) strip_sweep_kernel(const KernelArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    StripSmem &s = *reinterpret_cast<StripSmem *>(smem_raw);
    const int tid = threadIdx.x;
    const Geometry &g = a.g;
    const int NS = g.n_strips;
    bool bars_live = false;
    while (true) {
        __syncthreads();  // every thread is done with the previous unit (ring, barriers, table)
        if (tid == 0) s.unit = atomicAdd(a.work_counter, 1);
        __syncthreads();
        const int u = s.unit;
        if (u >= a.n_clips * NS) break;
        const int ci = u / NS, strip = u - ci * NS;
        const cpt_clip clip = a.clips[ci];
        const int y0 = strip * g.H / NS, rows = (strip + 1) * g.H / NS - y0;
        if (tid == 0) {
            if (bars_live)
                for (int i = 0; i < kBarRing; ++i) { mbar_inval(&s.full[i]); mbar_inval(&s.done[i]); mbar_inval(&s.folded[i]); }
            for (int i = 0; i < kBarRing; ++i) {
                mbar_init(&s.full[i], 1);           // the copy warp's arrive.expect_tx
                mbar_init(&s.done[i], kConsWarps);  // one arrival per consumer warp
                mbar_init(&s.folded[i], 1);         // the fold warp
            }
            for (int i = 0; i < 16; ++i) s.ref_ring[i] = kRefDefault;  // (what the first kRefLag passes read)
            mbar_fence_init();
            bars_live = true;
        }
        {
            const WeightTable wt = a.tables[clip.weight_table & 3];
            for (int i = tid; i < kStripTable; i += kStripThreads) {
                const uint32_t e = (i <= wt.max_count) ? __ldg(wt.thr + i) : 0xffffu;  // beyond the table: never keep
                s.wthr[i] = (uint16_t)(e & 0xffffu);
                s.wbnd[i] = (uint16_t)(e >> 16);
            }
        }
        __syncthreads();
        if (tid < kConsThreads) {
            const bool full = rows * g.qpr == kConsThreads;  // every consumer thread owns a quad
            if (clip.flags & CPT_CLIP_FRAME_STATS) {
                if (a.labels && full) strip_consumer<true, true, true>(a, s, clip, ci, y0, rows, tid);
                else if (a.labels) strip_consumer<true, true, false>(a, s, clip, ci, y0, rows, tid);
                else strip_consumer<true, false, false>(a, s, clip, ci, y0, rows, tid);
            } else {
                if (a.labels && full) strip_consumer<false, true, true>(a, s, clip, ci, y0, rows, tid);
                else if (a.labels) strip_consumer<false, true, false>(a, s, clip, ci, y0, rows, tid);
                else strip_consumer<false, false, false>(a, s, clip, ci, y0, rows, tid);
            }
        } else if (tid < kConsThreads + 32) {
            strip_copier(a, s, clip, y0, rows, tid - kConsThreads);
        } else {
            strip_folder(a, s, clip, ci, strip, tid - kConsThreads - 32);
        }
    }
}

size_t strip_sweep_smem_bytes() { return sizeof(StripSmem); }

// ================================================================================================
// frame_scalars_kernel: one warp per clip, lanes = 32 consecutive passes.
// ================================================================================================
__global__ void __launch_bounds__(128) frame_scalars_kernel(const KernelArgs a) {
    const Geometry &g = a.g;
    const int lane = threadIdx.x & 31;
    const int ci = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (ci >= a.n_clips) return;
    const cpt_clip clip = a.clips[ci];
    const int n = clip.n_frames, NS = g.n_strips, npx = g.npx;
    const bool update_bg = clip.flags & CPT_CLIP_UPDATE_BACKGROUND;
    const bool skip_first = clip.flags & CPT_CLIP_SKIP_FIRST_UPDATE;
    const bool want_stats = clip.flags & CPT_CLIP_FRAME_STATS;
    const bool denoise = clip.flags & CPT_CLIP_DENOISE;
    double average = 0.0;  // WeightedBackground.average: carried from pass to pass
    int frames_seen = 0, last_fmin = 0, last_fmax = 0;
    if (n == 0) {
        // no pass ran: the initial average straight from the initialising frame (np.average of the crop, unrounded)
        const uint16_t *init = a.frames + (size_t)clip.init_offset * npx;
        uint32_t sum = 0;
        for (int i = lane; i < npx; i += 32) {
            const int y = i / g.W, x = i - y * g.W;
            if (x >= g.edge && x < g.W - g.edge && y >= g.edge && y < g.H - g.edge) sum += __ldg(init + i);
        }
        sum = __reduce_add_sync(0xffffffffu, sum);
        average = (double)sum / (double)g.ncrop;
    }
    for (int base = 0; base <= n && n > 0; base += 32) {
        const int t = base + lane;
        const bool is_frame = t < n;
        const bool upd = update_bg && t > 0 && t <= n && !(skip_first && clip.first_frame + t == 1);
        const bool valid = t <= n && (is_frame || upd);
        const size_t o = (size_t)(clip.out_offset + t);
        // ---- fold the strips' records of this pass
        uint32_t psum = 0, fabs_sum = 0, changed = 0;
        int fmin = INT32_MAX, fmax = INT32_MIN, pmin = INT32_MAX, pmax = INT32_MIN;
        long long nbsum = 0;
        int ref_s[kMaxStrips], fmax_s[kMaxStrips];
        if (valid) {
            const uint4 *rp = reinterpret_cast<const uint4 *>(a.prec + (is_frame ? o : (size_t)(a.total_frames + ci)) * NS);
#pragma unroll
            for (int sidx = 0; sidx < kMaxStrips; ++sidx) {
                ref_s[sidx] = 0;
                fmax_s[sidx] = INT32_MIN;
                if (sidx < NS) {
                    const uint4 r0 = __ldcg(rp + 2 * sidx), r1 = __ldcg(rp + 2 * sidx + 1);
                    psum += r0.x;
                    fmin = min(fmin, (int)r0.y);
                    fmax = max(fmax, (int)r0.z);
                    nbsum += (int)r0.w;
                    pmin = min(pmin, (int)r1.x);
                    pmax = max(pmax, (int)r1.y);
                    fabs_sum += r1.z;
                    changed |= r1.w & 1u;
                    ref_s[sidx] = (int)r1.w >> 1;
                    fmax_s[sidx] = (int)r0.z;
                }
            }
        }
        // ---- WeightedBackground.average: set by pass 0 (np.average of the initial crop, unrounded) and by every update
        // that changed the background (int(round(np.average(background))), motiondetector.py:232, half to even)
        const uint32_t bsum = (uint32_t)(-nbsum);
        double mine = 0.0;
        bool sets = false;
        if (valid && t == 0) {
            mine = (double)bsum / (double)g.ncrop;
            sets = true;
        } else if (valid && upd && changed) {
            mine = rounded_background_average(bsum, (uint32_t)g.ncrop);
            sets = true;
        }
        const uint32_t set_mask = __ballot_sync(0xffffffffu, sets);
        const uint32_t below = set_mask & (0xffffffffu >> (31 - lane));  // lanes <= this one
        const int src = below ? 31 - __clz((int)below) : lane;
        const double got = __shfl_sync(0xffffffffu, mine, src);
        const double avg_here = below ? got : average;
        average = __shfl_sync(0xffffffffu, avg_here, 31);
        frames_seen += __popc(__ballot_sync(0xffffffffu, valid && upd));
        if (is_frame) {
            const FrameScalars fs = frame_scalars_of(psum, fmin, fmax, avg_here, clip.background_thresh, npx);
            a.info[o] = frame_info_of(fs, avg_here, psum, fmin, fmax, want_stats, pmin, pmax, fabs_sum, denoise ? ((t > 0) ? 2 : 1) : 0);
            FrameHdr h;
            h.nmagic = fs.nmagic; h.nshift = fs.nshift;
            h.flags = kHdrValid | (t == 0 ? kHdrFirst : 0u) | (denoise ? kHdrDenoise : 0u);
            h.threshold = fs.thr; h.avg_change = fs.ac; h.norm_min = fs.gmn; h.norm_max = fs.gmx;
            h.hot_strips = 0;
            bool dense = fs.fth == INT32_MIN;
#pragma unroll
            for (int sidx = 0; sidx < kMaxStrips; ++sidx) {
                int th = 127;
                if (sidx < NS && !dense) {
                    // stored b = clamp(max F - ref, -128, 127); hot <=> b >= clamp(fth - ref, ., 127): a superset of
                    // max F >= fth whenever fth - ref >= -127 (else every quad of the strip could be hot: dense frame)
                    const long long dq = (long long)fs.fth - (long long)ref_s[sidx];
                    if (dq < -127) dense = true;
                    th = (int)min(dq, 127ll);
                    if (fmax_s[sidx] >= fs.fth) h.hot_strips |= 1u << sidx;
                }
                h.theta[sidx] = (int16_t)th;
            }
            if (dense) { h.flags |= kHdrDense; h.hot_strips = 0xffffffffu; }
            uint4 *hp = reinterpret_cast<uint4 *>(a.fhdr + o);
            const uint4 *hs = reinterpret_cast<const uint4 *>(&h);
            hp[0] = hs[0]; hp[1] = hs[1]; hp[2] = hs[2]; hp[3] = hs[3];
        }
        if (t == n - 1) { last_fmin = fmin; last_fmax = fmax; }
    }
    if (a.state) {
        // header of the clip's state record (the strips wrote background, counters, sums and the last filtered image)
        const int holder = n > 0 ? (n - 1) & 31 : 0;
        last_fmin = __shfl_sync(0xffffffffu, last_fmin, holder);
        last_fmax = __shfl_sync(0xffffffffu, last_fmax, holder);
        if (lane == 0) {
            StateHeader *hd = reinterpret_cast<StateHeader *>(a.state + (size_t)ci * state_bytes(npx));
            hd->average = average;
            hd->frames_seen = frames_seen;
            hd->initialised = 1;
            hd->prev_fmin = n > 0 ? last_fmin : 0;
            hd->prev_fmax = n > 0 ? last_fmax : 0;
            hd->have_prev = n > 0 ? 1 : 0;
        }
    }
}

}  // namespace cpt
