// extract_kernel.cu -- the extraction kernels (launch plans and stages: cptrack_kernels.cuh, DESIGN.md section 3.1).
//
// extract_clips_kernel: one CTA per clip, three roles that run concurrently on consecutive frames:
//   sweep warps (19):     frame t+2: the recurrence -- background update of the previous frame fused with K1 / K7 sum / K8
//   mask warps (4):       frame t+1: scalars (K2), hot quads -> work lists, normalise (K2), blur + threshold (K4)
//   component warps (8):  frame t:   close, run-based labelling, statistics, variance (K4, K5, K6)
//   Messages (frame sums + per-quad maxima, then the thresholded bit image) are double buffered and handed over
//   with named barriers (full / empty per buffer); everything else the roles touch is disjoint shared memory.
// Split path: after strip_sweep_kernel and frame_scalars_kernel (strip_sweep.cu), frame_regions_kernel /
//   frame_components_kernel / region_variance_kernel do the per-frame stages one CTA (warp) per frame.
#include "cptrack_kernels.cuh"

namespace cpt {

namespace {

// Optional phase timing (build with -DCPT_PHASE_TIMING): thread 0 of each role accumulates clock64()
// deltas per phase into a.debug[blockIdx.x][32].
#ifdef CPT_PHASE_TIMING
#define CPT_TICK_START(cond) long long tick_last_ = clock64(); (void)tick_last_
#define CPT_TICK(cond, i)                                                                     \
    do {                                                                                      \
        if ((cond) && a.debug) {                                                              \
            long long now_ = clock64();                                                       \
            atomicAdd((unsigned long long *)&a.debug[(blockIdx.x % 128u) * 32 + (i)], (unsigned long long)(now_ - tick_last_)); \
            tick_last_ = now_;                                                                \
        }                                                                                     \
    } while (0)
#define CPT_COUNT(cond, i, v) do { if ((cond) && a.debug) atomicAdd((unsigned long long *)&a.debug[(blockIdx.x % 128u) * 32 + (i)], (unsigned long long)(v)); } while (0)
#define CPT_TICK_START2(cond) long long tick2_last_ = clock64(); (void)tick2_last_
#define CPT_TICK2(cond, i)                                                                    \
    do {                                                                                      \
        if ((cond) && a.debug) {                                                              \
            long long now_ = clock64();                                                       \
            atomicAdd((unsigned long long *)&a.debug[(blockIdx.x % 128u) * 32 + (i)], (unsigned long long)(now_ - tick2_last_)); \
            tick2_last_ = now_;                                                               \
        }                                                                                     \
    } while (0)
#else
#define CPT_COUNT(cond, i, v) do { } while (0)
#define CPT_TICK_START2(cond) do { } while (0)
#define CPT_TICK2(cond, i) do { } while (0)
#define CPT_TICK_START(cond) do { } while (0)
#define CPT_TICK(cond, i) do { } while (0)
#endif

enum : int {
    BAR_P = 1, BAR_M = 2, BAR_C = 3,               // inside a role
    BAR_SM_FULL = 4, BAR_SM_EMPTY = 6,             // sweep -> mask warps (+buffer)
    BAR_FULL = 8, BAR_EMPTY = 10,                  // mask -> component warps (+buffer)
    BAR_DONE = 12, BAR_INIT = 13,
    BAR_QFREE = 14                                 // mask -> sweep warps: Smem::qmax8 has been consumed
};

// quad maximum of a slot the thread does not own / of a pass without a frame: far below any F, and kNoQuad - qref cannot wrap
constexpr int kNoQuad = -(1 << 30);
// the byte stored for a quad: max F relative to qref, saturated to int8
__device__ __forceinline__ int8_t quad_byte(int gmax, int qref) {
    int d;
    asm("cvt.sat.s8.s32 %0, %1;" : "=r"(d) : "r"(gmax - qref));
    return (int8_t)d;
}
__device__ __forceinline__ void bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void bar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ bool bar_or(int id, int n, bool pred) {
    int r;
    asm volatile(
        "{\n\t.reg .pred p, q;\n\tsetp.ne.s32 q, %3, 0;\n\tbar.red.or.pred p, %1, %2, q;\n\tselp.s32 %0, 1, 0, p;\n\t}"
        : "=r"(r)
        : "r"(id), "r"(n), "r"((int)pred)
        : "memory");
    return r != 0;
}

__device__ __forceinline__ const uint16_t *frame_ptr(const KernelArgs &a, const cpt_clip &c, int t) {
    int64_t idx = c.ring_frames ? (int64_t)((c.first_frame + t) % c.ring_frames) : (int64_t)t;
    return a.frames + (size_t)(c.frame_offset + idx) * a.g.npx;
}

__device__ __forceinline__ float *filtered_ptr(const KernelArgs &a, const cpt_clip &c, float *scratch, int t) {
    // frame t's fp32 filtered image: the caller's output, or an 8-deep per-CTA ring (the sweep warps may run four
    // frames ahead of the component warps, which read frames t and t-1)
    return a.filtered ? a.filtered + (size_t)(c.out_offset + t) * a.g.npx : scratch + (size_t)(t & 7) * a.g.npx;
}

// Replicate the edge_pixels border of B from the crop interior (motiondetector.py:239-244 copies rows,
// then columns; the net effect is "clamp the coordinate into the crop rectangle").  No barrier inside.
__device__ __forceinline__ void replicate_edges(Smem &s, const Geometry &g, int ptid) {
    const int W = g.W, H = g.H, e = g.edge;
    if (e == 0) return;
    const int per_row_pair = 2 * e * W;           // top and bottom bands
    const int side = 2 * e * (H - 2 * e);         // left and right bands of the interior rows
    for (int i = ptid; i < per_row_pair + side; i += kPThreads) {
        int y, x;
        if (i < per_row_pair) {
            int r = i / W;
            x = i - r * W;
            y = (r < e) ? r : H - 2 * e + r;
        } else {
            int k = i - per_row_pair, r = k / (2 * e), c = k - r * 2 * e;
            y = e + r;
            x = (c < e) ? c : W - 2 * e + c;
        }
        int sy = min(max(y, e), H - 1 - e), sx = min(max(x, e), W - 1 - e);
        s.B[y * W + x] = s.B[sy * W + sx];
    }
}

// normalize(F, new_max=255) of get_delta_frame (track/cliptracker.py:249-261), cast to fp32.
// exact_f32: 255*(max-min) < 2^24, so numerator and denominator are exact fp32 integers and the
// fp32 IEEE quotient is the correctly rounded value the reference's fp64-then-cast produces.
__device__ __forceinline__ float norm255(int f, int mn, int mx, bool exact_f32) {
    if (mx == mn) return (mx == 0) ? 0.0f : (exact_f32 ? __fdiv_rn((float)f, (float)mx) : (float)((double)f / (double)mx));
    if (exact_f32) return __fdiv_rn((float)(255 * (f - mn)), (float)(mx - mn));
    return (float)(255.0 * ((double)f - (double)mn) / ((double)mx - (double)mn));
}

// norm255's exact_f32 for the two frames of a delta frame
__device__ __forceinline__ bool norm255_exact(int cur_fmin, int cur_fmax, int prev_fmin, int prev_fmax) {
    return 255ll * max(cur_fmax - cur_fmin, prev_fmax - prev_fmin) < (1ll << 24) &&
           max(max(abs(cur_fmax), abs(cur_fmin)), max(abs(prev_fmax), abs(prev_fmin))) < (1 << 24);
}

// K6 for one region record: variance of |norm255(F_t) - norm255(F_t-1)| over the component's bounding box (l, tp, bw, bh);
// one warp, lane 0 stores it to *var.  Every frame's variances are summed in this one order (pixels lane, lane + 32, ...
// of the box, then one shuffle tree), whichever kernel computes them.  kLdg: the images are read-only for the whole launch
// (region_variance_kernel); the extraction kernel reads images its own launch wrote, through coherent loads.
template <bool kLdg>
__device__ __forceinline__ void region_variance(const Geometry &g, int l, int tp, int bw, int bh, const float *fcur,
                                                const float *fprev, int cur_fmin, int cur_fmax, int prev_fmin, int prev_fmax,
                                                bool exact, int lane, double *var) {
    const int npix = bw * bh;
    double s1 = 0.0, s2 = 0.0;
    const uint32_t rcp = 0xffffffffu / (uint32_t)bw + 1u;  // i / bw == umulhi(i, rcp) for i * bw < 2^32
    for (int i = lane; i < npix; i += 32) {
        const int yy = bw == 1 ? i : (int)__umulhi((uint32_t)i, rcp), xx = i - yy * bw, p = (tp + yy) * g.W + l + xx;  // (rcp wraps to 0 for bw == 1)
        const float fc = kLdg ? __ldg(fcur + p) : fcur[p], fp = kLdg ? __ldg(fprev + p) : fprev[p];
        const float d = fabsf(norm255((int)fc, cur_fmin, cur_fmax, exact) - norm255((int)fp, prev_fmin, prev_fmax, exact));
        s1 += (double)d;
        s2 += (double)d * (double)d;
    }
    for (int off = 16; off; off >>= 1) {
        s1 += __shfl_xor_sync(0xffffffffu, s1, off);
        s2 += __shfl_xor_sync(0xffffffffu, s2, off);
    }
    if (lane == 0) {
        const double cnt = (double)npix, mean = s1 / cnt, v = s2 / cnt - mean * mean;
        *var = v > 0.0 ? v : 0.0;
    }
}

// ================================================================================================
// components of a frame's mask (K4 second half, K5): the passes of both drivers, components_of_frame (component warps,
// frame_components_kernel, mask_components_kernel: full-size tables) and components_lean (frame_regions_kernel).
// Tables C, ST and base hold one entry per word w of the closed mask, word wi of its row of rw words.
// ================================================================================================
// closed word C[y] = M[y-1] | (M[y] & M[y-2]) (C[0] = M[0]) of mask word w, image row y
__device__ __forceinline__ uint32_t closed_word(const uint32_t *M, int w, int y, int rw) {
    const uint32_t m0 = M[w];
    return y == 0 ? m0 : M[w - rw] | (m0 & (y >= 2 ? M[w - 2 * rw] : 0u));
}

// run-start bits of closed word c = C[w] into ST[w], and the runs that start in the earlier words of its row into base[w]
template <class SM>
__device__ __forceinline__ uint32_t word_run_starts(SM &s, int w, int wi, uint32_t c, int &base) {
    uint32_t carry = 0;
    base = 0;
    for (int q = 0; q < wi; ++q) {
        const uint32_t cq = s.C[w - wi + q];
        base += __popc(cq & ~((cq << 1) | carry));
        carry = cq >> 31;
    }
    const uint32_t stw = c & ~((c << 1) | carry);
    s.ST[w] = stw;
    s.base[w] = (uint8_t)base;
    return stw;
}

// 8-connectivity: unions of the runs of closed word c = C[w] (row `row` > 0 of the table) with the runs of the row above
template <class SM>
__device__ __forceinline__ void unite_with_row_above(SM &s, int w, int wi, int rw, uint32_t c, int row, int rpr) {
    const int up = w - rw;
    const uint32_t u = s.C[up];
    const uint32_t u_l = (wi > 0) ? (s.C[up - 1] >> 31) : 0u, u_r = (wi + 1 < rw) ? (s.C[up + 1] & 1u) : 0u;
    const uint32_t c_l = (wi > 0) ? (s.C[w - 1] >> 31) : 0u, c_r = (wi + 1 < rw) ? (s.C[w + 1] & 1u) : 0u;
    const uint32_t ul = (u << 1) | u_l, ur = (u >> 1) | (u_r << 31);
    const uint32_t cl = (c << 1) | c_l, cr = (c >> 1) | (c_r << 31);
    uint32_t needA = c & u & ~(cl & ul);   // pixel above, unless the left neighbour already links to it
    uint32_t needB = c & ul & ~u & ~cl;    // upper-left only
    uint32_t needC = c & ur & ~u & ~cr;    // upper-right only
    const int w0 = w - wi, u0 = up - wi, xb = wi * 32;
    while (needA) {
        const int b = __ffs(needA) - 1;
        needA &= needA - 1;
        uf_union(s.parent, run_id(s, w0, row, rpr, xb + b), run_id(s, u0, row - 1, rpr, xb + b));
    }
    while (needB) {
        const int b = __ffs(needB) - 1;
        needB &= needB - 1;
        uf_union(s.parent, run_id(s, w0, row, rpr, xb + b), run_id(s, u0, row - 1, rpr, xb + b - 1));
    }
    while (needC) {
        const int b = __ffs(needC) - 1;
        needC &= needC - 1;
        uf_union(s.parent, run_id(s, w0, row, rpr, xb + b), run_id(s, u0, row - 1, rpr, xb + b + 1));
    }
}

template <class SM>
__device__ __forceinline__ void reset_slot(SM &s, int i) {
    s.c_key[i] = INT32_MAX; s.c_area[i] = 0; s.c_sx[i] = 0; s.c_sy[i] = 0;
    s.c_l[i] = INT32_MAX; s.c_t[i] = INT32_MAX; s.c_r[i] = -1; s.c_b[i] = -1;
}

// length of the run that starts at bit b of closed word c = C[w]
template <class SM>
__device__ __forceinline__ int run_length(const SM &s, int w, int wi, int rw, uint32_t c, int b) {
    const uint32_t inv = ~(c >> b);
    int len = (inv == 0) ? 32 : (__ffs(inv) - 1);
    if (b + len >= 32) {  // run continues into the following words
        len = 32 - b;
        for (int q = wi + 1; q < rw; ++q) {
            const uint32_t cn = ~s.C[w - wi + q];
            if (cn == 0) { len += 32; continue; }
            len += __ffs(cn) - 1;
            break;
        }
    }
    return len;
}

// the run of len pixels from (xs, y) into the statistics of its component's slot
template <class SM>
__device__ __forceinline__ void add_run(SM &s, const Geometry &g, int slot, int xs, int y, int len) {
    atomicMin(&s.c_key[slot], (y >> 1) * g.block_w + (xs >> 1));
    atomicAdd(&s.c_area[slot], len);
    atomicAdd(&s.c_sx[slot], len * (2 * xs + len - 1) / 2);
    atomicAdd(&s.c_sy[slot], len * y);
    atomicMin(&s.c_l[slot], xs);
    atomicMax(&s.c_r[slot], xs + len - 1);
    atomicMin(&s.c_t[slot], y);
    atomicMax(&s.c_b[slot], y);
}

// OpenCV label order: rank of slot i among slots 0 .. nslots - 1 by the key of the component's first 2x2 block
template <class SM>
__device__ __forceinline__ int slot_rank(const SM &s, int i, int nslots) {
    const int key = s.c_key[i];
    int rank = 0;
    for (int q = 0; q < nslots; ++q) rank += (s.c_key[q] < key);
    return rank;
}

// region record of slot i; pixel_variance is K6's
template <class SM>
__device__ __forceinline__ cpt_region region_record(const SM &s, int i) {
    cpt_region r;
    r.x = s.c_l[i]; r.y = s.c_t[i];
    r.width = s.c_r[i] - r.x + 1; r.height = s.c_b[i] - r.y + 1;
    r.area = s.c_area[i]; r.sum_x = s.c_sx[i]; r.sum_y = s.c_sy[i];
    r.key = s.c_key[i];
    r.pixel_variance = 0.0;
    return r;
}

__device__ __forceinline__ void store_label_run(uint8_t *lab_frame, const Geometry &g, int xs, int y, int len, uint8_t lab) {
    uint8_t *px = lab_frame + y * g.W + xs;
    for (int k = 0; k < len; ++k) px[k] = lab;
}

struct RunCursor {
    uint32_t c, stw;
    int y, wi, base;
};

// K4 second half + K5 for the mask in s.M[buf]: close, labelling, statistics, label image and region records of output
// frame o.  Called by all kT threads of the role (kBar: their named barrier).  var_deferred: region_variance_kernel computes
// the frame's variances (info.reserved[0]).  Returns the number of region records.
template <class SM, int kT, int kBar>
__device__ int components_of_frame(const KernelArgs &a, SM &s, const Geometry &g, int ctid, int buf, size_t o, bool var_deferred) {
    const int rw = g.row_words;
    constexpr int kIter = (kMaxWords + kT - 1) / kT;  // 3
    RunCursor rc[kIter];
    bool any = false;
    CPT_TICK_START2(ctid == 0);
    // ---- close; slot tables reset
#pragma unroll
    for (int it = 0; it < kIter; ++it) {
        int w = ctid + it * kT;
        rc[it].c = 0; rc[it].stw = 0; rc[it].y = 0; rc[it].wi = 0; rc[it].base = 0;
        if (w < g.words) {
            int y = (int)(((uint32_t)w * g.rw_magic) >> 13);
            const uint32_t c = closed_word(s.M[buf], w, y, rw);
            s.C[w] = c;
            rc[it].c = c; rc[it].y = y; rc[it].wi = w - y * rw;
            any |= (c != 0);
        }
    }
    // (a component's slot is initialised by the thread that allocates it; only the overflow sink is reset here)
    if (ctid == 0) {
        s.ncomp = 0;
        reset_slot(s, CPT_MAX_COMPONENTS);
    }
    if (!bar_or(kBar, kT, any)) return 0;  // no foreground: info.n_components stays 0
    CPT_TICK2(ctid == 0, 20);  // close + reset + barrier

    // ---- run starts and ids
#pragma unroll
    for (int it = 0; it < kIter; ++it) {
        int w = ctid + it * kT;
        if (w < g.words && rc[it].c != 0) {  // (ST / base of an empty word are never looked up)
            int base;
            const uint32_t stw = word_run_starts(s, w, rc[it].wi, rc[it].c, base);
            rc[it].stw = stw; rc[it].base = base;
            int id = rc[it].y * kRunsPerRow + base;
            for (uint32_t bitsleft = stw; bitsleft; bitsleft &= bitsleft - 1, ++id) s.parent[id] = (uint16_t)id;
        }
    }
    bar_sync(kBar, kT);
    CPT_TICK2(ctid == 0, 21);  // run starts + barrier
    // ---- unions with the row above
#pragma unroll
    for (int it = 0; it < kIter; ++it) {
        int w = ctid + it * kT;
        if (w < g.words && rc[it].y > 0 && rc[it].c != 0) unite_with_row_above(s, w, rc[it].wi, rw, rc[it].c, rc[it].y, kRunsPerRow);
    }
    bar_sync(kBar, kT);
    CPT_TICK2(ctid == 0, 22);  // unions + barrier
    // ---- roots -> component slots
#pragma unroll
    for (int it = 0; it < kIter; ++it) {
        uint32_t bitsleft = rc[it].stw;
        int n = 0;
        while (bitsleft) {
            bitsleft &= bitsleft - 1;
            int id = rc[it].y * kRunsPerRow + rc[it].base + n;
            if (s.parent[id] == id) {
                int slot = atomicAdd(&s.ncomp, 1);
                if (slot < CPT_MAX_COMPONENTS) reset_slot(s, slot);
                s.parent[id] = (uint16_t)(kSlotFlag | (slot < CPT_MAX_COMPONENTS ? slot : CPT_MAX_COMPONENTS));
            }
            ++n;
        }
    }
    bar_sync(kBar, kT);
    CPT_TICK2(ctid == 0, 23);  // roots + barrier
    const int ncomp = s.ncomp;
    if (ncomp > CPT_MAX_COMPONENTS) {
        // More components than slots, and the slots above went in scheduling order.  Hand them again, to the components that
        // come first in OpenCV label order: each root's parent entry takes the least key of its runs (keys are unique per
        // component: the pixels of a 2x2 block are all 8-connected), a bitmap over the keys ranks them, and the first
        // CPT_MAX_COMPONENTS ranks are the slots.  The bitmap lives in c_area until the slot tables are reset.
        static_assert(((kMaxH + 1) / 2) * ((kMaxW + 1) / 2) <= 32 * kCompSlots && ((kMaxH + 1) / 2) * ((kMaxW + 1) / 2) < 0x7fff,
                      "a bit per key fits in c_area, and a key in a parent entry");
        uint32_t *keybits = reinterpret_cast<uint32_t *>(s.c_area);
        const int nkw = (((g.H + 1) >> 1) * g.block_w + 31) >> 5;
        for (int i = ctid; i < nkw; i += kT) keybits[i] = 0u;
#pragma unroll
        for (int it = 0; it < kIter; ++it) {
            const int id0 = rc[it].y * kRunsPerRow + rc[it].base, n = __popc(rc[it].stw);
            for (int k = 0; k < n; ++k)
                if (s.parent[id0 + k] & kSlotFlag) s.parent[id0 + k] = (uint16_t)(kSlotFlag | 0x7fffu);
        }
        bar_sync(kBar, kT);
#pragma unroll
        for (int it = 0; it < kIter; ++it) {
            uint32_t bitsleft = rc[it].stw;
            int id = rc[it].y * kRunsPerRow + rc[it].base;
            while (bitsleft) {
                const int b = __ffs(bitsleft) - 1;
                bitsleft &= bitsleft - 1;
                const int root = uf_find(s.parent, id++);
                const unsigned short key = (unsigned short)(kSlotFlag | ((rc[it].y >> 1) * g.block_w + ((rc[it].wi * 32 + b) >> 1)));
                unsigned short *p = reinterpret_cast<unsigned short *>(s.parent + root);
                for (unsigned short old = *(volatile unsigned short *)p; key < old;) {
                    const unsigned short seen = atomicCAS(p, old, key);
                    if (seen == old) break;
                    old = seen;
                }
            }
        }
        bar_sync(kBar, kT);
#pragma unroll
        for (int it = 0; it < kIter; ++it) {
            const int id0 = rc[it].y * kRunsPerRow + rc[it].base, n = __popc(rc[it].stw);
            for (int k = 0; k < n; ++k) {
                const int p = s.parent[id0 + k];
                if (p & kSlotFlag) atomicOr(&keybits[(p & 0x7fff) >> 5], 1u << (p & 31));
            }
        }
        bar_sync(kBar, kT);
#pragma unroll
        for (int it = 0; it < kIter; ++it) {
            const int id0 = rc[it].y * kRunsPerRow + rc[it].base, n = __popc(rc[it].stw);
            for (int k = 0; k < n; ++k) {
                const int p = s.parent[id0 + k];
                if (!(p & kSlotFlag)) continue;
                const int key = p & 0x7fff;
                int rank = __popc(keybits[key >> 5] & ((1u << (key & 31)) - 1u));
                for (int q = 0; q < (key >> 5); ++q) rank += __popc(keybits[q]);
                s.parent[id0 + k] = (uint16_t)(kSlotFlag | min(rank, CPT_MAX_COMPONENTS));
            }
        }
        bar_sync(kBar, kT);
        for (int slot = ctid; slot < CPT_MAX_COMPONENTS; slot += kT) reset_slot(s, slot);
        bar_sync(kBar, kT);
    }
    // ---- per-run statistics into the slot tables
#pragma unroll
    for (int it = 0; it < kIter; ++it) {
        const int w = ctid + it * kT;
        uint32_t bitsleft = rc[it].stw;
        int id = rc[it].y * kRunsPerRow + rc[it].base;
        while (bitsleft) {
            const int b = __ffs(bitsleft) - 1;
            bitsleft &= bitsleft - 1;
            const int slot = uf_slot(s.parent, id);
            s.parent[id++] = (uint16_t)(kSlotFlag | slot);
            add_run(s, g, slot, rc[it].wi * 32 + b, rc[it].y, run_length(s, w, rc[it].wi, rw, rc[it].c, b));
        }
    }
    bar_sync(kBar, kT);
    CPT_TICK2(ctid == 0, 24);  // run statistics + barrier
    const int nslots = min(ncomp, CPT_MAX_COMPONENTS);
    const int nout = min(nslots, g.max_regions);
    for (int i = ctid; i < nslots; i += kT) s.c_rank[i] = (uint8_t)slot_rank(s, i, nslots);
    bar_sync(kBar, kT);
    CPT_TICK2(ctid == 0, 25);  // rank + barrier
    // ---- label image: the pixel warps already stored zeros for this frame; write the runs
    if (a.labels) {
        uint8_t *lab_frame = a.labels + o * g.npx;
#pragma unroll
        for (int it = 0; it < kIter; ++it) {
            const int w = ctid + it * kT;
            uint32_t bitsleft = rc[it].stw;
            int id = rc[it].y * kRunsPerRow + rc[it].base;
            while (bitsleft) {
                const int b = __ffs(bitsleft) - 1;
                bitsleft &= bitsleft - 1;
                const int slot = s.parent[id++] & 0xff;
                const uint8_t lab = (slot < CPT_MAX_COMPONENTS) ? (uint8_t)(s.c_rank[slot] + 1) : (uint8_t)255;
                store_label_run(lab_frame, g, rc[it].wi * 32 + b, rc[it].y, run_length(s, w, rc[it].wi, rw, rc[it].c, b), lab);
            }
        }
    }
    CPT_TICK2(ctid == 0, 26);  // label writes
    for (int i = ctid; i < nslots; i += kT) {
        const int rank = s.c_rank[i];
        if (rank < nout) a.regions[o * g.max_regions + rank] = region_record(s, i);
    }
    if (ctid == 0) {
        a.info[o].n_components = ncomp;
        if (var_deferred) a.info[o].reserved[0] = 1;  // region_variance_kernel fills pixel_variance
    }
    return nout;
}

__device__ void component_warps(const KernelArgs &a, Smem &s, const cpt_clip &clip, int ctid, float *scratch,
                                const StateHeader *st_hdr, const float *st_F) {
    const Geometry &g = a.g;
    const int lane = ctid & 31;
    int prev_fmin = 0, prev_fmax = 0;
    bool have_prev = false;
    if (clip.flags & CPT_CLIP_RESUME) {
        prev_fmin = st_hdr->prev_fmin;
        prev_fmax = st_hdr->prev_fmax;
        have_prev = st_hdr->have_prev != 0;
    }
    // denoise clips: the pixel warps only emit the normalised image; masks and components come from the
    // NLM + mask_components passes that follow the launch
    const int n_here = (clip.flags & CPT_CLIP_DENOISE) ? 0 : clip.n_frames;
    bar_sync(BAR_INIT, kThreads);
    for (int t = 0; t < n_here; ++t) {
        CPT_TICK_START(ctid == 0);
        const int buf = t & 1;
        bar_sync(BAR_FULL + buf, kMThreads + kCThreads);  // mask of frame t is in s.M[buf]
        CPT_TICK(ctid == 0, 11);  // waiting for a mask
        const int cur_fmin = s.msg[buf][0], cur_fmax = s.msg[buf][1];
        const size_t o = (size_t)(clip.out_offset + t);
        // frames after the first of a launch have both filtered images in the caller's buffer: their variances
        // are left to region_variance_kernel (a wide second launch) instead of this 7-warp critical path
        const bool var_later = a.defer_variance && t > 0;
        const int nout = components_of_frame<Smem, kCThreads, BAR_C>(a, s, g, ctid, buf, o, have_prev && var_later);
        if (have_prev && !var_later && nout > 0) {
            // K6 of the other frames: one warp per region record
            CPT_TICK_START2(ctid == 0);
            bar_sync(BAR_C, kCThreads);  // the records are stored
            const float *fcur = filtered_ptr(a, clip, scratch, t);
            const float *fprev = (t == 0) ? st_F : filtered_ptr(a, clip, scratch, t - 1);
            const bool exact = norm255_exact(cur_fmin, cur_fmax, prev_fmin, prev_fmax);
            for (int r = ctid >> 5; r < nout; r += kCWarps) {
                cpt_region *reg = a.regions + o * g.max_regions + r;
                region_variance<false>(g, reg->x, reg->y, reg->width, reg->height, fcur, fprev, cur_fmin, cur_fmax, prev_fmin,
                                       prev_fmax, exact, lane, &reg->pixel_variance);
            }
            CPT_TICK2(ctid == 0, 27);  // variance + barrier (0 for the frames left to region_variance_kernel)
        }
        prev_fmin = cur_fmin;
        prev_fmax = cur_fmax;
        have_prev = true;
        // all component threads are past the close, the only reader of s.M[buf]: hand it back zeroed, the pixel warps
        // only write the bytes of the groups they blurred
        for (int i = ctid; i < g.words; i += kCThreads) s.M[buf][i] = 0;
        CPT_TICK(ctid == 0, 12);  // components of the frame
        if (t + 2 < n_here) bar_arrive(BAR_EMPTY + buf, kMThreads + kCThreads);
    }
    // the saved state (previous filtered frame, header) may be overwritten now
    bar_arrive(BAR_DONE, kThreads);
}

// ================================================================================================
// pixel warps
// ================================================================================================

// K4 first half for one group of 8 pixels: 5x5 binomial blur of s.U (fixed point, one rounding,
// BORDER_REFLECT_101) in packed 16-bit lanes and threshold `> ith` -> one byte of the bit rows in s.M[buf].
// Only outputs of the marked quads (q2: one bit per quad of the group) are evaluated: the others cannot exceed the threshold (every input
// of their window is <= ith) and their windows may reach inputs that were not refreshed.
// u_row0: image row held by the first row of s.U (frame_regions_kernel keeps one band of rows; 0 everywhere else); or_bits:
// the byte is OR-ed into the mask (bands overlap) instead of stored.
template <class SM>
__device__ __forceinline__ void blur_group(SM &s, const Geometry &g, int grp, uint32_t q2, int buf, int ith, int u_row0 = 0,
                                           bool or_bits = false) {
    const int W = g.W, H = g.H;
    uint8_t *M8 = reinterpret_cast<uint8_t *>(s.M[buf]);
    const uint32_t T = (ith >= 0 && ith < 255) ? (uint32_t)(((ith + 1) << 8) - 128) : 0u;
    const int y = (int)(((uint32_t)grp * g.gpr_magic) >> 17), gx = grp - y * g.gpr, x0 = gx * 8;
    uint32_t bits = 0;
    if (ith < 0) {
        bits = 0xffu;
    } else if (ith < 255 && q2) {
        uint32_t V[6] = {0, 0, 0, 0, 0, 0};
        const bool left_edge = (x0 == 0), right_edge = (x0 + 8 == W);
#pragma unroll
        for (int r = 0; r < 5; ++r) {
            const uint32_t wgt = (r == 0 || r == 4) ? 1u : ((r == 2) ? 6u : 4u);
            int yy = y + r - 2;
            yy = (yy < 0) ? -yy : yy;              // H >= 4: one reflection is enough
            yy = (yy >= H) ? 2 * H - 2 - yy : yy;
            const uint8_t *row = s.U + (yy - u_row0) * W + x0;
            uint2 m = *reinterpret_cast<const uint2 *>(row);
            uint32_t lw = left_edge ? 0u : *reinterpret_cast<const uint32_t *>(row - 4);
            uint32_t rw = right_edge ? 0u : *reinterpret_cast<const uint32_t *>(row + 8);
            uint32_t lp = left_edge ? __byte_perm(m.x, 0, 0x4142) : __byte_perm(lw, 0, 0x4342);
            uint32_t rp = right_edge ? __byte_perm(m.y, 0, 0x4142) : __byte_perm(rw, 0, 0x4140);
            V[0] += wgt * lp;
            V[1] += wgt * __byte_perm(m.x, 0, 0x4140);
            V[2] += wgt * __byte_perm(m.x, 0, 0x4342);
            V[3] += wgt * __byte_perm(m.y, 0, 0x4140);
            V[4] += wgt * __byte_perm(m.y, 0, 0x4342);
            V[5] += wgt * rp;
        }
        uint32_t odd[5];
#pragma unroll
        for (int q = 0; q < 5; ++q) odd[q] = __byte_perm(V[q], V[q + 1], 0x5432);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            uint32_t sum = V[q] + V[q + 2] + 6u * V[q + 1] + 4u * (odd[q] + odd[q + 1]);
            bits |= ((sum & 0xffffu) >= T ? 1u : 0u) << (2 * q);
            bits |= ((sum >> 16) >= T ? 1u : 0u) << (2 * q + 1);
        }
        bits &= ((q2 & 1u) ? 0x0fu : 0u) | ((q2 & 2u) ? 0xf0u : 0u);
    }
    if (or_bits) M8[y * g.row_words * 4 + gx] |= (uint8_t)bits;
    else M8[y * g.row_words * 4 + gx] = (uint8_t)bits;
}

// K2 for one group of 8 pixels: U = uint8(255 * (G - min) / (max - min)), G = max(F - avg_change, 0) with F the
// filtered image the sweep wrote (exact integers), in the reference's own fp32 arithmetic
// (imageprocessing.py:151-169: multiply, then IEEE divide, truncate).
template <class SM>
__device__ __forceinline__ void normalise_values(SM &s, const float4 f0, const float4 f1, int grp, int ac, int gmn, int gmx,
                                                 uint32_t nmagic, int nshift, uint8_t *u_global = nullptr, int u_off = 0) {
    const float fv[8] = {f0.x, f0.y, f0.z, f0.w, f1.x, f1.y, f1.z, f1.w};
    const bool degenerate = (gmx == gmn);
    const float range_f = (float)gmx - (float)gmn;
    const uint32_t degen_val = (gmx == 0) ? 0u : 1u;
    uint32_t u[8];
    if (nmagic) {
        // exact integer form of the fp32 quotient (see norm_u8_int): no divide on the mask warps' critical path
#pragma unroll
        for (int i = 0; i < 8; ++i) u[i] = norm_u8_int(max((int)fv[i] - ac, 0) - gmn, nmagic, nshift);
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int gv = max((int)fv[i] - ac, 0) - gmn;  // G - min
            u[i] = degenerate ? degen_val : norm_u8(gv, range_f);
        }
    }
    uint2 w;
    w.x = u[0] | (u[1] << 8) | (u[2] << 16) | (u[3] << 24);
    w.y = u[4] | (u[5] << 8) | (u[6] << 16) | (u[7] << 24);
    if (u_global) *reinterpret_cast<uint2 *>(u_global + grp * 8) = w;
    else *reinterpret_cast<uint2 *>(s.U + (grp * 8 - u_off)) = w;
}

template <class SM>
__device__ __forceinline__ void normalise_group(SM &s, const float *F, int grp, int ac, int gmn, int gmx,
                                                uint32_t nmagic, int nshift, uint8_t *u_global = nullptr, int u_off = 0) {
    // written by the sweep warps of this CTA a moment ago: plain (coherent) loads, an L2 hit
    const float4 f0 = *reinterpret_cast<const float4 *>(F + grp * 8), f1 = *reinterpret_cast<const float4 *>(F + grp * 8 + 4);
    normalise_values(s, f0, f1, grp, ac, gmn, gmx, nmagic, nshift, u_global, u_off);
}

// Work lists, one row at a time: near = the row's hot-quad bits OR-ed over the rows around it (bit q: quad q), rowmask = the
// row's quads.  Group g of the row is listed, as row_grp + g, if either of its quads (bits 2g, 2g + 1) is marked; count is
// the list's length in shared memory (one atomic per row).  kCapped: entries from kListCap on are counted, not stored (the
// single kernel turns an overflow into dense work; frame_regions_kernel's lists hold every group of a band).
// emit_norm_groups: the groups to normalise, the marks widened by two quads.
template <bool kCapped>
__device__ __forceinline__ void emit_norm_groups(unsigned long long near, unsigned long long rowmask, int row_grp, int *count,
                                                 uint16_t *list) {
    if (!near) return;
    const unsigned long long mk = (near | (near << 1) | (near >> 1) | (near << 2) | (near >> 2)) & rowmask;
    unsigned long long grp_bits = (mk | (mk >> 1)) & 0x5555555555555555ull;
    int base = atomicAdd(count, __popcll(grp_bits));
    while (grp_bits) {
        const int bit = __ffsll((long long)grp_bits) - 1;
        grp_bits &= grp_bits - 1;
        if (kCapped && base >= kListCap) { ++base; continue; }
        list[base++] = (uint16_t)(row_grp + (bit >> 1));
    }
}

// emit_blur_groups: the groups to blur, the marks widened by one quad; an entry carries the group's two quad marks in
// bits 14-15 (blur_group's q2).
template <bool kCapped>
__device__ __forceinline__ void emit_blur_groups(unsigned long long near, unsigned long long rowmask, int row_grp, int *count,
                                                 uint16_t *list) {
    if (!near) return;
    const unsigned long long mk = (near | (near << 1) | (near >> 1)) & rowmask;
    unsigned long long grp_bits = (mk | (mk >> 1)) & 0x5555555555555555ull;
    int base = atomicAdd(count, __popcll(grp_bits));
    while (grp_bits) {
        const int bit = __ffsll((long long)grp_bits) - 1;
        grp_bits &= grp_bits - 1;
        if (kCapped && base >= kListCap) { ++base; continue; }
        list[base++] = (uint16_t)((row_grp + (bit >> 1)) | ((uint32_t)((mk >> bit) & 3ull) << 14));
    }
}

// L2 policy of the bulk prefetch of the next frame: a fraction of its lines is kept (evict_last) until the frame is read
// again, 45 frames later, as P_old
__device__ __forceinline__ unsigned long long l2_policy_keep() {
    unsigned long long p;
    // (measured: 0.4 -> 33.9 ms, 1.0 -> 34.3 ms, evict_normal -> 34.5 ms, no hints at all -> 35.1 ms per step)
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 0.4;" : "=l"(p));
    return p;
}
// ------------------------------------------------------------------------------------------------
// The fused pixel sweep.  For every owned quad (4 pixels) in one pass over the on-chip state:
//   [update]  WeightedBackground.process_frame for the PREVIOUS frame (K7): A = floor(S / cnt),
//             keep = B < A - w_k (table form), B' = keep ? B : A, k' = keep ? k + 1 : 0
//   [frame]   K1 for THIS frame against B': F = P - B', S += P - P_old, sum P, min / max F (+ K8 scalars),
//             fp32 filtered store, label image zero fill
// so B, k and S are read and written once per frame.  Border columns live inside owned quads and copy their
// neighbour's B'; border rows are produced by the owner of the adjacent row (edge replication of
// motiondetector.py:239-244 folded into the sweep).
struct SweepMode {
    bool update;      // apply the background update of the previous frame
    bool frame;       // filter the current frame
    bool slow;        // exact unpacked keep test (bounds / 16-bit overflow possible)
    bool first_mean;  // cnt == 1: A = S
    int table;        // 0: thr = k + 1, 1: table in shared memory, 2: table in global memory
    uint32_t magic;   // floor(S / cnt) == umulhi(S, magic)
};

struct SweepAcc {
    uint32_t psum = 0, bsum = 0, changed = 0, fabs_sum = 0;
    uint32_t bmax2 = 0;  // packed uint16 pair
    int fmin = INT32_MAX, fmax = INT32_MIN, pmin = INT32_MAX, pmax = INT32_MIN;
};

__device__ __forceinline__ uint2 ldg8(const void *p) { return __ldg(reinterpret_cast<const uint2 *>(p)); }

// K1 + sliding sum + statistics of one quad against the packed background words nb (2 x 2 pixels)
template <bool kSlide = true>
__device__ __forceinline__ int filter_quad(uint2 pw, uint2 ow, int p4, uint2 nb, uint4 sv, uint32_t *S, float *fcur,
                                           uint8_t *lab_frame, bool want_stats, SweepAcc &acc) {
    const int f0 = dp2a_us(pw.x, kLoP, dp2a_us(nb.x, kLoN, 0)), f1 = dp2a_us(pw.x, kHiP, dp2a_us(nb.x, kHiN, 0));
    const int f2 = dp2a_us(pw.y, kLoP, dp2a_us(nb.y, kLoN, 0)), f3 = dp2a_us(pw.y, kHiP, dp2a_us(nb.y, kHiN, 0));
    if (kSlide) {
        sv.x = (uint32_t)dp2a_us(pw.x, kLoP, dp2a_us(ow.x, kLoN, (int)sv.x));
        sv.y = (uint32_t)dp2a_us(pw.x, kHiP, dp2a_us(ow.x, kHiN, (int)sv.y));
        sv.z = (uint32_t)dp2a_us(pw.y, kLoP, dp2a_us(ow.y, kLoN, (int)sv.z));
        sv.w = (uint32_t)dp2a_us(pw.y, kHiP, dp2a_us(ow.y, kHiN, (int)sv.w));
        *reinterpret_cast<uint4 *>(S + p4) = sv;
    }
    acc.psum = (uint32_t)dp2a_us(pw.x, kBoth, dp2a_us(pw.y, kBoth, (int)acc.psum));
    const int lo = min(min(f0, f1), min(f2, f3)), hi = max(max(f0, f1), max(f2, f3));
    acc.fmin = min(acc.fmin, lo);
    acc.fmax = max(acc.fmax, hi);
    if (want_stats) {
        const int p0 = (int)(pw.x & 0xffffu), p1 = (int)(pw.x >> 16), p2 = (int)(pw.y & 0xffffu), p3 = (int)(pw.y >> 16);
        acc.pmin = min(acc.pmin, min(min(p0, p1), min(p2, p3)));
        acc.pmax = max(acc.pmax, max(max(p0, p1), max(p2, p3)));
        acc.fabs_sum += (uint32_t)(abs(f0) + abs(f1) + abs(f2) + abs(f3));
    }
    *reinterpret_cast<float4 *>(fcur + p4) = make_float4((float)f0, (float)f1, (float)f2, (float)f3);
    if (lab_frame) *reinterpret_cast<uint32_t *>(lab_frame + p4) = 0u;
    return hi;
}

// Per-thread constants of the sweep: thread ptid owns column quad qx of rows r0, r0 + rows_per_it, ... of the
// owned rows (kPThreads = rows_per_it * qpr threads are active: 20 rows x 40 quads at 160 pixels).
struct SweepThread {
    int p4_0;        // pixel index of the thread's first quad
    int stride;      // pixels between its consecutive quads (rows_per_it * W)
    int r0;          // owned-row index of the first quad
    int last_it;     // iteration that holds the last owned row, if this thread owns it; else -1
    int p4_last;     // pixel index of the thread's quad in the last iteration (kQIter - 1), see sweep_thread_init
    bool has_last;   // the thread has a quad in the last iteration
    bool skip0;      // the thread's quad of iteration 0 was handed to another thread (balanced 160x120 mapping)
    int lane;
    bool active;     // ptid < rows_per_it * qpr
    bool prefetch;   // first quad of a 128-byte line
    bool first_col, last_col;  // the quad holds a crop-border column (edge == 1)
    uint32_t perm_x, perm_y;   // crop-border columns copy their neighbour (motiondetector.py:239-244)
    int sel_x, sel_y;          // ... and stay out of the background sum (dp2a selectors)
};

// keep mask (0xffff per kept pixel) of one packed pair (K7: `background < frame - weight` in table form, see
// cptrack_kernels.cuh).  kTable: 0 thr = k + 1 (no bounds), 1 table in shared memory, 2 table in global memory;
// kPacked: 16-bit SIMD form, valid while B + thr cannot overflow 16 bits.
template <bool kPacked, int kTable>
__device__ __forceinline__ uint32_t keep_pair(uint32_t b2, uint32_t k2, uint32_t A0, uint32_t A1, const uint32_t *smem_table,
                                               const WeightTable &wt) {
    uint32_t e0 = 0, e1 = 0;
    if (kTable == 1) { e0 = smem_table[k2 & 0xffffu]; e1 = smem_table[k2 >> 16]; }
    if (kTable == 2) { e0 = __ldg(wt.thr + (k2 & 0xffffu)); e1 = __ldg(wt.thr + (k2 >> 16)); }
    if (kPacked) {
        // keep <=> A >= B + thr - (B < bound)
        uint32_t thr2;
        if (kTable == 0) {
            thr2 = __vadd2(k2, 0x00010001u);
        } else {
            thr2 = __byte_perm(e0, e1, 0x5410);
            bool ge_hi, ge_lo;
            (void)__vibmax_u16x2(b2, __byte_perm(e0, e1, 0x7632), &ge_hi, &ge_lo);  // B >= bound per half
            if (!ge_lo) thr2 -= 0x00000001u;  // thr >= 1 whenever bound > 0: no borrow
            if (!ge_hi) thr2 -= 0x00010000u;
        }
        bool hi, lo;
        (void)__vibmax_u16x2(A0 | (A1 << 16), __vadd2(b2, thr2), &hi, &lo);  // A >= B + thr per half
        return (lo ? 0x0000ffffu : 0u) | (hi ? 0xffff0000u : 0u);
    }
    if (kTable == 0) { e0 = (k2 & 0xffffu) + 1u; e1 = (k2 >> 16) + 1u; }
    const int b0 = (int)(b2 & 0xffffu), b1 = (int)(b2 >> 16);
    const int t0 = (int)(e0 & 0xffffu) - ((b0 < (int)(e0 >> 16)) ? 1 : 0);
    const int t1 = (int)(e1 & 0xffffu) - ((b1 < (int)(e1 >> 16)) ? 1 : 0);
    return (((int)A0 - b0 >= t0) ? 0x0000ffffu : 0u) | (((int)A1 - b1 >= t1) ? 0xffff0000u : 0u);
}

// One owned quad: [update] then [frame].  Returns the quad's max F (kNoQuad without a frame); nb_out = B'.
template <bool kUpdate, bool kFrame, bool kPacked, int kTable, bool kStats>
__device__ __forceinline__ int sweep_quad(Smem &s, const WeightTable &wt, const SweepThread &th, const SweepMode &m, int p4,
                                          uint2 pw, uint2 ow, float *fcur, uint8_t *lab_frame, SweepAcc &acc, uint2 &nb_out) {
    const uint2 bw = *reinterpret_cast<const uint2 *>(s.B + p4);
    const uint4 sv = *reinterpret_cast<const uint4 *>(s.S + p4);
    uint2 nb = bw;
    if (kUpdate) {
        const uint2 kw = *reinterpret_cast<const uint2 *>(s.K + p4);
        uint32_t A0, A1, A2, A3;
        if (!kPacked && m.first_mean) { A0 = sv.x; A1 = sv.y; A2 = sv.z; A3 = sv.w; }
        else { A0 = __umulhi(sv.x, m.magic); A1 = __umulhi(sv.y, m.magic); A2 = __umulhi(sv.z, m.magic); A3 = __umulhi(sv.w, m.magic); }
        const uint32_t keep_x = keep_pair<kPacked, kTable>(bw.x, kw.x, A0, A1, s.wthr, wt);
        const uint32_t keep_y = keep_pair<kPacked, kTable>(bw.y, kw.y, A2, A3, s.wthr, wt);
        nb.x = __byte_perm((bw.x & keep_x) | ((A0 | (A1 << 16)) & ~keep_x), 0, th.perm_x);
        nb.y = __byte_perm((bw.y & keep_y) | ((A2 | (A3 << 16)) & ~keep_y), 0, th.perm_y);
        uint2 nk;
        nk.x = __vadd2(kw.x, 0x00010001u) & keep_x;
        nk.y = __vadd2(kw.y, 0x00010001u) & keep_y;
        // a border column always equals its neighbour, before and after: it cannot change `changed`; the dp2a
        // selectors leave it out of the sum
        acc.changed |= (nb.x ^ bw.x) | (nb.y ^ bw.y);
        acc.bsum = (uint32_t)dp2a_us(nb.x, th.sel_x, dp2a_us(nb.y, th.sel_y, (int)acc.bsum));
        *reinterpret_cast<uint2 *>(s.B + p4) = nb;
        *reinterpret_cast<uint2 *>(s.K + p4) = nk;
    }
    acc.bmax2 = __vmaxu2(acc.bmax2, __vmaxu2(nb.x, nb.y));
    nb_out = nb;
    return kFrame ? filter_quad(pw, ow, p4, nb, sv, s.S, fcur, lab_frame, kStats, acc) : kNoQuad;
}

// The quad's pixels of this frame and of the frame leaving the 45-frame window (a frame of zeros while the window
// is still filling, so the load is unconditional).
template <bool kFrame>
__device__ __forceinline__ void load_quad(int p4, const uint16_t *P, const uint16_t *Pold, uint2 &pw, uint2 &ow) {
    pw = make_uint2(0, 0);
    ow = make_uint2(0, 0);
    if (!kFrame) return;
    pw = ldg8(P + p4);
    ow = ldg8(Pold + p4);
}

// Which quads a sweep thread processes: iteration `it` covers owned row r0 + it * rows_per_it, except that the last
// iteration's quad may have been remapped and the first one handed away (SweepThread::p4_last / has_last / skip0).
template <bool kLepton>
__device__ __forceinline__ bool sweep_mine(const SweepThread &th, int it, int rows_per_it, int owned_rows) {
    if (it == kQIter - 1) return th.has_last;
    if (it == 0) return th.active && !th.skip0 && (kLepton || th.r0 < owned_rows);
    return th.active && (kLepton || th.r0 + it * rows_per_it < owned_rows);  // 160x120: iterations 1 .. kQIter - 2 are full
}
__device__ __forceinline__ int sweep_p4(const SweepThread &th, int it, int stride) {
    return it == kQIter - 1 ? th.p4_last : th.p4_0 + it * stride;
}

// kUnrolled: straight-line code with the per-quad maxima in registers (the steady state); otherwise a rolled
// loop whose maxima go through local memory (first frame, tail pass, exact keep test: once per clip).
// kLepton: the geometry is 160x120 with a 1-pixel border (20 rows x 40 quads per iteration), so every offset of the
// straight-line code is an immediate.
template <bool kUpdate, bool kFrame, bool kPacked, int kTable, bool kStats, bool kUnrolled, bool kLepton>
__device__ __forceinline__ void pixel_sweep(const KernelArgs &a, Smem &s, const WeightTable &wt, const SweepThread &th,
                                            const SweepMode &m, const uint16_t *P, const uint16_t *Pold, float *fcur,
                                            uint8_t *lab_frame, SweepAcc &acc, int (&gmaxq)[kQIter]) {
    const Geometry &g = a.g;
    const int owned_rows = kLepton ? 118 : g.H - 2 * g.edge;
    constexpr int kLeptonRows = kPThreads / 40;  // rows per iteration at 160 pixels
    static_assert((118 - kLeptonRows) / kLeptonRows + 1 >= kQIter - 1, "160x120: only the last iteration is partial");
    const int rows_per_it = kLepton ? kLeptonRows : g.rows_per_it;
    const int stride = kLepton ? kLeptonRows * 160 : th.stride;
    uint2 nb_top = make_uint2(0, 0), nb_bottom = make_uint2(0, 0);
    if (kUnrolled) {
        // software pipeline: the global loads of quad it + 1 are in flight while quad it is processed
        // (two quads ahead, or the next frame's first quad across the message, cost registers the 80-register budget of
        // 21 warps does not have: measured slower)
        uint2 pw_next, ow_next;
        if (sweep_mine<kLepton>(th, 0, rows_per_it, owned_rows)) load_quad<kFrame>(th.p4_0, P, Pold, pw_next, ow_next);
#pragma unroll
        for (int it = 0; it < kQIter; ++it) {
            gmaxq[it] = kNoQuad;
            const bool mine = sweep_mine<kLepton>(th, it, rows_per_it, owned_rows);
            const uint2 pw = pw_next, ow = ow_next;
            if (it + 1 < kQIter && sweep_mine<kLepton>(th, it + 1, rows_per_it, owned_rows))
                load_quad<kFrame>(sweep_p4(th, it + 1, stride), P, Pold, pw_next, ow_next);
            if (!mine) continue;
            uint2 nb;
            gmaxq[it] = sweep_quad<kUpdate, kFrame, kPacked, kTable, kStats>(s, wt, th, m, sweep_p4(th, it, stride), pw, ow, fcur,
                                                                              lab_frame, acc, nb);
            if (it == 0) nb_top = nb;
            if (it == th.last_it) nb_bottom = nb;
        }
    } else {
#pragma unroll
        for (int j = 0; j < kQIter; ++j) gmaxq[j] = kNoQuad;
#pragma unroll 1
        for (int it = 0; it < kQIter; ++it) {
            const bool mine_it = sweep_mine<false>(th, it, rows_per_it, owned_rows);
            uint2 nb, pw, ow;
            if (!mine_it) continue;
            load_quad<kFrame>(sweep_p4(th, it, stride), P, Pold, pw, ow);
            const int hi = sweep_quad<kUpdate, kFrame, kPacked, kTable, kStats>(s, wt, th, m, sweep_p4(th, it, stride), pw, ow, fcur,
                                                                                lab_frame, acc, nb);
            // (selects, not an indexed store: the maxima stay in registers in every instantiation)
#pragma unroll
            for (int j = 0; j < kQIter; ++j)
                if (j == it) gmaxq[j] = hi;
            if (it == 0) nb_top = nb;
            if (it == th.last_it) nb_bottom = nb;
        }
    }
    // A border row takes the adjacent owned row's background (edge replication); run by that row's owner thread.
    // One rolled body for both rows: two rows of the frame do not deserve straight-line copies.
    if (g.edge && th.active && (th.r0 == 0 || th.last_it >= 0)) {
#pragma unroll 1
        for (int side = 0; side < 2; ++side) {
            if (side == 0 ? (th.r0 != 0) : (th.last_it < 0)) continue;
            const int pb = side == 0 ? th.p4_0 - g.W : th.p4_0 + th.last_it * stride + g.W;
            const uint2 nb = side == 0 ? nb_top : nb_bottom;
            if (kUpdate) *reinterpret_cast<uint2 *>(s.B + pb) = nb;
            if (kFrame) {
                // (a border pixel's background is a copy of its neighbour's: its sliding sum is never used)
                const uint2 pw = ldg8(P + pb);
                const int hi = filter_quad<false>(pw, make_uint2(0, 0), pb, nb, make_uint4(0, 0, 0, 0), s.S, fcur, lab_frame, kStats, acc);
                const int slot = side == 0 ? 0 : th.last_it;
#pragma unroll
                for (int it = 0; it < kQIter; ++it)
                    if (it == slot) gmaxq[it] = max(gmaxq[it], hi);
            }
        }
    }
}

// Runtime mode -> instantiation.
template <bool kStats>
__device__ __forceinline__ void pixel_sweep_dispatch(const KernelArgs &a, Smem &s, const WeightTable &wt, const SweepThread &th,
                                                     const SweepMode &m, const uint16_t *P, const uint16_t *Pold, float *fcur,
                                                     uint8_t *lab_frame, SweepAcc &acc, int (&gmaxq)[kQIter]) {
    const bool steady = m.update && m.frame && !m.slow && !m.first_mean && a.g.W == 160 && a.g.H == 120 && a.g.edge == 1;
    constexpr bool kUnroll = true;
    if (steady && m.table == 0)
        pixel_sweep<true, true, true, 0, kStats, kUnroll, true>(a, s, wt, th, m, P, Pold, fcur, lab_frame, acc, gmaxq);
    else if (steady && m.table == 1)
        pixel_sweep<true, true, true, 1, kStats, kUnroll, true>(a, s, wt, th, m, P, Pold, fcur, lab_frame, acc, gmaxq);
    else if (!m.update)
        pixel_sweep<false, true, false, 2, kStats, false, false>(a, s, wt, th, m, P, Pold, fcur, lab_frame, acc, gmaxq);
    else if (m.frame)
        pixel_sweep<true, true, false, 2, kStats, false, false>(a, s, wt, th, m, P, Pold, fcur, lab_frame, acc, gmaxq);
    else
        pixel_sweep<true, false, false, 2, kStats, false, false>(a, s, wt, th, m, P, Pold, fcur, lab_frame, acc, gmaxq);
}

// a frame's sums / extrema, folded by the sweep warps (one shared-memory atomic per value and warp)
__device__ __forceinline__ void frame_msg_reset(FrameMsg &fm) {
    uint32_t *r = fm.red;
    r[0] = 0; r[1] = (uint32_t)INT32_MAX; r[2] = (uint32_t)INT32_MIN; r[3] = (uint32_t)INT32_MAX; r[4] = (uint32_t)INT32_MIN;
    r[5] = 0; r[6] = 0; r[7] = 0; r[8] = 0xffffffffu; r[9] = 0;
}

__device__ __forceinline__ uint32_t sweep_reduce_store(FrameMsg &fm, int lane, const SweepAcc &acc, bool want_stats) {
    const uint32_t psum = __reduce_add_sync(0xffffffffu, acc.psum), bsum = __reduce_add_sync(0xffffffffu, acc.bsum);
    const uint32_t changed = __reduce_or_sync(0xffffffffu, acc.changed);
    const int fmin = __reduce_min_sync(0xffffffffu, acc.fmin), fmax = __reduce_max_sync(0xffffffffu, acc.fmax);
    const uint32_t bmax = __reduce_max_sync(0xffffffffu, max(acc.bmax2 & 0xffffu, acc.bmax2 >> 16));
    uint32_t *r = fm.red;
    if (lane == 0) atomicAdd(r + 0, psum);
    if (lane == 1) atomicMin(reinterpret_cast<int *>(r + 1), fmin);
    if (lane == 2) atomicMax(reinterpret_cast<int *>(r + 2), fmax);
    if (lane == 6) atomicAdd(r + 6, bsum);
    if (lane == 7 && changed) atomicOr(r + 7, changed);
    if (want_stats) {
        const int pmin = __reduce_min_sync(0xffffffffu, acc.pmin), pmax = __reduce_max_sync(0xffffffffu, acc.pmax);
        const uint32_t fabs_sum = __reduce_add_sync(0xffffffffu, acc.fabs_sum);
        if (lane == 3) atomicMin(reinterpret_cast<int *>(r + 3), pmin);
        if (lane == 4) atomicMax(reinterpret_cast<int *>(r + 4), pmax);
        if (lane == 5) atomicAdd(r + 5, fabs_sum);
    }
    return bmax;
}

// ================================================================================================
// sweep warps: the recurrence.  Per frame: fused sweep -> fold the frame's sums into the message of the mask
// warps -> hot-quad ballots against a PREDICTED bound (the mask warps compute the true one; if the prediction
// turns out too high they fall back to dense work, so the ballots are always a superset) -> next frame.
// ================================================================================================
__device__ void sweep_warps(const KernelArgs &a, Smem &s, const cpt_clip &clip, int ptid, float *scratch,
                            uint8_t *st_raw) {
    constexpr int kAll = kThreads;
    const Geometry &g = a.g;
    const int lane = ptid & 31, warp = ptid >> 5;
    const int W = g.W, npx = g.npx;
    const WeightTable wt = a.tables[clip.weight_table & 3];
    StateHeader *st_hdr = reinterpret_cast<StateHeader *>(st_raw);
    uint16_t *st_B = reinterpret_cast<uint16_t *>(st_raw + sizeof(StateHeader));
    uint16_t *st_K = st_B + npx;
    uint32_t *st_S = reinterpret_cast<uint32_t *>(st_K + npx);
    float *st_F = reinterpret_cast<float *>(st_S + npx);
    const bool want_stats = clip.flags & CPT_CLIP_FRAME_STATS;
    const bool update_bg = clip.flags & CPT_CLIP_UPDATE_BACKGROUND;
    const bool skip_first_update = clip.flags & CPT_CLIP_SKIP_FIRST_UPDATE;
    int frames_seen = 0;

    // ---------------------------------------------------------------- init / resume
    for (int i = ptid; i < 2 * kMaxWords; i += kPThreads) (&s.M[0][0])[i] = 0;
    for (int i = ptid; i < kSmemWeights; i += kPThreads) s.wthr[i] = (i <= wt.max_count) ? __ldg(wt.thr + i) : 0xffffu;  // beyond the table: never keep
    if (ptid < 2) frame_msg_reset(s.fm[ptid]);
    if (ptid == 0) {
        s.fth_latest = INT32_MIN;
        s.bcast_i[10] = 0;
    }
    if (clip.flags & CPT_CLIP_RESUME) {
        bar_sync(BAR_P, kPThreads);
        int kmax = 0;
        for (int i = ptid; i < npx; i += kPThreads) {
            const uint16_t k = st_K[i];
            s.B[i] = st_B[i];
            s.K[i] = k;
            s.S[i] = st_S[i];
            kmax = max(kmax, (int)k);
        }
        kmax = __reduce_max_sync(0xffffffffu, kmax);
        if (lane == 0) atomicMax(&s.bcast_i[10], kmax);
        if (ptid == 0) s.init_average = st_hdr->average;
        bar_sync(BAR_P, kPThreads);
        // the number of updates applied so far bounds every weight counter; the record may also have been
        // advanced by the stand-alone background kernels, so trust the counters themselves as well
        frames_seen = max(st_hdr->frames_seen, s.bcast_i[10]);
    } else {
        // WeightedBackground first call: motiondetector.py:199-212
        const uint16_t *init = a.frames + (size_t)clip.init_offset * npx;
        uint32_t csum = 0;
        for (int i = ptid; i < npx; i += kPThreads) {
            int y = i / W, x = i - y * W;
            uint16_t v = __ldg(init + i);
            s.B[i] = v;
            s.K[i] = 0;
            s.S[i] = 0;
            if (x >= g.edge && x < W - g.edge && y >= g.edge && y < g.H - g.edge) csum += v;
        }
        csum = __reduce_add_sync(0xffffffffu, csum);
        if (lane == 0) s.red_u[warp] = csum;
        bar_sync(BAR_P, kPThreads);
        if (warp == 0) {
            uint32_t v = (lane < kPWarps) ? s.red_u[lane] : 0u;
            v = __reduce_add_sync(0xffffffffu, v);
            if (lane == 0) s.init_average = (double)v / (double)g.ncrop;  // unrounded (np.average) until the background first changes
        }
        replicate_edges(s, g, ptid);
        bar_sync(BAR_P, kPThreads);
    }
    SweepThread th;
    {
        const int r0 = ptid / g.qpr, qx = ptid - r0 * g.qpr;
        th.r0 = r0;
        th.active = r0 < g.rows_per_it;
        th.p4_0 = (r0 + g.edge) * W + qx * 4;
        th.stride = g.rows_per_it * W;
        th.prefetch = (qx & 15) == 0;
        th.first_col = g.edge && qx == 0;
        th.last_col = g.edge && qx == g.qpr - 1;
        th.perm_x = th.first_col ? 0x3232u : 0x3210u;
        th.perm_y = th.last_col ? 0x1010u : 0x3210u;
        th.sel_x = th.first_col ? kHiP : kBoth;
        th.sel_y = th.last_col ? kLoP : kBoth;
        const int last_row = g.H - 2 * g.edge - 1;  // owned-row index
        th.last_it = (th.active && last_row % g.rows_per_it == r0) ? last_row / g.rows_per_it : -1;
        th.has_last = th.active && r0 + (kQIter - 1) * g.rows_per_it <= last_row;
        th.p4_last = th.p4_0 + (kQIter - 1) * th.stride;
        th.skip0 = false;
        th.lane = lane;
        if (g.balanced) {
            // 160x120: 118 owned rows + 2 border rows.  The owners of the first and last owned row also produce a border
            // row, so each hands one of its rows to a group whose last iteration is free: no thread has more than 8
            // quads per frame (owned_row_slot() is the inverse map).
            if (r0 == 0) th.has_last = false;
            if (r0 == g.bal_a_r) { th.has_last = true; th.p4_last = (g.bal_a_oy + g.edge) * W + qx * 4; }
            if (r0 == g.bal_b_oy) th.skip0 = true;  // (the last owned row's group index equals its first row's index)
            if (r0 == g.bal_b_r) {
                th.has_last = true;
                th.p4_last = (g.bal_b_oy + g.edge) * W + qx * 4;
            }
        }
    }
    bar_sync(BAR_INIT, kAll);  // the state and the initial average are in place: the other roles may start

    uint32_t magic_cnt = 0, magic_val = 0;
    bool slow = true;  // the first update of a launch takes the exact path (no background extrema yet)
    // t == n_frames is the tail pass: only the background update of the last frame
    for (int t = 0; t <= clip.n_frames; ++t) {
        CPT_TICK_START(ptid == 0);
        const bool is_frame = t < clip.n_frames;
        const int t_abs = clip.first_frame + t;
        const int b = t & 1;
        const size_t o = (size_t)(clip.out_offset + t);
        SweepMode m;
        // (rawdb.py:84-122: no update follows the frame that initialised the background when it is also the first kept frame)
        m.update = update_bg && t > 0 && !(skip_first_update && t_abs == 1);
        m.frame = is_frame;
        if (!m.update && !m.frame) break;
        {
            // the update belongs to frame t-1: the mean covers min(t_abs, 45) frames
            const uint32_t cnt = (uint32_t)min(max(t_abs, 1), kMeanFrames);
            m.first_mean = (cnt == 1u);
            // floor(S / cnt) == umulhi(S, magic): exact for S < 2^22, cnt <= 45 (the count saturates: one division per clip then)
            if (cnt != magic_cnt) {
                magic_cnt = cnt;
                magic_val = (cnt == 1u) ? 0u : 0xffffffffu / cnt + 1u;
            }
            m.magic = magic_val;
            m.slow = slow;
            const int k_cap = frames_seen;  // no weight counter can exceed the number of updates so far
            m.table = (k_cap < wt.linear_upto) ? 0 : ((k_cap < kSmemWeights) ? 1 : 2);
        }
        const uint16_t *P = is_frame ? frame_ptr(a, clip, t) : nullptr;
        const bool window_full = t_abs >= kMeanFrames;
        const uint16_t *Pold = (is_frame && window_full) ? frame_ptr(a, clip, t - kMeanFrames) : a.zero_frame;
        // linear clips: pull the next frame (and the next frame leaving the window) towards L2 with two bulk prefetches
        if (ptid == 0 && is_frame && t + 1 < clip.n_frames && clip.ring_frames == 0) {
            const uint32_t bytes = (uint32_t)npx * 2u;
            asm volatile("cp.async.bulk.prefetch.L2.global.L2::cache_hint [%0], %1, %2;" ::"l"(P + npx), "r"(bytes), "l"(l2_policy_keep()) : "memory");
            if (t_abs + 1 >= kMeanFrames)
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(frame_ptr(a, clip, t + 1 - kMeanFrames)), "r"(bytes) : "memory");
        }
        float *fcur = is_frame ? filtered_ptr(a, clip, scratch, t) : nullptr;
        uint8_t *lab_frame = (is_frame && a.labels) ? a.labels + o * npx : nullptr;

        // ------------------------------------------------------------ fused sweep (K7 of frame t-1, K1/K8 of frame t)
        SweepAcc acc;
        int gmaxq[kQIter];
        if (want_stats) pixel_sweep_dispatch<true>(a, s, wt, th, m, P, Pold, fcur, lab_frame, acc, gmaxq);
        else pixel_sweep_dispatch<false>(a, s, wt, th, m, P, Pold, fcur, lab_frame, acc, gmaxq);
        CPT_TICK(ptid == 0, 14);  // sweep
        // ------------------------------------------------------------ message to the mask warps / the scalar warp
        if (t >= 2) bar_sync(BAR_SM_EMPTY + b, kPThreads + kMThreads);  // they are done with the message of frame t-2
        if (t >= 1 && is_frame) bar_sync(BAR_QFREE, kPThreads + kMThreads);  // ... and with the quad maxima of frame t-1
        CPT_TICK(ptid == 0, 6);   // wait for the message buffer
        FrameMsg &fm = s.fm[b];
        const uint32_t warp_bmax = sweep_reduce_store(fm, lane, acc, want_stats);
        // quad maxima relative to the last bound the mask warps computed (any reference is exact, see mask_warps)
        const int latest = *(volatile int32_t *)&s.fth_latest;
        const int qref = (latest == INT32_MIN) ? 0 : latest;
        if (ptid == 0) {
            fm.qref = qref;
            fm.update = m.update;
            fm.is_frame = is_frame;
        }
        {
            // mode of this warp's NEXT update: the packed keep test needs B + thr < 2^16 for the pixels it owns
            const int k_next = min(frames_seen + 1, wt.max_count);
            const uint32_t thr_cap = (k_next < wt.linear_upto) ? (uint32_t)k_next + 1u
                                     : ((k_next < kSmemWeights ? s.wthr[k_next] : __ldg(wt.thr + k_next)) & 0xffffu);
            slow = warp_bmax + thr_cap > 65535u;
        }
        if (is_frame) {
            // a border row's quads count for the owned row next to them, which only widens the marks;
            // unowned slots hold kNoQuad -> -128
#pragma unroll
            for (int it = 0; it < kQIter; ++it) s.qmax8[it * kPThreads + ptid] = quad_byte(gmaxq[it], qref);
        }
        if (m.update) ++frames_seen;
        bar_arrive(BAR_SM_FULL + b, kPThreads + kMThreads);
        CPT_TICK(ptid == 0, 2);   // message
    }

    // ---------------------------------------------------------------- save state
    // (the other roles read the resumed state's filtered frame and header until their last frame is done)
    bar_sync(BAR_DONE, kAll);
    if (st_raw) {
        for (int i = ptid; i < npx; i += kPThreads) {
            st_B[i] = s.B[i];
            st_K[i] = s.K[i];
            st_S[i] = s.S[i];
        }
        if (clip.n_frames > 0) {
            const float *flast = filtered_ptr(a, clip, scratch, clip.n_frames - 1);
            for (int i = ptid; i < npx; i += kPThreads) st_F[i] = flast[i];
        }
        if (ptid == 0) {
            st_hdr->average = s.final_average;
            st_hdr->frames_seen = frames_seen;
            st_hdr->initialised = 1;
            st_hdr->prev_fmin = s.final_prev[0];
            st_hdr->prev_fmax = s.final_prev[1];
            st_hdr->have_prev = s.final_prev[2];
        }
    }
}

// K2 / K7 scalars of one frame from the sweep's message (one thread): WeightedBackground.average, the frame's scalars
// (frame_scalars_of) and the byte threshold for the stored quad maxima.  Writes the frame's info record and
// s.bcast_i[0..5, 8, 13, 14].
__device__ __forceinline__ void frame_scalars(const KernelArgs &a, Smem &s, const cpt_clip &clip, FrameMsg &fm, size_t o,
                                              bool is_frame, bool want_stats, double &average) {
    const Geometry &g = a.g;
    const uint32_t v0 = fm.red[0];
    const int v1 = (int)fm.red[1], v2 = (int)fm.red[2];
    if (fm.update && fm.red[7]) average = rounded_background_average(fm.red[6], (uint32_t)g.ncrop);  // the background changed
    if (is_frame) {
        const FrameScalars fs = frame_scalars_of(v0, v1, v2, average, clip.background_thresh, g.npx);
        s.bcast_i[0] = fs.ac; s.bcast_i[1] = fs.gmn; s.bcast_i[2] = fs.gmx;
        s.bcast_i[3] = v1; s.bcast_i[4] = v2;
        s.bcast_i[5] = __float_as_int(fs.thr);
        s.bcast_i[13] = (int)fs.nmagic; s.bcast_i[14] = fs.nshift;
        // byte threshold for the quad maxima the sweep stored relative to qref (0: no usable bound, dense work):
        // stored v = clamp(max F - qref, -128, 127) + 128, hot <=> v >= clamp(fth - qref, -127, 127) + 128.
        // v == 0 means max F <= qref - 128 < fth; v == 255 means max F >= qref + 127 >= fth unless the
        // threshold was clamped from above, which only widens the marks.
        {
            int tu = 0;
            if (fs.fth != INT32_MIN) {
                const long long dq = (long long)fs.fth - (long long)fm.qref;
                if (dq >= -127) tu = (int)min(dq, 127ll) + 128;
            }
            s.bcast_i[8] = tu;
        }
        if (fs.fth != INT32_MIN) *(volatile int32_t *)&s.fth_latest = fs.fth;
        a.info[o] = frame_info_of(fs, average, v0, v1, v2, want_stats, (int)fm.red[3], (int)fm.red[4], fm.red[5], 0);
    }
    frame_msg_reset(fm);
}

// ================================================================================================
// mask warps: one frame behind the sweep.  Scalars (K2) from the sweep's message, hot quads -> per-row marks ->
// work lists, normalise (K2) and blur + threshold (K4) of the listed groups -> bit rows for the component warps.
// ================================================================================================
__device__ void mask_warps(const KernelArgs &a, Smem &s, const cpt_clip &clip, int mtid, float *scratch,
                           const StateHeader *st_hdr) {
    const Geometry &g = a.g;
    const int npx = g.npx;
    const bool want_stats = clip.flags & CPT_CLIP_FRAME_STATS;
    const bool update_bg = clip.flags & CPT_CLIP_UPDATE_BACKGROUND;
    const bool denoise = clip.flags & CPT_CLIP_DENOISE;
    bar_sync(BAR_INIT, kThreads);
    double average = s.init_average;  // WeightedBackground.average: only thread 0 of the role uses it
    int prev_fmin = 0, prev_fmax = 0, have_prev = 0;
    if (clip.flags & CPT_CLIP_RESUME) {
        prev_fmin = st_hdr->prev_fmin;
        prev_fmax = st_hdr->prev_fmax;
        have_prev = st_hdr->have_prev;
    }
    // frame-at-a-time denoise: the caller has put the previous frame's outputs at out_offset - 1
    const bool prev_in_output = have_prev && (clip.flags & CPT_CLIP_PREV_IN_OUTPUT);
    for (int t = 0; t <= clip.n_frames; ++t) {
        CPT_TICK_START2(mtid == 0);
        const bool is_frame = t < clip.n_frames;
        if (!(update_bg && t > 0 && !((clip.flags & CPT_CLIP_SKIP_FIRST_UPDATE) && clip.first_frame + t == 1)) && !is_frame) break;
        const int b = t & 1;
        const size_t o = (size_t)(clip.out_offset + t);
        bar_sync(BAR_SM_FULL + b, kPThreads + kMThreads);  // the sweep of frame t is done
        CPT_TICK2(mtid == 0, 7);   // waiting for the sweep
        FrameMsg &fm = s.fm[b];
        // ------------------------------------------------------------ scalars (K2, K7 average)
        if (mtid == 0) frame_scalars(a, s, clip, fm, o, is_frame, want_stats, average);
        CPT_TICK2(mtid == 0, 16);  // scalars: thread 0
        bar_sync(BAR_M, kMThreads);
        CPT_TICK2(mtid == 0, 3);   // scalars + barrier
        if (!is_frame) break;  // tail pass: only the average
        const int ac = s.bcast_i[0], gmn = s.bcast_i[1], gmx = s.bcast_i[2];
        const int cur_fmin = s.bcast_i[3], cur_fmax = s.bcast_i[4];
        const float thr = __int_as_float(s.bcast_i[5]);
        const int tu = s.bcast_i[8];
        const uint32_t nmagic = (uint32_t)s.bcast_i[13];
        const int nshift = s.bcast_i[14];
        const int ith = (int)floorf(thr);
        const float *fcur = filtered_ptr(a, clip, scratch, t);
        // the sweep warps reuse this frame's message buffer two iterations from now, if there is one
        const bool sweep_comes_back = (t + 2 < clip.n_frames) || (t + 2 == clip.n_frames && update_bg);
        prev_fmin = cur_fmin;
        prev_fmax = cur_fmax;
        have_prev = 1;
        if (denoise) {
            // K3 sits between K2 and K4: emit the whole normalised image; cv2.fastNlMeansDenoising, blur, threshold,
            // close and components run as separate wide passes over all frames (nlm_quads_kernel, mask_components_kernel)
            uint8_t *u_frame = a.u8_frames + o * npx;
            for (int grp = mtid; grp < g.groups; grp += kMThreads) normalise_group(s, fcur, grp, ac, gmn, gmx, nmagic, nshift, u_frame);
            if (mtid == 0) a.info[o].reserved[1] = (t > 0 || prev_in_output) ? 2 : 1;  // 2: the previous filtered image is frame o - 1
            if (sweep_comes_back) bar_arrive(BAR_SM_EMPTY + b, kPThreads + kMThreads);
            if (t + 1 < clip.n_frames) bar_arrive(BAR_QFREE, kPThreads + kMThreads);
            continue;
        }

        // ------------------------------------------------------------ hot quads -> per-row marks -> work lists
        // Blur weights sum to 256, so an output can fire only within rows +-2 / neighbouring quads of a hot quad, and
        // reads U within rows +-4 / quads +-2.
        const bool no_fg = ith >= 255;  // nothing can exceed the threshold: the mask stays empty
        bool dense = tu == 0;           // no usable bound: every group is normalised and blurred
        int n_u = 0, n_b = 0;
        const int owned = g.H - 2 * g.edge;
        if (!no_fg && !dense) {
            // one thread per owned row: its quads' maxima -> one bit per quad
            for (int oy = mtid; oy < owned; oy += kMThreads) {
                int hit, hr;
                owned_row_slot(g, oy, hit, hr);
                const int pos = hit * kPThreads + hr * g.qpr;
                unsigned long long bits = 0;
                if (((pos | g.qpr) & 3) == 0) {
                    const uint32_t *q4 = reinterpret_cast<const uint32_t *>(s.qmax8 + pos);
                    const uint32_t t4 = (uint32_t)tu * 0x01010101u;
                    for (int w = 0; w < (g.qpr >> 2); ++w) {
                        const uint32_t ge = __vcmpgeu4(q4[w] ^ 0x80808080u, t4) & 0x01010101u;  // byte i -> bit 8 i
                        bits |= (unsigned long long)((ge * 0x10204080u) >> 28) << (4 * w);  // -> bits 0..3
                    }
                } else {
                    for (int q = 0; q < g.qpr; ++q) bits |= (unsigned long long)((int)s.qmax8[pos + q] >= tu - 128 ? 1u : 0u) << q;
                }
                s.hot64[oy] = bits;
            }
            if (mtid == 0) { s.bcast_i[11] = 0; s.bcast_i[12] = 0; }
            bar_sync(BAR_M, kMThreads);
        }
        CPT_TICK2(mtid == 0, 15);  // quad maxima -> hot rows
        if (t + 1 < clip.n_frames) bar_arrive(BAR_QFREE, kPThreads + kMThreads);  // the next sweep may store its maxima
        if (!no_fg && !dense) {
            // one thread per frame row: OR the hot rows around the row, widen by the neighbouring quads, and turn the
            // marks into list entries (groups of 8 pixels; a blur entry carries its two quad marks)
            const unsigned long long rowmask = (1ull << g.qpr) - 1ull;
            for (int rrow = mtid; rrow < g.H; rrow += kMThreads) {
                unsigned long long near_b = 0, near_u = 0;
#pragma unroll
                for (int dy = -4; dy <= 4; ++dy) {
                    const int yy = rrow - g.edge + dy;  // owned-row index
                    if (yy < 0 || yy >= owned) continue;
                    const unsigned long long h = s.hot64[yy];
                    near_u |= h;
                    if (dy >= -2 && dy <= 2) near_b |= h;
                }
                emit_norm_groups<true>(near_u, rowmask, rrow * g.gpr, &s.bcast_i[11], s.list_u);
                emit_blur_groups<true>(near_b, rowmask, rrow * g.gpr, &s.bcast_i[12], s.list_b);
            }
            bar_sync(BAR_M, kMThreads);
            n_u = s.bcast_i[11];
            n_b = s.bcast_i[12];
            // lists overflowed: dense work (every quad evaluated; a superset of the marks, so still exact)
            if (n_u > kListCap || n_b > kListCap) dense = true;
        }
        CPT_COUNT(mtid == 0, 28, n_u);
        CPT_COUNT(mtid == 0, 29, n_b);
        CPT_COUNT(mtid == 0 && dense, 30, 1);
        CPT_COUNT(mtid == 0 && no_fg, 31, 1);
        if (sweep_comes_back) bar_arrive(BAR_SM_EMPTY + b, kPThreads + kMThreads);  // message consumed
        CPT_TICK2(mtid == 0, 4);   // marks + lists
        // ------------------------------------------------------------ sweep 2b: U (K2), from the filtered image
        if (!no_fg) {
            if (dense) {
                for (int grp = mtid; grp < g.groups; grp += kMThreads) normalise_group(s, fcur, grp, ac, gmn, gmx, nmagic, nshift);
            } else {
                // all of a thread's loads are in flight before the first value is used (L2 latency paid once)
                constexpr int kBatch = 4;
                for (int i0 = mtid; i0 < n_u; i0 += kBatch * kMThreads) {
                    int grp[kBatch];
                    float4 f0[kBatch], f1[kBatch];
#pragma unroll
                    for (int j = 0; j < kBatch; ++j) {
                        const int i = i0 + j * kMThreads;
                        grp[j] = (i < n_u) ? (int)s.list_u[i] : -1;
                        if (grp[j] >= 0) {
                            f0[j] = *reinterpret_cast<const float4 *>(fcur + grp[j] * 8);
                            f1[j] = *reinterpret_cast<const float4 *>(fcur + grp[j] * 8 + 4);
                        }
                    }
#pragma unroll
                    for (int j = 0; j < kBatch; ++j)
                        if (grp[j] >= 0) normalise_values(s, f0[j], f1[j], grp[j], ac, gmn, gmx, nmagic, nshift);
                }
            }
            bar_sync(BAR_M, kMThreads);
        }
        CPT_TICK2(mtid == 0, 5);   // normalise + barrier

        // ------------------------------------------------------------ blur + threshold (K4) -> s.M[b]
        // (the component warps hand the buffer back zeroed)
        if (t >= 2) bar_sync(BAR_EMPTY + b, kMThreads + kCThreads);  // component warps are done with frame t-2's mask
        CPT_TICK2(mtid == 0, 8);   // wait for the mask buffer
        if (!no_fg) {
            if (dense) {
                for (int grp = mtid; grp < g.groups; grp += kMThreads) blur_group(s, g, grp, 3u, b, ith);
            } else {
                for (int i = mtid; i < n_b; i += kMThreads) {
                    const uint32_t e = s.list_b[i];
                    blur_group(s, g, (int)(e & 0x3fffu), e >> 14, b, ith);
                }
            }
        }
        if (mtid == 0) { s.msg[b][0] = cur_fmin; s.msg[b][1] = cur_fmax; }
        bar_arrive(BAR_FULL + b, kMThreads + kCThreads);
        CPT_TICK2(mtid == 0, 9);   // blur
    }
    if (mtid == 0) {
        s.final_average = average;
        s.final_prev[0] = prev_fmin; s.final_prev[1] = prev_fmax; s.final_prev[2] = have_prev;
    }
    bar_arrive(BAR_DONE, kThreads);
}

}  // namespace

__global__ void __launch_bounds__(kThreads, 1) extract_clips_kernel(const KernelArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem &s = *reinterpret_cast<Smem *>(smem_raw);
    const int tid = threadIdx.x;
    const int npx = a.g.npx;

    // clips are handed out dynamically so that ragged batches stay balanced
    while (true) {
        __syncthreads();
        if (tid == 0) s.bcast_i[15] = atomicAdd(a.work_counter, 1);
        __syncthreads();
        const int ci = s.bcast_i[15];
        if (ci >= a.n_clips) break;
        const cpt_clip clip = a.clips[ci];
        uint8_t *st_raw = a.state ? a.state + (size_t)ci * state_bytes(npx) : nullptr;
        float *scratch = a.scratch ? a.scratch + (size_t)blockIdx.x * 8 * npx : nullptr;
        const StateHeader *st_hdr = reinterpret_cast<const StateHeader *>(st_raw);
        if (tid < kPThreads) {
            sweep_warps(a, s, clip, tid, scratch, st_raw);
        } else if (tid < kPThreads + kMThreads) {
            mask_warps(a, s, clip, tid - kPThreads, scratch, st_hdr);
        } else {
            const float *st_F = reinterpret_cast<const float *>(st_raw + sizeof(StateHeader) + (size_t)npx * 8);
            component_warps(a, s, clip, tid - kPThreads - kMThreads, scratch, st_hdr, st_F);
        }
    }
}

// One row of quad bytes (strip_sweep_kernel) against its strip's byte threshold, any row length: bit q = quad q may hold a
// pixel that reaches the threshold.
__device__ __forceinline__ unsigned long long quad_row_bits_bytes(const Geometry &g, const int8_t *row, int th) {
    unsigned long long bits = 0;
    for (int q = 0; q < g.qpr; ++q) bits |= (unsigned long long)((int)row[q] >= th ? 1u : 0u) << q;
    return bits;
}

// ---- components of a small mask inside frame_regions_kernel's CTA ---------------------------------------------------------
// The passes of components_of_frame (close, runs, unions with the row above, statistics, OpenCV label order, label runs,
// region records), restricted to the rows [r0, r1] the mask stage can have set and sized for the masks real frames have:
// the tables are indexed by word of the extent, run ids are (row of the extent) * rpr + index with
// rpr = min(80, kLeanParents / rows), at most kLeanSlots components.
// Returns 0 when the frame is done; when it does not fit (a row with more runs, more components) -- found before anything is
// written to global memory -- the number of threads that are still there (threads 0 .. n - 1; the others got 0 and left):
// they store the mask for frame_components_kernel, which redoes the frame.  Called by all kFThreads threads.
__device__ int components_lean(const KernelArgs &a, MaskSmem &s, const Geometry &g, int tid, size_t o, int r0, int r1, bool have_prev) {
    const int rw = g.row_words;
    const int c0 = r0, c1 = min(r1 + 1, g.H - 1), nrows = c1 - c0 + 1, nw = nrows * rw;
    const int rpr = min(kRunsPerRow, kLeanParents / nrows);
    // ---- close; rows outside [c0, c1] are empty.  The non-empty words go on a list (any order): every later pass walks the
    // list, a few dozen words for the masks real frames have.
    // (s.ncomp, s.overflow and s.nwords were zeroed by the caller before its last barrier)
    const int lane = tid & 31;
    for (int lw0 = 0; lw0 < nw; lw0 += kFThreads) {
        const int lw = lw0 + tid;
        uint32_t c = 0u;
        if (lw < nw) {
            const int ry = (int)(((uint32_t)lw * g.rw_magic) >> 13);
            c = closed_word(s.M[0], lw + c0 * rw, c0 + ry, rw);
            s.C[lw] = c;
        }
        const uint32_t nz = __ballot_sync(0xffffffffu, c != 0u);
        if (nz) {
            int base = 0;
            if (lane == 0) base = atomicAdd(&s.nwords, __popc(nz));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (c != 0u) s.wlist[base + __popc(nz & ((1u << lane) - 1u))] = (uint16_t)lw;
        }
    }
    __syncthreads();
    const int nwl = s.nwords;
    if (nwl == 0) return 0;  // no foreground: info.n_components stays 0
    // (letting only as many warps as the list needs continue, with barriers over those, was measured slower: 10.15 ms
    // against 9.82 ms for the per-frame stage of the bench batch)
    constexpr int nact = kFThreads;
    auto sync_act = [&]() { __syncthreads(); };
    // ---- run starts and ids
    for (int i = tid; i < nwl; i += nact) {
        const int lw = s.wlist[i];
        const int ry = (int)(((uint32_t)lw * g.rw_magic) >> 13);
        int base;
        const int n = __popc(word_run_starts(s, lw, lw - ry * rw, s.C[lw], base));
        if (base + n > rpr) { s.overflow = 1; continue; }
        for (int k = 0; k < n; ++k) s.parent[ry * rpr + base + k] = (uint16_t)(ry * rpr + base + k);
    }
    sync_act();
    if (s.overflow) return nact;
    // ---- unions with the row above
    for (int i = tid; i < nwl; i += nact) {
        const int lw = s.wlist[i];
        const int ry = (int)(((uint32_t)lw * g.rw_magic) >> 13);
        if (ry > 0) unite_with_row_above(s, lw, lw - ry * rw, rw, s.C[lw], ry, rpr);  // (the row above the extent is empty)
    }
    sync_act();
    // ---- roots -> component slots
    for (int i = tid; i < nwl; i += nact) {
        const int lw = s.wlist[i];
        const int ry = (int)(((uint32_t)lw * g.rw_magic) >> 13);
        const int n = __popc(s.ST[lw]), id0 = ry * rpr + (int)s.base[lw];
        for (int k = 0; k < n; ++k) {
            const int id = id0 + k;
            if (s.parent[id] == id) {
                const int slot = min(atomicAdd(&s.ncomp, 1), kLeanSlots);
                reset_slot(s, slot);
                s.parent[id] = (uint16_t)(kSlotFlag | slot);
            }
        }
    }
    sync_act();
    const int ncomp = s.ncomp;
    if (ncomp > kLeanSlots) return nact;
    // ---- per-run statistics into the slot tables; the run's slot is left in its parent entry for the label pass
    for (int i = tid; i < nwl; i += nact) {
        const int lw = s.wlist[i];
        const uint32_t c = s.C[lw];
        const int ry = (int)(((uint32_t)lw * g.rw_magic) >> 13), wi = lw - ry * rw;
        uint32_t bitsleft = s.ST[lw];
        int id = ry * rpr + (int)s.base[lw];
        while (bitsleft) {
            const int b = __ffs(bitsleft) - 1;
            bitsleft &= bitsleft - 1;
            const int slot = uf_slot(s.parent, id);
            s.parent[id++] = (uint16_t)(kSlotFlag | slot);
            add_run(s, g, slot, wi * 32 + b, c0 + ry, run_length(s, lw, wi, rw, c, b));
        }
    }
    sync_act();
    const int nout = min(ncomp, g.max_regions);
    if (tid < ncomp) {
        const int rank = slot_rank(s, tid, ncomp);
        s.c_rank[tid] = (uint8_t)rank;
        if (rank < nout) a.regions[o * g.max_regions + rank] = region_record(s, tid);
    }
    if (tid == 0) {
        a.info[o].n_components = ncomp;
        if (have_prev) a.info[o].reserved[0] = 1;  // region_variance_kernel fills pixel_variance
    }
    if (!a.labels) return 0;
    sync_act();
    // ---- label image: the sweep already stored zeros for this frame; write the runs
    uint8_t *lab_frame = a.labels + o * g.npx;
    for (int i = tid; i < nwl; i += nact) {
        const int lw = s.wlist[i];
        const uint32_t c = s.C[lw];
        const int ry = (int)(((uint32_t)lw * g.rw_magic) >> 13), wi = lw - ry * rw;
        uint32_t bitsleft = s.ST[lw];
        int id = ry * rpr + (int)s.base[lw];
        while (bitsleft) {
            const int b = __ffs(bitsleft) - 1;
            bitsleft &= bitsleft - 1;
            const uint8_t lab = (uint8_t)(s.c_rank[s.parent[id++] & 0xff] + 1);
            store_label_run(lab_frame, g, wi * 32 + b, c0 + ry, run_length(s, lw, wi, rw, c, b), lab);
        }
    }
    return 0;
}

// i / d for small i (i * d < 2^32) with magic = 0xffffffff / d + 1 (which wraps to 0 for d == 1)
__device__ __forceinline__ int div_magic(int i, int d, uint32_t magic) { return d == 1 ? i : (int)__umulhi((uint32_t)i, magic); }

// Split path, second launch: one CTA of four warps per frame, the frame's mask as bit rows in global memory.
// A pixel can only reach the threshold near a hot quad (blur weights sum to 256: an output fires only within rows +-2 /
// one quad of a hot quad and reads normalised values within rows +-4 / two quads), and hot quads are rare:
//   quad bytes of the strips that may hold hot quads (FrameHdr::hot_strips) against their byte thresholds -> hot quads;
//   then one BAND of up to 32 hot rows at a time (nearly always the only one): the extent of its hot quads (rows, quad
//   columns) -> normalise (K2, exact integer form of the reference's fp32 multiply-then-divide) the extent grown by
//   4 rows / 2 quads -> blur + threshold (K4: 5x5 binomial in packed 16-bit lanes) the quads within 2 rows / 1 quad of a
//   hot quad of the band,
// with the band's normalised bytes in a 6.4 kB window of shared memory (no full-frame image, no work lists): small CTAs
// with little shared memory, so that many frames are resident per SM and hide each other's dependent loads.  Bands
// overlap by their halos; both compute the same bits there and OR them into the mask.
__global__ void __launch_bounds__(kFThreads, kFMinBlocks) frame_regions_kernel(const KernelArgs a, long long total_frames) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    MaskSmem &s = *reinterpret_cast<MaskSmem *>(smem_raw);
    const Geometry &g = a.g;
    const int tid = threadIdx.x, lane = tid & 31;
    const long long o = blockIdx.x;
    if (o >= total_frames) return;
    const FrameHdr *fh = a.fhdr + o;
    CPT_TICK_START2(tid == 0);
    // the frame's header: one 64-byte line, four vector loads in flight together
    const uint4 hdr = __ldg(reinterpret_cast<const uint4 *>(fh));  // nmagic, nshift, flags, hot_strips
    const uint4 th_lo = __ldg(reinterpret_cast<const uint4 *>(fh) + 1), th_hi = __ldg(reinterpret_cast<const uint4 *>(fh) + 2);
    const uint4 sc = __ldg(reinterpret_cast<const uint4 *>(fh) + 3);  // threshold, avg_change, norm_min, norm_max
    const float thr = __uint_as_float(sc.x);
    const int ac = (int)sc.y, gmn = (int)sc.z, gmx = (int)sc.w;
    const bool dn_marker = (hdr.z & kHdrDenoise) != 0;
    if (!(hdr.z & kHdrValid)) return;  // no clip produced this output frame
    const uint32_t nmagic = hdr.x;
    const int nshift = (int)hdr.y;
    const float *fcur = a.filtered + (size_t)o * g.npx;
    if (dn_marker) {
        // denoise clips: K3 sits between K2 and K4 -- emit the whole normalised image; cv2.fastNlMeansDenoising, blur,
        // threshold, close and components follow as wide passes (nlm_quads_kernel, mask_components_kernel)
        uint8_t *u_frame = a.u8_frames + (size_t)o * g.npx;
        for (int grp = tid; grp < g.groups; grp += kFThreads) normalise_group(s, fcur, grp, ac, gmn, gmx, nmagic, nshift, u_frame);
        return;
    }
    const int ith = (int)floorf(thr);
    const bool no_fg = ith >= 255;  // nothing can exceed the threshold: the mask stays empty
    const bool dense = (hdr.z & kHdrDense) != 0;  // no usable bound for the quad bytes: every quad counts as hot
    CPT_TICK2(tid == 0, 7);  // header + info
    // nothing can reach the threshold (no strip holds a hot quad): the mask is empty, info.n_components stays 0
    if (no_fg || (!dense && hdr.w == 0u)) return;
    const int8_t *qb = a.qbytes + (size_t)o * (g.H * g.qpr);
    const int wpr = g.qpr >> 2;  // words of quad bytes per row (rows of whole words: qpr % 4 == 0)
    const bool wordq = (g.qpr & 3) == 0;
    const unsigned long long rowmask = g.qpr >= 64 ? ~0ull : (1ull << g.qpr) - 1ull;
    const uint32_t wmagic = g.qw_magic;
    // ---- hot quads of the whole frame: the quad bytes of the hot strips, one warp per strip (strip s belongs to warp s & 3),
    // four words of four quads per lane (a strip has at most kStripPxMax / 16 = 120 words); the first strip's words are
    // requested before anything waits
    constexpr int kWarpsF = kFThreads / 32;
    static_assert(kWarpsF == 4, "strip s belongs to warp s & 3");
    static_assert(kStripPxMax / 16 <= 4 * 32, "four words of a strip's quad bytes per lane");
    const int warp = tid >> 5;
    uint32_t pre[4] = {0x80808080u, 0x80808080u, 0x80808080u, 0x80808080u};  // (-128: never hot)
    const uint32_t my_strips = (dense ? 0u : hdr.w) & (0x11111111u << warp);
    const int my_first = my_strips ? __ffs(my_strips) - 1 : -1;
    if (my_first >= 0 && wordq) {
        const int y0 = g.strip_y0[my_first], nw = ((int)g.strip_y0[my_first + 1] - y0) * wpr;
        const uint32_t *qw = reinterpret_cast<const uint32_t *>(qb + y0 * g.qpr);
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (4 * lane + j < nw) pre[j] = __ldg(qw + 4 * lane + j);
    }
    const bool vec = (g.words & 3) == 0;
    if (vec) {
        for (int i = tid; i < g.words / 4; i += kFThreads) reinterpret_cast<uint4 *>(s.M[0])[i] = make_uint4(0, 0, 0, 0);
    } else {
        for (int i = tid; i < g.words; i += kFThreads) s.M[0][i] = 0;
    }
    if (tid == 0) {
        reinterpret_cast<uint4 *>(s.theta)[0] = th_lo;
        reinterpret_cast<uint4 *>(s.theta)[1] = th_hi;
    }
    for (int r = tid; r < g.H; r += kFThreads) s.hot64[r] = dense ? rowmask : 0ull;
    __syncthreads();
    {
        uint32_t hs = my_strips;
        uint32_t *hot32 = reinterpret_cast<uint32_t *>(s.hot64);
        while (hs) {
            const int sidx = __ffs(hs) - 1;
            hs &= hs - 1;
            const int y0 = g.strip_y0[sidx], nrows = (int)g.strip_y0[sidx + 1] - y0;
            const int th = s.theta[sidx];
            if (!wordq) {
                for (int r = lane; r < nrows; r += 32) s.hot64[y0 + r] = quad_row_bits_bytes(g, qb + (y0 + r) * g.qpr, th);
                continue;
            }
            const int nw = nrows * wpr;
            const uint32_t t4 = (uint32_t)(th + 128) * 0x01010101u;
            const uint32_t *qw = reinterpret_cast<const uint32_t *>(qb + y0 * g.qpr);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int i = 4 * lane + j;
                uint32_t v = pre[j];
                if (sidx != my_first) v = i < nw ? __ldg(qw + i) : 0x80808080u;
                const uint32_t ge = __vcmpgeu4(v ^ 0x80808080u, t4) & 0x01010101u;  // byte i -> bit 8 i
                const uint32_t nib = (ge * 0x10204080u) >> 28;                      // -> bits 0..3
                if (nib) {
                    const int r = div_magic(i, wpr, wmagic), c = i - r * wpr;
                    atomicOr(hot32 + 2 * (y0 + r) + (c >> 3), nib << ((4 * c) & 31));
                }
            }
        }
    }
    __syncthreads();
    CPT_TICK2(tid == 0, 15);  // quad bytes -> hot rows
    // ---- the set of hot rows, kept by warp 0 (bit r & 31 of rb[r >> 5]): it cuts the bands and hands them to the CTA
    uint32_t rb[4] = {0u, 0u, 0u, 0u};
    if (warp == 0) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int r = 32 * j + lane;
            rb[j] = __ballot_sync(0xffffffffu, r < g.H && s.hot64[r] != 0ull);
        }
    }
    int m_r0 = g.H, m_r1 = -1;  // rows the mask can have set
    for (int bp = 0;; bp ^= 1) {  // (band parity)
        if (warp == 0) {
            // the band: kBandRows rows from the first hot row on, [lo, hi] = its first and last hot row
            int blo = 0, bhi = -1;
            if (rb[0] | rb[1] | rb[2] | rb[3]) {
                int w = 0;
                uint32_t cur = rb[0], nxt = rb[1];
                if (!cur) { w = 1; cur = rb[1]; nxt = rb[2]; }
                if (!cur) { w = 2; cur = rb[2]; nxt = rb[3]; }
                if (!cur) { w = 3; cur = rb[3]; nxt = 0u; }
                const int b = __ffs(cur) - 1;
                blo = 32 * w + b;
                constexpr uint32_t kWin = kBandRows >= 32 ? 0xffffffffu : (1u << kBandRows) - 1u;
                const uint32_t win = ((cur >> b) | (b ? (nxt << (32 - b)) : 0u)) & kWin;  // bit i: row lo + i is hot
                bhi = blo + 31 - __clz(win);
                const uint32_t m_cur = kWin << b, m_nxt = (b + kBandRows > 32) ? (1u << (b + kBandRows - 32)) - 1u : 0u;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (j == w) rb[j] &= ~m_cur;
                    if (j == w + 1) rb[j] &= ~m_nxt;
                }
            }
            if (lane == 0) {
                s.band[bp][0] = blo; s.band[bp][1] = bhi; s.count[bp][0] = 0; s.count[bp][1] = 0;
                s.ncomp = 0; s.overflow = 0; s.nwords = 0;  // (for the components stage)
            }
        }
        __syncthreads();  // the band record is there; the previous band is done with U and the lists, the mask has its bits
        const int lo = s.band[bp][0], hi = s.band[bp][1];
        if (hi < 0) break;
        const int ur0 = max(lo - kBandHalo, 0), ur1 = min(hi + kBandHalo, g.H - 1);
        const int br0 = max(lo - 2, 0), br1 = min(hi + 2, g.H - 1);
        m_r0 = min(m_r0, br0);
        m_r1 = max(m_r1, br1);
        // work lists, one thread per row: warps 0-1 the groups to normalise (rows +-4, quads +-2 around the band's hot
        // quads), warps 2-3 the groups to blur (rows +-2, one quad; an entry carries its two quad marks)
        if (tid < kFThreads / 2) {
            const int y = ur0 + tid;
            if (y <= ur1) {
                unsigned long long nearq = 0;
#pragma unroll
                for (int dy = -kBandHalo; dy <= kBandHalo; ++dy) {
                    const int rr = y + dy;
                    if (rr >= lo && rr <= hi) nearq |= s.hot64[rr];
                }
                emit_norm_groups<false>(nearq, rowmask, tid * g.gpr, &s.count[bp][0], s.list_u);  // (band row)
            }
        } else {
            const int y = br0 + tid - kFThreads / 2;
            if (y <= br1) {
                unsigned long long nearq = 0;
#pragma unroll
                for (int dy = -2; dy <= 2; ++dy) {
                    const int rr = y + dy;
                    if (rr >= lo && rr <= hi) nearq |= s.hot64[rr];
                }
                emit_blur_groups<false>(nearq, rowmask, y * g.gpr, &s.count[bp][1], s.list_b);  // (frame row)
            }
        }
        __syncthreads();
        CPT_TICK2(tid == 0, 4);  // marks + lists
        const int n_u = s.count[bp][0], n_b = s.count[bp][1];
        CPT_COUNT(tid == 0, 28, n_u);
        CPT_COUNT(tid == 0, 29, n_b);
        {
            const int grp0 = ur0 * g.gpr;
            for (int i = tid; i < n_u; i += kFThreads)
                normalise_group(s, fcur, grp0 + (int)s.list_u[i], ac, gmn, gmx, nmagic, nshift, nullptr, ur0 * g.W);
        }
        __syncthreads();
        CPT_TICK2(tid == 0, 5);  // normalise
        for (int i = tid; i < n_b; i += kFThreads) {
            const uint32_t e = s.list_b[i];
            blur_group(s, g, (int)(e & 0x3fffu), e >> 14, 0, ith, ur0, true);
        }
        CPT_TICK2(tid == 0, 8);  // blur + threshold
    }
    if (m_r1 < 0) return;  // the byte thresholds were only bounds: no hot quad after all, the mask is empty
    // (the mask is complete and the band's buffers are free: every thread has passed the barrier that follows the last blur)
    CPT_COUNT(tid == 0, 30, 1);  // frames that reach the components stage
    // ---- close, components, statistics, labels, region records (K4 second half, K5) in place; the variances are left to
    // region_variance_kernel
    const int left = components_lean(a, s, g, tid, (size_t)o, m_r0, m_r1, !(hdr.z & kHdrFirst));
    CPT_TICK2(tid == 0, 9);  // components
    if (left == 0) return;
    // a mask the in-place stage is not sized for: stored for frame_components_kernel
    uint32_t *mout = a.maskbits + (size_t)o * kMaxWords;
    if ((g.words & 3) == 0) {
        for (int i = tid; i < g.words / 4; i += left) reinterpret_cast<uint4 *>(mout)[i] = reinterpret_cast<const uint4 *>(s.M[0])[i];
    } else {
        for (int i = tid; i < g.words; i += left) mout[i] = s.M[0][i];
    }
    if (tid == 0) a.fallback[1 + atomicAdd(a.fallback, 1)] = (int)o;
}

// Split path, third launch: the frames frame_regions_kernel could not finish in place (a.fallback: very busy masks -- more than
// kLeanSlots components or more runs in a row than its run table holds).  The stored mask -> close -> components, statistics,
// labels (K4, K5) with the full-size tables; the variances are left to region_variance_kernel.  A small persistent grid
// over the list, which is nearly always empty.
__global__ void __launch_bounds__(kGThreads, 6) frame_components_kernel(const KernelArgs a, long long total_frames) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    CompSmem &s = *reinterpret_cast<CompSmem *>(smem_raw);
    const Geometry &g = a.g;
    const int tid = threadIdx.x;
    const int n = a.fallback[0];
    for (int idx = blockIdx.x; idx < n; idx += gridDim.x) {
        const long long o = a.fallback[1 + idx];
        if (o < 0 || o >= total_frames) continue;
        __syncthreads();  // the previous frame is done with the tables
        const uint32_t *min_ = a.maskbits + (size_t)o * kMaxWords;
        const uint32_t hflags = a.fhdr[o].flags;
        for (int i = tid; i < g.words; i += kGThreads) s.M[0][i] = min_[i];
        __syncthreads();
        const bool have_prev = !(hflags & kHdrFirst);  // not the first frame of its clip
        // (variances in this kernel were measured slower than the separate wide pass, whose warps hide the cold reads of
        // the filtered images: all warps over each box +4.1 ms, one warp per region record as a tail here +7.9 ms,
        // against the 2.4 ms of region_variance_kernel)
        components_of_frame<CompSmem, kGThreads, 1>(a, s, g, tid, 0, (size_t)o, have_prev);
    }
}

// Second half of the frame pipeline for denoise clips (info.reserved[1] != 0): the denoised normalised image of every
// frame -> K4 (blur, threshold, close) -> K5 (components, statistics, labels); the variances are left to
// region_variance_kernel.  One CTA per frame at a time; same roles, shared-memory layout and code as the
// persistent kernel, without the recurrence.
__global__ void __launch_bounds__(kThreads, 1) mask_components_kernel(const KernelArgs a, long long total_frames,
                                                                      const uint8_t *denoised) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem &s = *reinterpret_cast<Smem *>(smem_raw);
    const Geometry &g = a.g;
    const int tid = threadIdx.x;
    for (long long o = blockIdx.x; o < total_frames; o += gridDim.x) {
        const int marker = a.info[o].reserved[1];
        if (marker == 0) continue;  // (uniform: every thread reads the same record)
        const uint8_t *u = denoised + (size_t)o * g.npx;
        for (int i = tid; i < g.npx / 16; i += kThreads) reinterpret_cast<uint4 *>(s.U)[i] = __ldg(reinterpret_cast<const uint4 *>(u) + i);
        __syncthreads();
        const int ith = (int)floorf(a.info[o].threshold);
        if (tid < kThreads - kCThreads)
            for (int grp = tid; grp < g.groups; grp += kThreads - kCThreads) blur_group(s, g, grp, 3u, 0, ith);
        __syncthreads();
        if (tid >= kThreads - kCThreads)
            components_of_frame<Smem, kCThreads, BAR_C>(a, s, g, tid - (kThreads - kCThreads), 0, (size_t)o, marker == 2);
        __syncthreads();
        if (tid == 0) a.info[o].reserved[1] = 0;
    }
}

// K6 for the frames the extraction kernel deferred (info.reserved[0] == 1): per-region variance of the
// normalised delta frame |norm255(F_t) - norm255(F_t-1)| over the component's bounding box
// (track/cliptracker.py:249-261,316-318).  One warp per frame; both filtered images are in the output buffer.
__global__ void __launch_bounds__(kVarThreads, 2048 / kVarThreads > 32 ? 32 : 2048 / kVarThreads) region_variance_kernel(Geometry g, long long total_frames, const float *filtered,
                                                              cpt_frame_info *info, cpt_region *regions) {
    const long long o = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (o >= total_frames) return;
    cpt_frame_info *fi = info + o;
    if (o == 0 || fi->reserved[0] != 1) return;
    const int n = min(fi->n_components, g.max_regions);
    const int cur_fmin = fi->filtered_min, cur_fmax = fi->filtered_max;
    const int prev_fmin = fi[-1].filtered_min, prev_fmax = fi[-1].filtered_max;
    const bool exact = norm255_exact(cur_fmin, cur_fmax, prev_fmin, prev_fmax);
    const float *fcur = filtered + (size_t)o * g.npx, *fprev = fcur - g.npx;
    for (int r = 0; r < n; ++r) {
        cpt_region *reg = regions + (size_t)o * g.max_regions + r;
        const int l = reg->x, tp = reg->y, bw = reg->width, bh = reg->height;
        if (l < 0 || tp < 0 || bw < 1 || bh < 1 || l + bw > g.W || tp + bh > g.H) continue;  // not a record of this launch
        region_variance<true>(g, l, tp, bw, bh, fcur, fprev, cur_fmin, cur_fmax, prev_fmin, prev_fmax, exact, lane, &reg->pixel_variance);
    }
    if (lane == 0) fi->reserved[0] = 0;
}

static_assert(sizeof(Smem) <= 232448, "shared memory budget (227 KB per CTA on sm_100)");

}  // namespace cpt
