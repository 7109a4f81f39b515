// cptrack_kernels.cuh -- sm_100a kernels for thermal-clip track extraction (DESIGN.md section 3.1): launch sizes,
// shared-memory layouts and the per-frame rules both launch plans share.
//
// The per-clip recurrence of the reference (WeightedBackground: background + per-pixel weight counter, the 45-frame
// sliding sum that replaces np.mean(get_last_x(45)), piclassifier/motiondetector.py:178-248 and
// track/cliptrackextractor.py:168-176) streams through the frames from HBM, and each frame emits filtered fp32 (K1), the
// uint8 label image (K5) and a compact region list (K5/K6).  Stages of a frame (SURVEY.md section 8a):
//   fused sweep   weighted background update of the previous frame (K7), then F = P - B, sliding sum, sum P,
//                 min/max F, per-quad maxima of F                                               (K1, K7, K8)
//   scalars       avg_change, normalisation range, mapped threshold, bound below which no pixel can fire  (K2)
//   marks         hot quads -> rows of marks -> work lists of 8-pixel groups
//   normalise     U = uint8(255*(G-min)/(max-min)) for the listed groups                        (K2)
//   blur          5x5 binomial blur in packed 16-bit lanes, threshold -> bit rows               (K4)
//   close         C[y] = M[y-1] | (M[y] & M[y-2]) on 32-bit row words                           (K4)
//   label         run-based union-find on the bit rows, OpenCV label order                      (K5)
//   regions       bbox / area / centroid sums per component, delta-frame variance               (K5, K6)
// Two launch plans run these stages and must give the same bits:
//   split path (batch launches that keep the filtered images and resume from no state): strip_sweep_kernel (strip_sweep.cu:
//     the recurrence, one CTA per (clip, strip of rows)) -> frame_scalars_kernel -> frame_regions_kernel (one small CTA per
//     frame: marks .. regions in place; the rare very busy mask goes on a list for frame_components_kernel) ->
//     region_variance_kernel
//   single kernel (streaming, resumed clips, regions-only): extract_clips_kernel, the stages as three warp roles
//     (sweep / mask / component warps) running concurrently on consecutive frames of the clip
// Each rule that decides those bits has one copy both plans call: here the scalars of a frame (frame_scalars_of), the
// rounded background average (rounded_background_average), the frame's info record (frame_info_of), the normalise
// (norm_u8, norm_u8_int) and the union-find; in extract_kernel.cu the work-list emission (emit_norm_groups,
// emit_blur_groups), normalise, blur and components of a frame and the region variance.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/cptrack.h"

namespace cpt {

// warp-specialised pipeline over consecutive frames: sweep warps (the recurrence), mask warps (scalars, work lists,
// normalise, blur) and component warps (labelling).
// 19 sweep warps: 15 rows x 40 quads per iteration at 160 pixels (the last 8 threads idle).  120 rows / 15 row groups = 8
// quads for every thread once the two border rows are balanced (Geometry::balanced): no warp is ever ahead of another
// (other sweep-warp counts were measured slower, DESIGN.md section 7).
constexpr int kPThreads = 608;
constexpr int kPWarps = kPThreads / 32;
constexpr int kMThreads = 128;                  // 4 mask warps
constexpr int kCThreads = 256;                  // 8 component warps
constexpr int kCWarps = kCThreads / 32;
constexpr int kThreads = kPThreads + kMThreads + kCThreads;
constexpr int kWarps = kThreads / 32;
// split path: frame_regions_kernel turns every frame into its mask, labels and regions with one four-warp CTA per frame;
// frame_components_kernel (full-size tables) redoes the frames whose masks are too busy for it
constexpr int kFThreads = 128;   // frame_regions_kernel
constexpr int kGThreads = 256;   // frame_components_kernel
constexpr int kVarThreads = 256;  // region_variance_kernel: one warp per frame
constexpr int kMaxPx = 19200;
constexpr int kQIter = (kMaxPx / 4 + kPThreads - 1) / kPThreads;  // 6 quads of 4 pixels per pixel thread
constexpr int kMaxW = 160;
constexpr int kMaxH = 120;
constexpr int kRowWords = kMaxW / 32;           // 5
constexpr int kMaxWords = kMaxH * kRowWords;    // 600
constexpr int kRunsPerRow = kMaxW / 2;          // 80
constexpr int kMaxRuns = kMaxH * kRunsPerRow;   // 9600
constexpr int kCompSlots = 256;                 // slot 255 = overflow sink
constexpr int kMeanFrames = CPT_MEAN_FRAMES;
constexpr uint16_t kSlotFlag = 0x8000u;

struct Geometry {
    int W, H, edge;
    int npx;        // W*H
    int groups;     // npx / 8
    int gpr;        // groups per row = W/8
    int row_words;  // ceil(W/32)
    int words;      // H*row_words
    int crop_w, crop_h, ncrop;
    int block_w;    // ceil(W/2): key = (y/2)*block_w + x/2
    int max_regions;
    uint32_t gpr_magic;  // grp / gpr == (grp * gpr_magic) >> 17   (grp < 4096, gpr < 32)
    uint32_t rw_magic;   // w / row_words == (w * rw_magic) >> 13  (w < 1024, row_words < 8)
    // quads of 4 pixels: the unit of the fused pixel sweep.  Rows edge .. H-1-edge are "owned"; the owner of
    // the first / last owned row also produces the border rows above / below it.
    int qpr;             // quads per row = W/4
    int rows_per_it;     // owned rows the pixel threads cover per sweep iteration = kPThreads / qpr (16 at 160 pixels)
    // 160x120, edge 1: the owners of the first and last owned row also produce a border row, so two rows are remapped to
    // row groups whose last iteration is free (owned_row_slot): owned row bal_a_oy -> group bal_a_r, bal_b_oy -> bal_b_r
    int balanced;
    int bal_a_oy, bal_a_r, bal_b_oy, bal_b_r;
    // strip sweep (strip_sweep.cu): the frame is cut into n_strips bands of whole rows, strip s = rows
    // [s * H / n_strips, (s + 1) * H / n_strips), at most kStripPxMax pixels each
    int n_strips;
    uint32_t qpr_magic, h_magic;  // q / qpr == umulhi(q, qpr_magic), v / H == umulhi(v, h_magic)  (q * qpr, v * H < 2^32)
    uint32_t qw_magic;            // i / (qpr / 4) == umulhi(i, qw_magic) unless qpr / 4 == 1 (words of quad bytes per row)
    uint8_t strip_y0[20];         // first row of strip s (s <= n_strips <= kMaxStrips = 16)
};
// strip that holds image row y
__device__ __forceinline__ int strip_of_row(const Geometry &g, int y) { return (int)__umulhi((uint32_t)((y + 1) * g.n_strips - 1), g.h_magic); }

// sweep slot (iteration, row group) that processes owned row oy; its quads are sweep threads r * qpr .. r * qpr + qpr - 1
__host__ __device__ inline void owned_row_slot(const Geometry &g, int oy, int &it, int &r) {
    it = oy / g.rows_per_it;
    r = oy - it * g.rows_per_it;
    if (g.balanced) {
        if (oy == g.bal_a_oy) { it = kQIter - 1; r = g.bal_a_r; }
        else if (oy == g.bal_b_oy) { it = kQIter - 1; r = g.bal_b_r; }
    }
}

// Per-clip persistent record in global memory (cpt_state_bytes()).
struct StateHeader {
    double average;
    int32_t frames_seen;
    int32_t initialised;
    int32_t prev_fmin, prev_fmax;
    int32_t have_prev;
    int32_t pad[9];
};
static_assert(sizeof(StateHeader) == 64, "state header is one 64-byte line");

__host__ __device__ inline size_t state_bytes(int npx) {
    return sizeof(StateHeader) + (size_t)npx * (2 + 2 + 4 + 4);
}

// keep-test table for WeightedBackground (motiondetector.py:214-218):
//   keep  <=>  fp64(B) < fl64(fp64(A) - w_k)   for integers 0 <= B, A < 2^16, w_k accumulated in fp64.
// With c = ceil(w_k), g = c - w_k, d = A - B:  d > c keeps, d < c does not, and for d == c the exact
// right-hand side is B + g, which rounds above B iff g > ulp(B)/2, i.e. iff B < 2^E with
// E = ceil(log2 g) + 53 (any g > 0 when B == 0).  Entry layout (cpt_build_weight_table):
//   bits 0..15  thr   = c if E >= 16 (always rounds up), else c + 1   (clamped to 65535)
//   bits 16..31 bound = 0 if g == 0 or E >= 16, else 2^max(E, 0)
//   keep = (d >= thr) || (d == thr - 1 && B < bound)   ==   d >= thr - (B < bound)
struct WeightTable {
    const uint32_t *thr;
    int max_count;
    int has_bounds;   // some entry has a non-zero bound
    int max_bound;    // largest bound of the table: backgrounds >= max_bound never need the correction
    int linear_upto;  // entries [0, linear_upto) are exactly thr = k + 1, bound = 0 (weight_add == 1)
};
constexpr int kSmemWeights = 1024;

// ---- strip sweep (split path, strip_sweep.cu) -------------------------------------------------
constexpr int kStripPxMax = 1920;   // pixels of one strip (12 rows at 160 pixels): 480 quads, one per consumer thread
constexpr int kMaxStrips = 16;
constexpr int kStripThreads = kStripPxMax / 4 + 64;  // one consumer thread per quad + the copy warp + the fold warp
// What one strip CTA found in one pass (frame t, or the tail pass that only applies the last background update), folded
// over its warps.  [pass][strip] in global memory; frame_scalars_kernel folds the strips of a frame.
struct StripRec {
    uint32_t psum;     // sum of the strip's thermal pixels
    int32_t fmin, fmax;  // extrema of filtered = thermal - background over the strip
    int32_t nbsum;     // minus the sum of the background over the strip's crop pixels (after this pass's update)
    int32_t pmin, pmax;  // thermal extrema (CPT_CLIP_FRAME_STATS)
    uint32_t fabs_sum; // sum |filtered| (CPT_CLIP_FRAME_STATS)
    int32_t ref_changed;  // (reference the strip's quad bytes were stored against) << 1 | (some background pixel changed)
};
static_assert(sizeof(StripRec) == 32, "two 16-byte vectors");
// Per output frame, written by frame_scalars_kernel for frame_regions_kernel: one 64-byte line with everything the kernel
// needs to know about the frame before it touches pixels.
struct __align__(16) FrameHdr {
    uint32_t nmagic;   // (255 v) / range == (255 v * nmagic) >> nshift; 0: the fp32 divide
    int32_t nshift;
    uint32_t flags;    // kHdr*: valid, first frame of its clip, dense (no usable bound for the quad bytes), denoise clip
    uint32_t hot_strips;  // bit s: strip s may hold a hot quad
    int16_t theta[kMaxStrips];  // quad byte b of strip s is hot <=> b >= theta[s]
    float threshold;   // cpt_frame_info::threshold, avg_change, norm_min, norm_max (K2)
    int32_t avg_change, norm_min, norm_max;
};
static_assert(sizeof(FrameHdr) == 64, "four 16-byte vectors");
constexpr uint32_t kHdrValid = 1u, kHdrFirst = 2u, kHdrDense = 8u, kHdrDenoise = 16u;
constexpr int kQuadRefBias = 64;    // a strip's quad bytes are stored against (its min filtered value some frames ago) + bias
constexpr int kListCap = 1024;  // marked groups per frame handled through the work lists (more: dense sweep)

struct KernelArgs {
    Geometry g;
    const uint16_t *frames;
    const cpt_clip *clips;
    int n_clips;
    cpt_region *regions;
    cpt_frame_info *info;
    float *filtered;
    uint8_t *labels;
    float *scratch;       // [gridDim.x][4][npx] fp32 when filtered == nullptr
    uint8_t *state;       // n_clips * state_bytes or nullptr
    int *work_counter;    // zeroed before launch
    long long *debug;     // [gridDim.x][32] phase cycle counters (CPT_PHASE_TIMING builds), else nullptr
    int defer_variance;   // leave K6 of frames t > 0 to region_variance_kernel (needs `filtered`)
    uint8_t *u8_frames;   // [total_frames][npx] normalised images of denoise clips (ctx scratch), else nullptr
    const uint16_t *zero_frame;  // npx zeros: stands in for the frame leaving the 45-frame window while it fills
    uint32_t *maskbits;   // [total_frames][kMaxWords] thresholded masks of the frames left to frame_components_kernel
    int *fallback;        // [1 + total_frames]: count, then the frames frame_regions_kernel left to frame_components_kernel
    // strip sweep outputs (split path)
    int8_t *qbytes;       // [total_frames][H][qpr] per quad: max filtered - strip reference, saturated to int8
    StripRec *prec;       // [total_frames + n_clips][n_strips]: pass records (clip ci's tail pass at total_frames + ci)
    FrameHdr *fhdr;       // [total_frames]
    long long total_frames;
    WeightTable tables[4];
};

// sweep -> mask warps: what one frame's sweep found
struct FrameMsg {
    uint32_t red[12];  // sum P, min F, max F, min P, max P, sum |F|, sum B, changed
    int32_t qref;      // reference value the per-quad maxima in Smem::qmax8 are stored against
    int32_t update;    // the sweep applied a background update
    int32_t is_frame;  // 0: tail pass (update only)
    int32_t pad;
};

struct __align__(16) Smem {
    uint32_t S[kMaxPx];        // sliding sum of the last <=45 frames
    uint16_t B[kMaxPx];        // background (integer valued)
    uint16_t K[kMaxPx];        // weight counter k (background_weight = w_k)
    uint8_t U[kMaxPx];         // normalised uint8 image; reused as the label image
    uint16_t parent[kMaxRuns]; // union-find over runs
    uint32_t M[2][kMaxWords];  // thresholded mask, bit rows (byte g = 8 pixels of group g), double buffered
    uint32_t C[kMaxWords];     // closed mask
    uint32_t ST[kMaxWords];    // run-start bits of C
    uint8_t base[kMaxWords + 8]; // run starts in earlier words of the same row
    int32_t c_key[kCompSlots], c_area[kCompSlots], c_sx[kCompSlots], c_sy[kCompSlots];
    int32_t c_l[kCompSlots], c_t[kCompSlots], c_r[kCompSlots], c_b[kCompSlots];
    uint8_t c_rank[kCompSlots];
    uint32_t red_u[(kWarps * 12 > 2 * kPWarps * 8) ? kWarps * 12 : 2 * kPWarps * 8];  // per-warp partial results
    int32_t bcast_i[16];
    int32_t msg[2][4];         // pixel warps -> component warps, per mask buffer: filtered min, max
    double bcast_d[4];
    uint32_t wthr[kSmemWeights];                   // first entries of the clip's keep-test table
    // per owned quad q = it * kPThreads + ptid (= owned row * qpr + column quad): max F - qref saturated to int8,
    // written by the sweep warps at the end of a frame, turned into hot64 by the mask warps
    int8_t qmax8[kQIter * kPThreads];
    unsigned long long hot64[kMaxH];  // per owned row, one bit per quad: some pixel can exceed the threshold
    FrameMsg fm[2];
    int32_t fth_latest;      // last bound the mask warps computed (INT32_MIN: none yet): the next qref
    int32_t final_prev[3];   // filtered min / max of the last frame, have_prev (for the state record)
    double init_average, final_average;
    uint16_t list_u[kListCap];  // groups of 8 pixels to normalise this frame (need_u)
    uint16_t list_b[kListCap];  // groups of 8 pixels to blur this frame: group | quad marks << 14
    int32_t ncomp;
};

// shared memory of frame_regions_kernel (one frame per CTA, one band of rows at a time: hot quads -> work lists -> normalise
// -> blur + threshold)
constexpr int kBandHalo = 4;    // rows of normalised values a blur output can reach above / below a hot quad
constexpr int kBandRows = 24;     // hot rows one band covers
constexpr int kFMinBlocks = 13;   // frame_regions_kernel CTAs per SM the register allocation allows
constexpr int kBandURows = kBandRows + 2 * kBandHalo;
constexpr int kBandList = kBandURows * (kMaxW / 8);  // every group of every row of the band: the lists cannot overflow
constexpr int kLeanParents = 1024;  // run ids of the in-CTA components stage: rows of the mask's extent * runs per row
constexpr int kLeanSlots = 32;      // components it numbers; slot kLeanSlots is the overflow sink (more: the fallback kernel)
struct __align__(16) MaskSmem {
    union {
        struct {
            uint8_t U[kBandURows * kMaxW];     // normalised bytes of the band's rows
            uint16_t list_u[kBandList];        // groups of 8 pixels to normalise: band row * gpr + group
            uint16_t list_b[kBandList];        // groups to blur: frame group | quad marks << 14
        };
        // ... and once the mask is complete, the components stage: closed mask, run-start bits, run starts in earlier words
        // of the row (all indexed by word within the mask's row extent)
        struct {
            uint32_t C[kMaxWords];
            uint32_t ST[kMaxWords];
            uint8_t base[kMaxWords + 8];
            uint16_t wlist[kMaxWords];     // the non-empty words of C
        };
    };
    alignas(16) unsigned long long hot64[kMaxH];   // per frame row, one bit per quad
    alignas(16) uint32_t M[1][kMaxWords];          // the frame's mask, bit rows (moved as 16-byte vectors)
    uint16_t parent[kLeanParents];     // union-find over runs
    int32_t c_key[kLeanSlots + 1], c_area[kLeanSlots + 1], c_sx[kLeanSlots + 1], c_sy[kLeanSlots + 1];
    int32_t c_l[kLeanSlots + 1], c_t[kLeanSlots + 1], c_r[kLeanSlots + 1], c_b[kLeanSlots + 1];
    uint8_t c_rank[kLeanSlots + 4];
    alignas(16) int16_t theta[kMaxStrips];         // (written as two 16-byte vectors)
    // per band parity (warp 0 prepares the next band's record while the others may still read this one's):
    int32_t count[2][2];               // list lengths
    int32_t band[2][2];                // first / last hot row of the band (last < 0: none left)
    int32_t ncomp, overflow, nwords;
};
static_assert(kMaxH <= 128, "frame_regions_kernel keeps the set of hot rows in four ballot words");
static_assert(kMaxH * (kMaxW / 8) <= (1 << 14), "a blur list entry keeps the group in 14 bits");

// shared memory of frame_components_kernel (one frame per CTA: close -> components, statistics, labels)
struct __align__(16) CompSmem {
    uint16_t parent[kMaxRuns];
    uint32_t C[kMaxWords];
    uint32_t M[1][kMaxWords];
    uint32_t ST[kMaxWords];
    uint8_t base[kMaxWords + 8];
    int32_t c_key[kCompSlots], c_area[kCompSlots], c_sx[kCompSlots], c_sy[kCompSlots];
    int32_t c_l[kCompSlots], c_t[kCompSlots], c_r[kCompSlots], c_b[kCompSlots];
    uint8_t c_rank[kCompSlots];
    int32_t bcast_i[16];
    int32_t ncomp;
};

__device__ __forceinline__ uint4 ldg16(const void *p) { return __ldg(reinterpret_cast<const uint4 *>(p)); }

// dp2a on packed uint16 pairs (IDP runs beside IMAD/FFMA, not on the half-rate integer ALU pipe):
//   c + a.lo * b.byte0 + a.hi * b.byte1, a unsigned 16-bit halves, b signed bytes.
__device__ __forceinline__ int dp2a_us(uint32_t a, int b, int c) {
    int d;
    asm("dp2a.lo.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
constexpr int kLoP = 0x0001, kLoN = 0x00ff, kHiP = 0x0100, kHiN = 0xff00, kBoth = 0x0101;

__device__ __forceinline__ void unpack8(const uint4 &v, int (&o)[8]) {
    o[0] = v.x & 0xffff; o[1] = v.x >> 16; o[2] = v.y & 0xffff; o[3] = v.y >> 16;
    o[4] = v.z & 0xffff; o[5] = v.z >> 16; o[6] = v.w & 0xffff; o[7] = v.w >> 16;
}

__device__ __forceinline__ uint4 pack8(const int (&o)[8]) {
    uint4 v;
    v.x = (uint32_t)o[0] | ((uint32_t)o[1] << 16); v.y = (uint32_t)o[2] | ((uint32_t)o[3] << 16);
    v.z = (uint32_t)o[4] | ((uint32_t)o[5] << 16); v.w = (uint32_t)o[6] | ((uint32_t)o[7] << 16);
    return v;
}

// K2: uint8(255*(v)/(range)) exactly as numpy fp32: fl(fl(255*v)/range), truncated.
__device__ __forceinline__ uint32_t norm_u8(int v, float range_f) {
    float num = __fmul_rn(255.0f, (float)v);
    return (uint32_t)__fdiv_rn(num, range_f);
}
// Same value in integers when 255*range < 2^24 (every product exact in fp32): the fp32
// quotient of two integers n < 2^24, r < 2^17 can only round up to an integer q when
// q - n/r <= ulp/2 <= 2^-17 < 1/r, i.e. never unless exact, so trunc(fl(n/r)) == n / r.
// n / r by multiplication: m = ceil(2^(24+l) / r), l = ceil(log2 r)  (Granlund-Montgomery).
__device__ __forceinline__ uint32_t norm_u8_int(int v, uint32_t m, int shift) {
    return (uint32_t)(((unsigned long long)(uint32_t)(255 * v) * m) >> shift);
}

// WeightedBackground.average after an update that changed the background: int(round(np.average(background))),
// motiondetector.py:232, of the background summed over the ncrop crop pixels -- half to even, in integers.
__device__ __forceinline__ double rounded_background_average(uint32_t bsum, uint32_t ncrop) {
    uint32_t qa = bsum / ncrop;
    const uint32_t ra = bsum - qa * ncrop;
    if (2u * ra > ncrop || (2u * ra == ncrop && (qa & 1u))) qa += 1u;
    return (double)qa;
}

struct FrameScalars {
    int ac, gmn, gmx, fth;
    float thr;
    uint32_t nmagic;
    int nshift;
};

// K2 scalars of one frame (track/cliptracker.py:93-122, imageprocessing.py:151-169) from its sums: avg_change, the
// normalisation range, the mapped threshold (fp32 as numpy >= 2 evaluates it), the bound F >= fth below which a pixel cannot
// reach the threshold (INT32_MIN: no usable bound) and the Granlund-Montgomery constants of the integer normalise.
__device__ __forceinline__ FrameScalars frame_scalars_of(uint32_t psum, int fmin, int fmax, double average, int background_thresh, int npx) {
    FrameScalars r;
    // avg_change = int(round(np.average(thermal) - background average)), cliptracker.py:103-105
    const double avg_int = rint(average);
    if (avg_int == average && average >= 0.0 && average < 65536.0) {
        // integer average (always, once the background has changed): round_half_even((sum - avg * n) / n) in integers;
        // identical to the fp64 expression because the only ties are exact.  |sum - avg * n| < 2^31.
        const int num = (int)psum - (int)avg_int * npx;
        int qd = num / npx, rem = num - qd * npx;
        if (rem < 0) { rem += npx; qd -= 1; }
        if (2 * rem > npx || (2 * rem == npx && (qd & 1))) qd += 1;
        r.ac = qd;
    } else {
        r.ac = (int)rint((double)psum / (double)npx - average);
    }
    r.gmx = max(fmax - r.ac, 0);
    r.gmn = max(fmin - r.ac, 0);
    r.fth = INT32_MIN;
    r.nmagic = 0;  // 0: the fp32 divide; else (255 v) / range == (255 v * nmagic) >> nshift for 255 v < 2^24
    r.nshift = 0;
    if (r.gmx == r.gmn) {
        r.thr = (float)background_thresh;  // cliptracker.py:118-119
    } else {
        const float range = (float)r.gmx - (float)r.gmn;
        r.thr = __fmul_rn(__fdiv_rn((float)background_thresh, range), 255.0f);
        const unsigned rr = (unsigned)(r.gmx - r.gmn);
        if (255ull * rr < (1ull << 24)) {
            // every product is exact in fp32 here, so trunc(fl(255 v / r)) == (255 v) / r and a quad can only produce
            // foreground if one of its pixels has U > floor(thr):  U >= ith + 1  <=>  v >= ceil((ith + 1) r / 255),
            // v = max(F - ac, 0) - gmn, i.e. F >= fth (the bound is >= 1, so the clamp never matters)
            const int it = (int)floorf(r.thr);
            if (it >= 0 && it < 255) r.fth = (int)(((unsigned)(it + 1) * rr + 254u) / 255u) + r.ac + r.gmn;
            // Granlund-Montgomery: l = ceil(log2 r), m = ceil(2^(24 + l) / r) < 2^25.  The fp64 quotient is exact for powers
            // of two and otherwise at least 1/r >= 2^-17 away from an integer: its ceiling is m.
            const int l = (rr <= 1u) ? 0 : 32 - __clz((int)(rr - 1u));
            r.nshift = 24 + l;
            r.nmagic = (uint32_t)ceil(ldexp(1.0, r.nshift) / (double)rr);
        }
    }
    return r;
}

// The frame's info record from its scalars and sums; the thermal extrema and sum |filtered| only with
// CPT_CLIP_FRAME_STATS.  dn_marker goes to reserved[1], the denoise marker (0: not a denoise clip; 1: a clip's first
// frame; 2: the previous filtered image is frame o - 1).  frame_scalars_kernel knows it here; the single kernel passes 0
// and its mask warps write the marker once they have emitted the frame's normalised image.
__device__ __forceinline__ cpt_frame_info frame_info_of(const FrameScalars &fs, double average, uint32_t psum, int fmin, int fmax,
                                                        bool want_stats, int pmin, int pmax, uint32_t fabs_sum, int dn_marker) {
    cpt_frame_info fi;
    fi.background_average = average;
    fi.threshold = fs.thr; fi.norm_min = fs.gmn; fi.norm_max = fs.gmx; fi.avg_change = fs.ac;
    fi.filtered_min = fmin; fi.filtered_max = fmax; fi.n_components = 0;
    fi.thermal_min = want_stats ? pmin : 0; fi.thermal_max = want_stats ? pmax : 0;
    fi.thermal_sum = psum; fi.abs_filtered_sum = want_stats ? fabs_sum : 0u; fi.thermal_median = 0.f;
    fi.reserved[0] = 0;
    fi.reserved[1] = dn_marker;
    return fi;
}

// normalize(F, new_max=255) of get_delta_frame (track/cliptracker.py:249-261): fp64 arithmetic
// because min/max are float64 scalars there; result cast to fp32.
__device__ __forceinline__ float norm255_f64(float f, double mn, double mx) {
    if (mx == mn) return (mx == 0.0) ? 0.0f : (float)((double)f / mx);
    return (float)(255.0 * ((double)f - mn) / (mx - mn));
}

// ---- run bookkeeping on the closed mask ------------------------------------------------------
// Id of the run that holds pixel x of a row whose first word in the tables is w0 (row `row` of the table, rpr ids per row):
// the runs that start in the earlier words of the row (base) and in bits 0 .. x & 31 of word x >> 5.
template <class SM>
__device__ __forceinline__ int run_id(const SM &s, int w0, int row, int rpr, int x) {
    const int w = w0 + (x >> 5), b = x & 31;
    return row * rpr + (int)s.base[w] + __popc(s.ST[w] & (0xffffffffu >> (31 - b))) - 1;
}

__device__ __forceinline__ int uf_find(volatile uint16_t *parent, int a) {
    // follows parents until a root (parent == self) or a flagged slot entry
    while (true) {
        int p = parent[a];
        if (p == a || (p & kSlotFlag)) return a;
        a = p;
    }
}

__device__ __forceinline__ void uf_union(uint16_t *parent, int a, int b) {
    volatile uint16_t *vp = parent;
    while (true) {
        a = uf_find(vp, a);
        b = uf_find(vp, b);
        if (a == b) return;
        if (a < b) { int t = a; a = b; b = t; }  // a > b: hang the larger root under the smaller
        unsigned short old = atomicCAS(reinterpret_cast<unsigned short *>(parent + a), (unsigned short)a,
                                       (unsigned short)b);
        if (old == (unsigned short)a) return;
    }
}

__device__ __forceinline__ int uf_slot(volatile uint16_t *parent, int a) {
    while (true) {
        int p = parent[a];
        if (p & kSlotFlag) return p & 0xff;
        a = p;
    }
}

}  // namespace cpt
