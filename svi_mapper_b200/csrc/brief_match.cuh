// brief_match.cuh -- BRIEF-32 on box-sum images, dense scan-line Hamming search, triangulation.
//
// Replaces the bodies of (reference paths):
//   cv::xfeatures2d::BriefDescriptorExtractor::compute        src/core/CTriangulator.cpp:83,217,288
//   cv::BFMatcher(NORM_HAMMING)::match (1 x N arg-min)         src/core/CTriangulator.cpp:93,227,298
//   CTriangulator::getPointTriangulatedInRIGHT[Full]          src/core/CTriangulator.cpp:51-119,185-253
//   CTriangulator::getPointTriangulatedInLEFT (7 args)        src/core/CTriangulator.cpp:255-324
//   CTriangulator::getPointInLEFT                             src/core/CTriangulator.cpp:326-356
//   the per-key-point loop of addNewLandmarks                  src/core/CFundamentalMatcher.cpp:109-175
//   trackManual stage 1                                        src/core/CFundamentalMatcher.cpp:1404-1538
//
// Work decomposition: one warp per query.  The candidates of a scan-line search are consecutive
// pixels of one image row, so lane l evaluates candidates 2l and 2l+1 of a 64-candidate chunk
// from ONE 32-bit shared-memory load per test point: the u16 box sums of two neighbouring
// candidates are neighbours in memory.  The 256 test pairs are template constants
// (brief_pattern_32.h), so every shared-memory offset is an instruction immediate.  Both
// comparisons of a pair are one packed half-precision compare (values <= 20655 < 0x7C00 are
// positive finite fp16 bit patterns, ordered like the integers): see lt_mask_u16x2.
#pragma once
#include <cuda.h>  // CUtensorMap (types only; the encoder is fetched through cudaGetDriverEntryPoint)
#include <utility>
#ifdef SVI_BRIEF_PATTERN_HEADER   // another pair table (tools/gen_pattern_header.py --table ... --out ...)
#include SVI_BRIEF_PATTERN_HEADER
#else
#include "brief_pattern_32.h"
#endif
#include "common.cuh"

namespace svi {

constexpr signed char kPat[SVI_BRIEF_NTESTS][4] = SVI_BRIEF_PATTERN_INIT;
__device__ __align__(16) const signed char d_pat[SVI_BRIEF_NTESTS][4] = SVI_BRIEF_PATTERN_INIT;   // rows are 4-byte aligned: read as char4
__device__ __forceinline__ char4 brief_pattern(int t) { return __ldg(reinterpret_cast<const char4*>(d_pat) + t); }

constexpr int PATCH_ROWS = 2 * kBriefReach + 1;        // 49
constexpr int PATCH_SLOTS = 64;                        // 2 candidate slots per lane and pass
constexpr int PATCH_CHUNK = PATCH_SLOTS - 2;           // candidates per pass (slot 0 is idle when the window parity is odd)
constexpr int PATCH_W = PATCH_SLOTS + 2 * kBriefReach + 8; // 120 u16 per row: window start rounded down to 8 elements
constexpr int PATCH_WORDS = PATCH_W / 2;               // 60
constexpr int PATCH_COPY_BYTES = PATCH_ROWS * PATCH_W * 2;          // 10976: one TMA box
constexpr int PATCH_COPY_STRIDE = (PATCH_COPY_BYTES + 127) / 128 * 128; // TMA destinations are 128-B aligned
constexpr int PATCH_COPY_WORDS = PATCH_COPY_STRIDE / 4;
constexpr int MATCH_WARPS = 3;                                      // 3 CTAs/SM -> 9 warps, 207 KB of windows
constexpr int MATCH_SMEM_PER_WARP = 2 * PATCH_COPY_STRIDE;          // even- and odd-aligned copies
constexpr int MATCH_SMEM = MATCH_WARPS * MATCH_SMEM_PER_WARP + MATCH_WARPS * 8;  // + one mbarrier per warp

// ------------------------------------------------------------------ TMA / mbarrier (sm_90+ PTX)
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int x, int y, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(dst), "l"(map), "r"(x), "r"(y), "r"(bar)
        : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(bar), "r"(parity)
        : "memory");
}

// Per-warp staging state: two shared copies of the box-sum window + the warp's mbarrier.
// TMA tile loads must start on a 16-byte boundary of the inner dimension (measured on B200: any
// other start faults with "illegal instruction"), so a window starts at a multiple of 8 columns and
// the copy that is one element further right comes from the plane stored shifted by one element.
struct PatchStage {
    const CUtensorMap* map;    // 2-D u16 tensor over S(y,x):   (W, frames*H), row pitch box_pitch
    const CUtensorMap* map_s;  // same geometry over the shifted plane S(y,x+1)
    int row_base;              // first tensor row of this query's frame
    uint32_t smem_a;          // shared address of copy A (copy B follows at +PATCH_COPY_STRIDE)
    const uint32_t* words;    // generic pointer to copy A
    uint32_t bar;             // shared address of the mbarrier
    uint32_t phase;           // parity of the next completion
};

// One elected lane arms the barrier and issues both box copies (col0 is a multiple of 8):
// A[r][k] = S[row0+r][col0+k], B[r][k] = S[row0+r][col0+1+k]; out-of-range elements are zero-filled.
__device__ __forceinline__ void patch_issue(const PatchStage& ps, int row0, int col0, int lane) {
    if (lane == 0) {
        fence_proxy_async();   // earlier generic-proxy reads of the buffers are ordered before the async writes
        mbar_expect_tx(ps.bar, 2 * PATCH_COPY_BYTES);
        tma_load_2d(ps.smem_a, ps.map, col0, ps.row_base + row0, ps.bar);
        tma_load_2d(ps.smem_a + PATCH_COPY_STRIDE, ps.map_s, col0, ps.row_base + row0, ps.bar);
    }
}
__device__ __forceinline__ void patch_wait(PatchStage& ps) {
    mbar_wait(ps.bar, ps.phase);
    ps.phase ^= 1u;
}

// ------------------------------------------------------------------ descriptor at one point
// Lanes = tests (8 rounds of 32).  Word format used throughout the kernels: word j holds tests
// 32j..32j+31 with test 32j+t at bit 31-t, i.e. the big-endian read of descriptor bytes 4j..4j+3.
__device__ __forceinline__ void brief_at_point(const uint16_t* __restrict__ box, int box_pitch, int cx,
                                               int cy, int lane, uint32_t (&w)[kDescWords]) {
#pragma unroll
    for (int j = 0; j < kDescWords; ++j) {
        const char4 p = brief_pattern(32 * j + lane);
        uint32_t s1 = box[(cy + p.x) * box_pitch + cx + p.y];
        uint32_t s2 = box[(cy + p.z) * box_pitch + cx + p.w];
        w[j] = __brev(__ballot_sync(0xFFFFFFFFu, s1 < s2));
    }
}

__device__ __forceinline__ uint32_t desc_word_to_bytes(uint32_t w) { return __byte_perm(w, 0, 0x0123); }

__device__ __forceinline__ void store_desc(uint8_t* dst, const uint32_t (&w)[kDescWords], int lane) {
    uint32_t v = 0;
#pragma unroll
    for (int j = 0; j < kDescWords; ++j) if (lane == j) v = w[j];
    if (lane < kDescWords) reinterpret_cast<uint32_t*>(dst)[lane] = desc_word_to_bytes(v);
}

__device__ __forceinline__ void load_desc(const uint8_t* src, uint32_t (&w)[kDescWords]) {
#pragma unroll
    for (int j = 0; j < kDescWords; ++j) w[j] = desc_word_to_bytes(reinterpret_cast<const uint32_t*>(src)[j]);
}

__device__ __forceinline__ int hamming_words(const uint32_t (&a)[kDescWords], const uint32_t (&b)[kDescWords]) {
    int d = 0;
#pragma unroll
    for (int j = 0; j < kDescWords; ++j) d += __popc(a[j] ^ b[j]);
    return d;
}

// ------------------------------------------------------------------ unrolled pair tests
// One 32-bit LDS per test point fetches the box sums of two adjacent candidates.  Box sums are
// <= 81*255 = 20655 < 0x7C00, i.e. bit patterns of positive finite fp16 numbers, whose order equals the
// integer order (denormals included, no flush): one packed half-precision compare on the FMA pipe tests
// both candidates and returns 0xFFFF per true half, so a test costs one compare and one LOP3 that keeps
// the bit of this test in a 16-test accumulator (low half = even candidate, high half = odd candidate).
__device__ __forceinline__ uint32_t lt_mask_u16x2(uint32_t a, uint32_t b) {
    uint32_t m;
    asm("set.lt.u32.f16x2 %0, %1, %2;" : "=r"(m) : "r"(a), "r"(b));
    return m;
}

// PW = 32-bit words per row of the staged window (the per-warp window of the scan-line kernels, or the tile a CTA of the
// binned matcher shares).
template <int T, int PW = PATCH_WORDS>
__device__ __forceinline__ void brief_pair_test(const uint32_t* __restrict__ Al, const uint32_t* __restrict__ Bl,
                                                uint32_t& acc) {
    constexpr int c1 = kPat[T][1] + kBriefReach, c2 = kPat[T][3] + kBriefReach;
    constexpr int o1 = (kPat[T][0] + kBriefReach) * PW + (c1 >> 1);
    constexpr int o2 = (kPat[T][2] + kBriefReach) * PW + (c2 >> 1);
    constexpr uint32_t bit = 0x00010001u << (15 - (T & 15));
    const uint32_t a = (c1 & 1) ? Bl[o1] : Al[o1];
    const uint32_t b = (c2 & 1) ? Bl[o2] : Al[o2];
    acc |= lt_mask_u16x2(a, b) & bit;
}

template <int G, int PW, int... I>
__device__ __forceinline__ uint32_t brief_pair_group(const uint32_t* __restrict__ Al, const uint32_t* __restrict__ Bl,
                                                     std::integer_sequence<int, I...>) {
    uint32_t acc = 0u;
    (brief_pair_test<G * 16 + I, PW>(Al, Bl, acc), ...);
    return acc;
}

template <int J, int PW = PATCH_WORDS>
__device__ __forceinline__ void brief_pair_word(const uint32_t* __restrict__ Al, const uint32_t* __restrict__ Bl,
                                                uint32_t& wlo, uint32_t& whi) {
    const uint32_t e = brief_pair_group<2 * J, PW>(Al, Bl, std::make_integer_sequence<int, 16>{});      // tests 32J .. 32J+15
    const uint32_t o = brief_pair_group<2 * J + 1, PW>(Al, Bl, std::make_integer_sequence<int, 16>{});  // tests 32J+16 .. 32J+31
    wlo = __byte_perm(o, e, 0x5410);   // (e.lo16 << 16) | o.lo16
    whi = __byte_perm(o, e, 0x7632);   // (e.hi16 << 16) | o.hi16
}

template <int PW, int... J>
__device__ __forceinline__ void brief_pair_all_pw(const uint32_t* __restrict__ Al, const uint32_t* __restrict__ Bl,
                                                  uint32_t (&wlo)[kDescWords], uint32_t (&whi)[kDescWords],
                                                  std::integer_sequence<int, J...>) {
    (brief_pair_word<J, PW>(Al, Bl, wlo[J], whi[J]), ...);
}
template <int... J>
__device__ __forceinline__ void brief_pair_all(const uint32_t* __restrict__ Al, const uint32_t* __restrict__ Bl,
                                               uint32_t (&wlo)[kDescWords], uint32_t (&whi)[kDescWords],
                                               std::integer_sequence<int, J...> seq) {
    brief_pair_all_pw<PATCH_WORDS>(Al, Bl, wlo, whi, seq);
}

// ------------------------------------------------------------------ one whole descriptor per LANE
// For pools of unrelated points (the corners of a stage-2 window, the samples of a stage-3 line) every lane describes its
// own point: the 512 box-sum gathers of a descriptor are issued 64 at a time (one 32-test word: offsets are compile-time
// constants, dy * pitch + dx), so a round of 32 points costs eight memory round trips instead of hundreds.
template <int T>
__device__ __forceinline__ void brief_gather_pair(const uint16_t* __restrict__ c, int pitch, uint32_t& a, uint32_t& b) {
    constexpr int y1 = kPat[T][0], x1 = kPat[T][1], y2 = kPat[T][2], x2 = kPat[T][3];
    a = __ldg(c + y1 * pitch + x1);
    b = __ldg(c + y2 * pitch + x2);
}
template <int J, int... I>
__device__ __forceinline__ uint32_t brief_lane_word(const uint16_t* __restrict__ c, int pitch, std::integer_sequence<int, I...>) {
    uint32_t a[32], b[32];
    (brief_gather_pair<32 * J + I>(c, pitch, a[I], b[I]), ...);
    uint32_t bits = 0u;
    ((bits |= (a[I] < b[I] ? 1u : 0u) << (31 - I)), ...);
    return bits;
}
template <int... J>
__device__ __forceinline__ void brief_lane_words(const uint16_t* __restrict__ c, int pitch, uint32_t (&w)[kDescWords],
                                                 std::integer_sequence<int, J...>) {
    ((w[J] = brief_lane_word<J>(c, pitch, std::make_integer_sequence<int, 32>{})), ...);
}
// descriptor (word format of the kernels) of the point (cx, cy) of a box-sum plane, computed by the calling lane alone
__device__ __forceinline__ void brief_at_point_lane(const uint16_t* __restrict__ box, int box_pitch, int cx, int cy,
                                                    uint32_t (&w)[kDescWords]) {
    brief_lane_words(box + cy * box_pitch + cx, box_pitch, w, std::make_integer_sequence<int, kDescWords>{});
}

struct SearchResult {
    int status, dist, idx;
    float u, v;
    uint32_t w[kDescWords];
};

// Geometry of one scan-line search, shared body of CTriangulator.cpp:59-117 (RIGHT, first = 0) and
// :264-322 (LEFT, first = 1): ROI by truncation, pool key-points (border + first + i, border),
// BRIEF's border filter inside the ROI.  Warp-uniform.
struct SearchPlan {
    int status;        // SVI_OK when there is at least one candidate to evaluate
    int n_valid, i_lo; // surviving pool key-points [i_lo, i_lo + n_valid)
    int gx_lo, gy;     // image column of candidate i_lo, image row of all candidates
    int first;
    float border, u_tl, v_tl;
};

__device__ __forceinline__ void search_plan(int W, int H, float img_width_f, float u_tl, float v_tl, float size,
                                            int first, int n_pool, int lane, SearchPlan& p) {
    const float border = 4.f * size, full_h = 8.f * size + 1.f;
    const float roi_w_f = fminf((float)n_pool + full_h, img_width_f - u_tl);
    const int rx = (int)u_tl, ry = (int)v_tl, rw = (int)roi_w_f, rh = (int)full_h;  // cv::Rect(float...) truncates
    p.border = border; p.u_tl = u_tl; p.v_tl = v_tl; p.first = first;
    p.n_valid = 0; p.i_lo = 0; p.gx_lo = 0; p.gy = 0;
    if (rx < 0 || ry < 0 || rw < 0 || rh < 0 || rx + rw > W || ry + rh > H) { p.status = SVI_TRI_BAD_ROI; return; }
    // KeyPointsFilter::runByImageBorder inside the ROI: keep 28 <= cvRound(pt) < size - 28
    // (a key-point whose sampling centre (int)(pt+0.5) falls outside the same range is erased too: for x.5
    //  coordinates the two roundings differ and the reference would read outside its integral image)
    const int ky_r = cv_round_f(border), ky_c = brief_centre(border);
    int i_lo = 0, i_hi = 0;
    const bool row_ok = ky_r >= kBriefBorder && ky_r < rh - kBriefBorder && ky_c >= kBriefBorder && ky_c < rh - kBriefBorder;
    if (row_ok && border == (float)ky_r && n_pool < (1 << 22)) {
        // integral border (every key-point size the reference produces): pool x = ky_r + first + i exactly, both
        // roundings coincide, and the survivors are the i with 28 <= x < rw - 28
        const int x0 = ky_r + first;
        i_lo = min(max(kBriefBorder - x0, 0), n_pool);
        i_hi = min(max(rw - kBriefBorder - x0, 0), n_pool);
    } else if (row_ok) {
        for (int i0 = 0; i0 < n_pool; i0 += 32) {
            int i = i0 + lane;
            const float kx = (border + (float)i) + (float)first;
            const int kr = cv_round_f(kx), kc = brief_centre(kx);
            bool in = i < n_pool;
            i_lo += __popc(__ballot_sync(0xFFFFFFFFu, in && (kr < kBriefBorder || kc < kBriefBorder)));
            i_hi += __popc(__ballot_sync(0xFFFFFFFFu, in && kr < rw - kBriefBorder && kc < rw - kBriefBorder));
        }
    }
    p.n_valid = i_hi - i_lo;
    p.i_lo = i_lo;
    if (p.n_valid <= 0) { p.status = SVI_TRI_NO_DESC; return; }
    const float kx_lo = (border + (float)i_lo) + (float)first;
    p.gx_lo = rx + brief_centre(kx_lo);
    p.gy = ry + brief_centre(border);
    p.status = SVI_OK;
}

// Window of the pass that starts at candidate `cb`: its left image column, rounded down to the TMA
// alignment.  The remainder splits into an even word offset and a parity that shifts the slots.
__device__ __forceinline__ int window_col(const SearchPlan& p, int cb) { return p.gx_lo + cb - kBriefReach; }
__device__ __forceinline__ int window_col_aligned(int col) { return (col >> 3) << 3; }

// Start staging the first window of a planned search.
__device__ __forceinline__ void search_prefetch(const SearchPlan& p, const PatchStage& ps, int lane) {
    if (p.status == SVI_OK) patch_issue(ps, p.gy - kBriefReach, window_col_aligned(window_col(p, 0)), lane);
}

// Descriptors of the surviving candidates, first arg-min against `ref`, cut-off (the first window must
// already be in flight: search_prefetch).
__device__ __forceinline__ void search_run(const SearchPlan& p, PatchStage& ps, const uint32_t (&ref)[kDescWords],
                                           float cutoff, int lane, SearchResult& out) {
    out.dist = -1;
    out.idx = -1;
    out.status = p.status;
    if (p.status != SVI_OK) return;
    uint32_t best_key = 0xFFFFFFFFu;
    for (int cb = 0; cb < p.n_valid; cb += PATCH_CHUNK) {
        const int col = window_col(p, cb), col_a = window_col_aligned(col);
        const int par = (col - col_a) & 1;             // slot s evaluates candidate cb + s - par
        const int woff = (col - col_a) >> 1;           // even part of the remainder, in 32-bit words
        if (cb > 0) {
            __syncwarp();
            patch_issue(ps, p.gy - kBriefReach, col_a, lane);
        }
        patch_wait(ps);
        // the farthest word any test reads: row 48, word (48 >> 1) of a lane's pair -> woff + lane + 48 * PATCH_WORDS + 24
        SVI_CHECK(3, woff >= 0 && woff + 31 + 2 * kBriefReach * PATCH_WORDS + kBriefReach < PATCH_COPY_WORDS);
        const uint32_t* Al = ps.words + woff + lane;
        const uint32_t* Bl = ps.words + PATCH_COPY_WORDS + woff + lane;
        uint32_t wlo[kDescWords], whi[kDescWords];
        brief_pair_all(Al, Bl, wlo, whi, std::make_integer_sequence<int, kDescWords>{});
        const int l_lo = 2 * lane - par, l_hi = l_lo + 1;   // candidate index within this pass
        const int c_lo = cb + l_lo, c_hi = cb + l_hi;
        uint32_t k_lo = (l_lo >= 0 && l_lo < PATCH_CHUNK && c_lo < p.n_valid) ? (((uint32_t)hamming_words(wlo, ref) << 16) | (uint32_t)(c_lo & 0xFFFF)) : 0xFFFFFFFFu;
        uint32_t k_hi = (l_hi < PATCH_CHUNK && c_hi < p.n_valid) ? (((uint32_t)hamming_words(whi, ref) << 16) | (uint32_t)(c_hi & 0xFFFF)) : 0xFFFFFFFFu;
        const uint32_t k_mine = min(k_lo, k_hi);
        const uint32_t k_min = warp_min_u32(k_mine);
        if (k_min < best_key) {  // strict: earlier chunks win ties (BFMatcher keeps the first minimum)
            best_key = k_min;
            const int owner = __ffs(__ballot_sync(0xFFFFFFFFu, k_mine == k_min)) - 1;
            const bool hi = (k_hi == k_min) && (k_lo != k_min);
#pragma unroll
            for (int j = 0; j < kDescWords; ++j) out.w[j] = __shfl_sync(0xFFFFFFFFu, hi ? whi[j] : wlo[j], owner);
        }
    }
    // the key carries the candidate index in 16 bits (n_valid < 65536: image widths are 16-bit)
    out.dist = (int)(best_key >> 16);
    out.idx = (int)(best_key & 0xFFFFu);
    if (!(cutoff > (float)out.dist)) { out.status = SVI_TRI_DISTANCE; return; }
    const float px = (p.border + (float)(p.i_lo + out.idx)) + (float)p.first;
    out.u = px + p.u_tl;
    out.v = p.border + p.v_tl;
    out.status = SVI_OK;
}

// CTriangulator::getPointInLEFT :326-356, fp64, evaluation order of the reference, no FMA.
__device__ __forceinline__ int point_in_left(const TriConst& tc, float xl, float yl, float xr, double* xyz) {
    const float d = __fsub_rn(xl, xr);
    if ((double)d < tc.min_disp) return SVI_TRI_ZERO_DISP;
    const double z = __ddiv_rn(tc.du_r_flipped, (double)d);
    const double fz = __dmul_rn(tc.f_inv, z);
    xyz[0] = __dmul_rn(fz, __dsub_rn((double)xl, tc.pu));
    xyz[1] = __dmul_rn(fz, __dsub_rn((double)yl, tc.pv));
    xyz[2] = z;
    return SVI_OK;
}

// getPointTriangulatedInRIGHT: range check + pool size (:63-67), then the shared plan.
__device__ __forceinline__ void plan_right(const FrameGeom& g, const TriConst& tc, float u_tl, float v_tl, float size,
                                           float xl, int lane, SearchPlan& p) {
    const float border = 4.f * size;
    if (xl <= u_tl + border) { p.status = SVI_TRI_RANGE; p.n_valid = 0; return; }
    const int n_pool = (int)ceilf((xl - u_tl) - border);
    search_plan(g.W, g.H, tc.width_right, u_tl, v_tl, size, 0, n_pool, lane, p);
}

// getPointTriangulatedInLEFT (7 args): :268-272, then the shared plan.
__device__ __forceinline__ void plan_left(const FrameGeom& g, const TriConst& tc, float search_range, float u_tl,
                                          float v_tl, float size, int lane, SearchPlan& p) {
    if (0.f >= search_range) { p.status = SVI_TRI_RANGE; p.n_valid = 0; return; }
    const int n_pool = (int)ceilf(fminf(search_range, tc.width_left - u_tl)) + 1;
    search_plan(g.W, g.H, tc.width_left, u_tl, v_tl, size, 1, n_pool, lane, p);
}

// Whole searches (plan, stage, evaluate, triangulate) for the callers that have nothing to overlap.
__device__ __forceinline__ void triangulate_right_dev(const FrameGeom& g, const TriConst& tc, PatchStage& ps, float u_tl,
                                                      float v_tl, float size, float xl, float yl,
                                                      const uint32_t (&ref)[kDescWords], int lane, SearchResult& r,
                                                      double* xyz) {
    SearchPlan p;
    plan_right(g, tc, u_tl, v_tl, size, xl, lane, p);
    search_prefetch(p, ps, lane);
    search_run(p, ps, ref, tc.match_cutoff, lane, r);
    if (r.status == SVI_OK) r.status = point_in_left(tc, xl, yl, r.u, xyz);
}

__device__ __forceinline__ void triangulate_left_dev(const FrameGeom& g, const TriConst& tc, PatchStage& ps,
                                                     float search_range, float u_tl, float v_tl, float size, float xr,
                                                     const uint32_t (&ref)[kDescWords], int lane, SearchResult& r,
                                                     double* xyz) {
    SearchPlan p;
    plan_left(g, tc, search_range, u_tl, v_tl, size, lane, p);
    search_prefetch(p, ps, lane);
    search_run(p, ps, ref, tc.match_cutoff, lane, r);
    if (r.status == SVI_OK) r.status = point_in_left(tc, r.u, r.v, xr, xyz);
}

// Carve the warp's staging buffers and barrier out of the CTA's dynamic shared memory.
__device__ __forceinline__ void patch_stage_init(PatchStage& ps, unsigned char* smem, const CUtensorMap* map,
                                                 const CUtensorMap* map_s, int row_base, int warp, int lane) {
    unsigned char* mine = smem + (size_t)warp * MATCH_SMEM_PER_WARP;
    ps.map = map;
    ps.map_s = map_s;
    ps.row_base = row_base;
    ps.smem_a = smem_u32(mine);
    ps.words = reinterpret_cast<const uint32_t*>(mine);
    ps.bar = smem_u32(smem + (size_t)MATCH_WARPS * MATCH_SMEM_PER_WARP + warp * 8);
    ps.phase = 0u;
    if (lane == 0) {
        mbar_init(ps.bar, 1);
        fence_barrier_init();
    }
    __syncwarp();
}

struct StereoOutDev {
    int cap;
    float* uv_l; float* uv_r; double* xyz; uint8_t* desc_l; uint8_t* desc_r;
    int* dist; int* idx; uint8_t* status;
};

// Raw box-sum gathers of one descriptor (lanes = tests): issued early, turned into bits later, so the
// global-memory round trip hides under other work.
struct BriefGather {
    uint16_t s1[kDescWords], s2[kDescWords];
};
// The element offsets of this lane's 8 test pairs inside a box-sum plane: the same for every key-point of a
// frame, so a warp computes them once.
struct BriefOffsets {
    int o1[kDescWords], o2[kDescWords];
};
__device__ __forceinline__ void brief_offsets_init(BriefOffsets& bo, int box_pitch, int lane) {
#pragma unroll
    for (int j = 0; j < kDescWords; ++j) {
        const char4 p = brief_pattern(32 * j + lane);
        bo.o1[j] = p.x * box_pitch + p.y;
        bo.o2[j] = p.z * box_pitch + p.w;
    }
}
__device__ __forceinline__ void brief_gather_issue(const uint16_t* __restrict__ box, int box_pitch, int cx, int cy,
                                                   const BriefOffsets& bo, BriefGather& gth) {
    const uint16_t* c = box + cy * box_pitch + cx;
#pragma unroll
    for (int j = 0; j < kDescWords; ++j) {
        gth.s1[j] = __ldg(c + bo.o1[j]);
        gth.s2[j] = __ldg(c + bo.o2[j]);
    }
}
__device__ __forceinline__ void brief_gather_issue(const uint16_t* __restrict__ box, int box_pitch, int cx, int cy,
                                                   int lane, BriefGather& gth) {
#pragma unroll
    for (int j = 0; j < kDescWords; ++j) {
        const char4 p = brief_pattern(32 * j + lane);
        gth.s1[j] = __ldg(box + (cy + p.x) * box_pitch + cx + p.y);
        gth.s2[j] = __ldg(box + (cy + p.z) * box_pitch + cx + p.w);
    }
}
__device__ __forceinline__ void brief_gather_finish(const BriefGather& gth, uint32_t (&w)[kDescWords]) {
#pragma unroll
    for (int j = 0; j < kDescWords; ++j) w[j] = __brev(__ballot_sync(0xFFFFFFFFu, gth.s1[j] < gth.s2[j]));
}

// K5: per key-point of addNewLandmarks (:109-175): LEFT descriptor, scan-line search in RIGHT
// with uTL = max(0, x - range - 4*size), vTL = y - 4*size (:120-121), triangulation, outputs.
// A warp walks MATCH_KP_PER_WARP consecutive key-points as a three-stage software pipeline:
//   stage A  key-point coordinates of slot i+2                      (one 4-byte load)
//   stage B  search plan, LEFT descriptor gathers of slot i+1       (16 loads per lane in flight)
//   stage C  tests / arg-min / triangulation of slot i from the shared window; the TMA for slot i+1
//            is issued as soon as the last lane has finished reading the window
// so every global round trip overlaps the ~1500 shared-memory/ALU instructions of stage C.
constexpr int MATCH_KP_PER_WARP = 8;   // for full batches; small calls spread their key-points over more warps (latency)
__global__ void __launch_bounds__(MATCH_WARPS * 32, 3)
stereo_match_kernel(const uint16_t* __restrict__ box_l, const __grid_constant__ CUtensorMap map_r,
                    const __grid_constant__ CUtensorMap map_rs, FrameGeom g, TriConst tc, float size, float range,
                    const ushort2* __restrict__ kp_xy, const int* __restrict__ n_kp, int max_corners, StereoOutDev out,
                    int out_frame0, int kp_per_warp) {
    extern __shared__ __align__(128) unsigned char match_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int f = blockIdx.y, slot0 = (blockIdx.x * MATCH_WARPS + warp) * kp_per_warp;
    const int n = n_kp[f];
    if (slot0 >= n) return;
    const int slot_end = min(slot0 + kp_per_warp, n);
    PatchStage ps;
    patch_stage_init(ps, match_smem, &map_r, &map_rs, f * g.H, warp, lane);
    const ushort2* kps = kp_xy + (size_t)f * max_corners;
    const uint16_t* bl = box_l + (size_t)f * g.H * g.box_pitch;

    // prologue: slot0 through stages A and B, slot0+1 through stage A
    ushort2 kp_b = kps[slot0];
    ushort2 kp_a = (slot0 + 1 < slot_end) ? kps[slot0 + 1] : kp_b;
    SearchPlan plan_b;
    BriefGather gth_b;
    BriefOffsets bo;
    brief_offsets_init(bo, g.box_pitch, lane);
    {
        const float x = (float)kp_b.x, y = (float)kp_b.y;
        plan_right(g, tc, fmaxf(0.f, (x - range) - 4.f * size), y - 4.f * size, size, x, lane, plan_b);
        search_prefetch(plan_b, ps, lane);
        brief_gather_issue(bl, g.box_pitch, kp_b.x, kp_b.y, bo, gth_b);
    }
    for (int slot = slot0; slot < slot_end; ++slot) {
        // ---- this slot enters stage C
        const ushort2 kp = kp_b;
        const SearchPlan plan = plan_b;
        uint32_t ref[kDescWords];
        brief_gather_finish(gth_b, ref);
        // ---- next slot enters stage B, the one after it stage A
        const bool has_next = slot + 1 < slot_end;
        if (has_next) {
            kp_b = kp_a;
            const float xn = (float)kp_b.x, yn = (float)kp_b.y;
            plan_right(g, tc, fmaxf(0.f, (xn - range) - 4.f * size), yn - 4.f * size, size, xn, lane, plan_b);
            brief_gather_issue(bl, g.box_pitch, kp_b.x, kp_b.y, bo, gth_b);
            if (slot + 2 < slot_end) kp_a = kps[slot + 2];
        }
        // ---- stage C
        const float x = (float)kp.x, y = (float)kp.y;
        SearchResult r;
        double xyz[3] = {0.0, 0.0, 0.0};
        search_run(plan, ps, ref, tc.match_cutoff, lane, r);
        if (has_next) {
            __syncwarp();                          // every lane is done reading this slot's window
            search_prefetch(plan_b, ps, lane);     // next window in flight under the epilogue below
        }
        if (r.status == SVI_OK) r.status = point_in_left(tc, x, y, r.u, xyz);
        SVI_CHECK(3, slot < out.cap && slot < max_corners);
        const size_t o = (size_t)(out_frame0 + f) * out.cap + slot;
        store_desc(out.desc_l + o * 32, ref, lane);
        if (r.status == SVI_OK) store_desc(out.desc_r + o * 32, r.w, lane);
        if (lane == 0) {
            out.uv_l[o * 2] = x; out.uv_l[o * 2 + 1] = y;
            out.status[o] = (uint8_t)r.status;
            out.dist[o] = r.dist;
            out.idx[o] = r.idx;
            if (r.status == SVI_OK) {
                out.uv_r[o * 2] = r.u; out.uv_r[o * 2 + 1] = r.v;
                out.xyz[o * 3] = xyz[0]; out.xyz[o * 3 + 1] = xyz[1]; out.xyz[o * 3 + 2] = xyz[2];
            }
        }
    }
}

// ------------------------------------------------------------------ the same search, G warps per key-point
// stereo_match_kernel runs 9 warps per SM (the windows fill the shared memory) and ncu shows those warps waiting on
// their own LDS -> HSET2 -> LOP3 chains.  Here the G warps of a GROUP share one window and one mbarrier and each of them
// evaluates kDescWords / G of the eight descriptor words (its share of the LDS / compares / popc); the partial Hamming
// distances of the 64 candidate slots cross a 2 x G x 32-word exchange buffer once per pass, after which every warp of
// the group holds the complete distances, finds the same arg-min and writes its own words of both descriptors.
// Same shared memory per key-point, G times the warps per SM, the instruction count per key-point unchanged apart from
// one named barrier per pass.
template <int G>
struct MatchSplit {
    static constexpr int WORDS = kDescWords / G;                       // descriptor words per warp
    static constexpr int THREADS = MATCH_WARPS * G * 32;               // MATCH_WARPS groups per CTA
    static constexpr int BAR_OFF = MATCH_WARPS * MATCH_SMEM_PER_WARP;  // one mbarrier per group
    static constexpr int XCH_OFF = BAR_OFF + 32;                       // exchange: [group][parity][warp of group][lane]
    static constexpr int SMEM = XCH_OFF + MATCH_WARPS * 2 * G * 32 * 4;
    static_assert(kDescWords % G == 0 && MATCH_WARPS * 8 <= 32, "group layout");
};

__device__ __forceinline__ void group_barrier(int grp, int threads) {
    asm volatile("bar.sync %0, %1;" ::"r"(1 + grp), "r"(threads) : "memory");
}

template <int BASE, int N, int... J>
__device__ __forceinline__ void brief_pair_range(const uint32_t* __restrict__ Al, const uint32_t* __restrict__ Bl,
                                                 uint32_t (&wlo)[N], uint32_t (&whi)[N], std::integer_sequence<int, J...>) {
    (brief_pair_word<BASE + J>(Al, Bl, wlo[J], whi[J]), ...);
}
// words [sub * N, (sub + 1) * N) for a warp-uniform run-time `sub`: one unrolled body per value
template <int G, int S = 0>
__device__ __forceinline__ void brief_pair_sub(int sub, const uint32_t* __restrict__ Al, const uint32_t* __restrict__ Bl,
                                               uint32_t (&wlo)[kDescWords / G], uint32_t (&whi)[kDescWords / G]) {
    if constexpr (S < G) {
        if (sub == S) brief_pair_range<S * (kDescWords / G)>(Al, Bl, wlo, whi, std::make_integer_sequence<int, kDescWords / G>{});
        else brief_pair_sub<G, S + 1>(sub, Al, Bl, wlo, whi);
    }
}

template <int N>
__device__ __forceinline__ void store_desc_part(uint8_t* dst, const uint32_t (&w)[N], int first_word, int lane) {
    uint32_t v = 0;
#pragma unroll
    for (int j = 0; j < N; ++j) if (lane == j) v = w[j];
    if (lane < N) reinterpret_cast<uint32_t*>(dst)[first_word + lane] = desc_word_to_bytes(v);
}

template <int N>
__device__ __forceinline__ void gather_part(const uint16_t* __restrict__ c, const int (&o1)[N], const int (&o2)[N],
                                            uint16_t (&s1)[N], uint16_t (&s2)[N]) {
#pragma unroll
    for (int j = 0; j < N; ++j) { s1[j] = __ldg(c + o1[j]); s2[j] = __ldg(c + o2[j]); }
}

template <int N>
struct SplitResult {
    int status, dist, idx;
    float u, v;
    uint32_t w[N];   // this warp's words of the best candidate's descriptor
};

template <int G>
__device__ __forceinline__ void search_run_split(const SearchPlan& p, PatchStage& ps, const uint32_t (&ref)[kDescWords / G],
                                                 float cutoff, int lane, int grp, int sub, uint32_t* __restrict__ xch,
                                                 uint32_t& xpar, SplitResult<kDescWords / G>& out) {
    constexpr int N = kDescWords / G;
    out.dist = -1;
    out.idx = -1;
    out.status = p.status;
    if (p.status != SVI_OK) return;
    uint32_t best_key = 0xFFFFFFFFu;
    for (int cb = 0; cb < p.n_valid; cb += PATCH_CHUNK) {
        const int col = window_col(p, cb), col_a = window_col_aligned(col);
        const int par = (col - col_a) & 1, woff = (col - col_a) >> 1;
        patch_wait(ps);
        SVI_CHECK(3, woff >= 0 && woff + 31 + 2 * kBriefReach * PATCH_WORDS + kBriefReach < PATCH_COPY_WORDS);
        const uint32_t* Al = ps.words + woff + lane;
        const uint32_t* Bl = ps.words + PATCH_COPY_WORDS + woff + lane;
        uint32_t wlo[N], whi[N];
        brief_pair_sub<G>(sub, Al, Bl, wlo, whi);
        int d_lo = 0, d_hi = 0;
#pragma unroll
        for (int j = 0; j < N; ++j) { d_lo += __popc(wlo[j] ^ ref[j]); d_hi += __popc(whi[j] ^ ref[j]); }
        uint32_t* x = xch + xpar * (G * 32);
        xpar ^= 1u;
        x[sub * 32 + lane] = (uint32_t)d_lo | ((uint32_t)d_hi << 16);
        group_barrier(grp, G * 32);   // partial distances visible; every warp of the group is done with the window
        const int cb_next = cb + PATCH_CHUNK;
        if (sub == 0 && cb_next < p.n_valid)
            patch_issue(ps, p.gy - kBriefReach, window_col_aligned(window_col(p, cb_next)), lane);
        uint32_t dsum = 0;
#pragma unroll
        for (int s = 0; s < G; ++s) dsum += x[s * 32 + lane];   // two 16-bit sums, each <= 256
        const int l_lo = 2 * lane - par, l_hi = l_lo + 1;
        const int c_lo = cb + l_lo, c_hi = cb + l_hi;
        const uint32_t k_lo = (l_lo >= 0 && l_lo < PATCH_CHUNK && c_lo < p.n_valid) ? (((dsum & 0xFFFFu) << 16) | (uint32_t)(c_lo & 0xFFFF)) : 0xFFFFFFFFu;
        const uint32_t k_hi = (l_hi < PATCH_CHUNK && c_hi < p.n_valid) ? ((dsum & 0xFFFF0000u) | (uint32_t)(c_hi & 0xFFFF)) : 0xFFFFFFFFu;
        const uint32_t k_mine = min(k_lo, k_hi);
        const uint32_t k_min = warp_min_u32(k_mine);
        if (k_min < best_key) {
            best_key = k_min;
            const int owner = __ffs(__ballot_sync(0xFFFFFFFFu, k_mine == k_min)) - 1;
            const bool hi = (k_hi == k_min) && (k_lo != k_min);
#pragma unroll
            for (int j = 0; j < N; ++j) out.w[j] = __shfl_sync(0xFFFFFFFFu, hi ? whi[j] : wlo[j], owner);
        }
    }
    out.dist = (int)(best_key >> 16);
    out.idx = (int)(best_key & 0xFFFFu);
    if (!(cutoff > (float)out.dist)) { out.status = SVI_TRI_DISTANCE; return; }
    const float px = (p.border + (float)(p.i_lo + out.idx)) + (float)p.first;
    out.u = px + p.u_tl;
    out.v = p.border + p.v_tl;
    out.status = SVI_OK;
}

// ------------------------------------------------------------------ LEFT descriptors of a chunk, ahead of the matcher
// In stereo_match_kernel the 512 box-sum gathers of a LEFT descriptor are 16 scattered LDG per lane: ncu counts 203
// wavefronts of the L1 data pipe per key-point for them (every LDG touches ~27 sectors of ~27 lines), one third of what
// the 256 tests of all 60 candidates cost, in a kernel whose binding unit is that pipe.  Here one TMA tile brings the
// 49 x 56 patch around the key-point into shared memory (not an LSU wavefront), the same 16 reads per lane become
// LDS.U16 with ordinary bank conflicts (~3 wavefronts each), and the matcher gets the descriptor as one 16-byte load.
constexpr int DL_COLS = 2 * kBriefReach + 8;                       // 56: the patch start is rounded down to 8 elements
constexpr int DL_BYTES = PATCH_ROWS * DL_COLS * 2;                 // 5488: one TMA box
constexpr int DL_STRIDE = (DL_BYTES + 127) / 128 * 128;
constexpr int DL_WARPS = 8;
constexpr int DL_KP_PER_WARP = 8;
constexpr int DL_SMEM = DL_WARPS * 2 * DL_STRIDE + DL_WARPS * 2 * 8;   // two patches and two mbarriers per warp

__global__ void __launch_bounds__(DL_WARPS * 32)
describe_left_kernel(const __grid_constant__ CUtensorMap map_l, FrameGeom g, const ushort2* __restrict__ kp_xy,
                     const int* __restrict__ n_kp, int max_corners, uint8_t* __restrict__ desc_l, int cap, int out_frame0) {
    extern __shared__ __align__(128) unsigned char dl_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int f = blockIdx.y, slot0 = (blockIdx.x * DL_WARPS + warp) * DL_KP_PER_WARP;
    const int n = n_kp[f];
    if (slot0 >= n) return;
    const int slot_end = min(slot0 + DL_KP_PER_WARP, n);
    unsigned char* mine = dl_smem + (size_t)warp * 2 * DL_STRIDE;
    const uint32_t buf0 = smem_u32(mine), bar0 = smem_u32(dl_smem + (size_t)DL_WARPS * 2 * DL_STRIDE + warp * 16);
    if (lane == 0) {
        mbar_init(bar0, 1);
        mbar_init(bar0 + 8, 1);
        fence_barrier_init();
    }
    __syncwarp();
    int o1[kDescWords], o2[kDescWords];   // this lane's test points as element offsets inside a patch whose column 0 is x - 24
#pragma unroll
    for (int j = 0; j < kDescWords; ++j) {
        const char4 pt = brief_pattern(32 * j + lane);
        o1[j] = (pt.x + kBriefReach) * DL_COLS + pt.y + kBriefReach;
        o2[j] = (pt.z + kBriefReach) * DL_COLS + pt.w + kBriefReach;
    }
    const ushort2* kps = kp_xy + (size_t)f * max_corners;
    const int row_base = f * g.H;
    auto issue = [&](ushort2 kp, int b) {
        if (lane == 0) {
            fence_proxy_async();
            mbar_expect_tx(bar0 + 8 * b, DL_BYTES);
            tma_load_2d(buf0 + b * DL_STRIDE, &map_l, ((kp.x - kBriefReach) >> 3) << 3, row_base + kp.y - kBriefReach, bar0 + 8 * b);
        }
    };
    ushort2 kp = kps[slot0];
    issue(kp, 0);
    uint32_t phase = 0u;   // bit b = parity of the next completion of buffer b
    for (int slot = slot0; slot < slot_end; ++slot) {
        const int b = (slot - slot0) & 1;
        ushort2 kp_next = kp;
        if (slot + 1 < slot_end) {
            kp_next = kps[slot + 1];
            issue(kp_next, b ^ 1);   // that buffer was read two slots ago; the __syncwarp below ordered those reads
        }
        mbar_wait(bar0 + 8 * b, (phase >> b) & 1u);
        phase ^= 1u << b;
        const uint16_t* patch = reinterpret_cast<const uint16_t*>(mine + b * DL_STRIDE) + ((kp.x - kBriefReach) & 7);
        uint32_t w[kDescWords];
#pragma unroll
        for (int j = 0; j < kDescWords; ++j) w[j] = __brev(__ballot_sync(0xFFFFFFFFu, patch[o1[j]] < patch[o2[j]]));
        SVI_CHECK(6, slot < cap && slot < max_corners);
        store_desc(desc_l + ((size_t)(out_frame0 + f) * cap + slot) * 32, w, lane);
        __syncwarp();
        kp = kp_next;
    }
}

// K5 with G warps per key-point: the software pipeline of stereo_match_kernel, per group.  PRE: the LEFT descriptors
// are already in out.desc_l (describe_left_kernel) and arrive as one load per warp instead of 2 * WORDS gathers per lane.
template <int G, bool PRE>
__global__ void __launch_bounds__(MatchSplit<G>::THREADS, 3)
stereo_match_split_kernel(const uint16_t* __restrict__ box_l, const __grid_constant__ CUtensorMap map_r,
                          const __grid_constant__ CUtensorMap map_rs, FrameGeom g, TriConst tc, float size, float range,
                          const ushort2* __restrict__ kp_xy, const int* __restrict__ n_kp, int max_corners, StereoOutDev out,
                          int out_frame0, int kp_per_group) {
    using MS = MatchSplit<G>;
    constexpr int N = MS::WORDS;
    extern __shared__ __align__(128) unsigned char match_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int grp = warp / G, sub = warp % G;
    const int f = blockIdx.y, slot0 = (blockIdx.x * MATCH_WARPS + grp) * kp_per_group;
    const int n = n_kp[f];
    if (slot0 >= n) return;   // whole groups leave together
    const int slot_end = min(slot0 + kp_per_group, n);
    PatchStage ps;
    {
        unsigned char* mine = match_smem + (size_t)grp * MATCH_SMEM_PER_WARP;
        ps.map = &map_r;
        ps.map_s = &map_rs;
        ps.row_base = f * g.H;
        ps.smem_a = smem_u32(mine);
        ps.words = reinterpret_cast<const uint32_t*>(mine);
        ps.bar = smem_u32(match_smem + MS::BAR_OFF + grp * 8);
        ps.phase = 0u;
        if (sub == 0 && lane == 0) {
            mbar_init(ps.bar, 1);
            fence_barrier_init();
        }
        group_barrier(grp, G * 32);
    }
    uint32_t* xch = reinterpret_cast<uint32_t*>(match_smem + MS::XCH_OFF) + grp * (2 * G * 32);
    uint32_t xpar = 0u;
    const ushort2* kps = kp_xy + (size_t)f * max_corners;
    const uint16_t* bl = box_l + (size_t)f * g.H * g.box_pitch;

    int o1[N], o2[N];   // this lane's test pairs of this warp's words, as element offsets in a box-sum plane
    if constexpr (!PRE) {
#pragma unroll
        for (int j = 0; j < N; ++j) {
            const char4 pt = brief_pattern(32 * (sub * N + j) + lane);
            o1[j] = pt.x * g.box_pitch + pt.y;
            o2[j] = pt.z * g.box_pitch + pt.w;
        }
    }
    uint16_t s1[N], s2[N];
    uint32_t ref_raw[N];   // PRE: this warp's words of the stored descriptor (byte order of the output)
    const uint32_t* dl = reinterpret_cast<const uint32_t*>(out.desc_l) + ((size_t)(out_frame0 + f) * out.cap) * kDescWords + sub * N;

    ushort2 kp_b = kps[slot0];
    ushort2 kp_a = (slot0 + 1 < slot_end) ? kps[slot0 + 1] : kp_b;
    SearchPlan plan_b;
    {
        const float x = (float)kp_b.x, y = (float)kp_b.y;
        plan_right(g, tc, fmaxf(0.f, (x - range) - 4.f * size), y - 4.f * size, size, x, lane, plan_b);
        if (sub == 0) search_prefetch(plan_b, ps, lane);
        if constexpr (PRE) {
#pragma unroll
            for (int j = 0; j < N; ++j) ref_raw[j] = __ldg(dl + (size_t)slot0 * kDescWords + j);
        } else {
            gather_part<N>(bl + kp_b.y * g.box_pitch + kp_b.x, o1, o2, s1, s2);
        }
    }
    for (int slot = slot0; slot < slot_end; ++slot) {
        const ushort2 kp = kp_b;
        const SearchPlan plan = plan_b;
        uint32_t ref[N];
#pragma unroll
        for (int j = 0; j < N; ++j) ref[j] = PRE ? desc_word_to_bytes(ref_raw[j]) : __brev(__ballot_sync(0xFFFFFFFFu, s1[j] < s2[j]));
        const bool has_next = slot + 1 < slot_end;
        if (has_next) {
            kp_b = kp_a;
            const float xn = (float)kp_b.x, yn = (float)kp_b.y;
            plan_right(g, tc, fmaxf(0.f, (xn - range) - 4.f * size), yn - 4.f * size, size, xn, lane, plan_b);
            if constexpr (PRE) {
#pragma unroll
                for (int j = 0; j < N; ++j) ref_raw[j] = __ldg(dl + (size_t)(slot + 1) * kDescWords + j);
            } else {
                gather_part<N>(bl + kp_b.y * g.box_pitch + kp_b.x, o1, o2, s1, s2);
            }
            if (slot + 2 < slot_end) kp_a = kps[slot + 2];
        }
        const float x = (float)kp.x, y = (float)kp.y;
        SplitResult<N> r;
        double xyz[3] = {0.0, 0.0, 0.0};
        search_run_split<G>(plan, ps, ref, tc.match_cutoff, lane, grp, sub, xch, xpar, r);
        if (has_next) {
            // a search that ran at least one pass ended on a group barrier after the last window read; one that was
            // never staged (status != OK) left the window untouched
            if (sub == 0) search_prefetch(plan_b, ps, lane);
        }
        SVI_CHECK(3, slot < out.cap && slot < max_corners);
        const size_t o = (size_t)(out_frame0 + f) * out.cap + slot;
        if constexpr (!PRE) store_desc_part(out.desc_l + o * 32, ref, sub * N, lane);
        if (r.status == SVI_OK) r.status = point_in_left(tc, x, y, r.u, xyz);   // every warp: the verdict gates its desc_r words
        if (r.status == SVI_OK) store_desc_part(out.desc_r + o * 32, r.w, sub * N, lane);
        if (sub == 0 && lane == 0) {
            out.uv_l[o * 2] = x; out.uv_l[o * 2 + 1] = y;
            out.status[o] = (uint8_t)r.status;
            out.dist[o] = r.dist;
            out.idx[o] = r.idx;
            if (r.status == SVI_OK) {
                out.uv_r[o * 2] = r.u; out.uv_r[o * 2 + 1] = r.v;
                out.xyz[o * 3] = xyz[0]; out.xyz[o * 3 + 1] = xyz[1]; out.xyz[o * 3 + 2] = xyz[2];
            }
        }
    }
}

// svi_describe: BRIEF-32 at n points of one image (full-image border filter).
__global__ void describe_kernel(const uint16_t* __restrict__ box, FrameGeom g, const float* __restrict__ xy, int n,
                                uint8_t* __restrict__ desc, uint8_t* __restrict__ kept) {
    const int lane = threadIdx.x & 31, q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (q >= n) return;
    const float x = xy[2 * q], y = xy[2 * q + 1];
    const int rx = cv_round_f(x), ry = cv_round_f(y), sx = brief_centre(x), sy = brief_centre(y);
    const bool ok = rx >= kBriefBorder && rx < g.W - kBriefBorder && ry >= kBriefBorder && ry < g.H - kBriefBorder &&
                    sx >= kBriefBorder && sx < g.W - kBriefBorder && sy >= kBriefBorder && sy < g.H - kBriefBorder;
    uint32_t w[kDescWords] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (ok) brief_at_point(box, g.box_pitch, brief_centre(x), brief_centre(y), lane, w);
    store_desc(desc + (size_t)q * 32, w, lane);
    if (lane == 0) kept[q] = ok ? 1 : 0;
}

// svi_match_hamming: BFMatcher(NORM_HAMMING).match, one warp per query row.
__global__ void hamming_match_kernel(const uint8_t* __restrict__ q32, int nq, const uint8_t* __restrict__ t32, int nt,
                                     int* __restrict__ index, int* __restrict__ distance) {
    const int lane = threadIdx.x & 31, q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (q >= nq) return;
    uint32_t ref[kDescWords];
    load_desc(q32 + (size_t)q * 32, ref);
    unsigned long long best = ~0ull;
    for (int t = lane; t < nt; t += 32) {
        uint32_t w[kDescWords];
        load_desc(t32 + (size_t)t * 32, w);
        unsigned long long k = ((unsigned long long)hamming_words(ref, w) << 32) | (unsigned)t;
        best = min(best, k);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = min(best, __shfl_xor_sync(0xFFFFFFFFu, best, o));
    if (lane == 0) {
        index[q] = nt > 0 ? (int)(best & 0xFFFFFFFFu) : -1;
        distance[q] = nt > 0 ? (int)(best >> 32) : -1;
    }
}

struct TriOutDev {
    float* uv; double* xyz; uint8_t* desc; int* dist; int* idx; uint8_t* status;
};

// svi_triangulate_right / svi_triangulate_left: one warp per query against one image.
template <bool kLeft>
__global__ void __launch_bounds__(MATCH_WARPS * 32, 3)
triangulate_kernel(const __grid_constant__ CUtensorMap map, const __grid_constant__ CUtensorMap map_s, FrameGeom g,
                   TriConst tc, int n,
                   const float* __restrict__ search_range, const float* __restrict__ top_left,
                   const float* __restrict__ uv_ref, const uint8_t* __restrict__ desc_ref, float size, TriOutDev out) {
    extern __shared__ __align__(128) unsigned char match_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = blockIdx.x * MATCH_WARPS + warp;
    if (q >= n) return;
    PatchStage ps;
    patch_stage_init(ps, match_smem, &map, &map_s, 0, warp, lane);
    uint32_t ref[kDescWords];
    load_desc(desc_ref + (size_t)q * 32, ref);
    SearchResult r;
    double xyz[3] = {0.0, 0.0, 0.0};
    const float u_tl = top_left[2 * q], v_tl = top_left[2 * q + 1], xq = uv_ref[2 * q], yq = uv_ref[2 * q + 1];
    if (kLeft) triangulate_left_dev(g, tc, ps, search_range[q], u_tl, v_tl, size, xq, ref, lane, r, xyz);
    else triangulate_right_dev(g, tc, ps, u_tl, v_tl, size, xq, yq, ref, lane, r, xyz);
    if (r.status == SVI_OK) store_desc(out.desc + (size_t)q * 32, r.w, lane);
    if (lane == 0) {
        out.status[q] = (uint8_t)r.status;
        out.dist[q] = r.dist;
        out.idx[q] = r.idx;
        if (r.status == SVI_OK) {
            out.uv[2 * q] = r.u; out.uv[2 * q + 1] = r.v;
            out.xyz[3 * q] = xyz[0]; out.xyz[3 * q + 1] = xyz[1]; out.xyz[3 * q + 2] = xyz[2];
        }
    }
}

__global__ void point_in_left_kernel(TriConst tc, int n, const float* __restrict__ uvl, const float* __restrict__ uvr,
                                     double* __restrict__ xyz, uint8_t* __restrict__ status) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double p[3] = {0.0, 0.0, 0.0};
    int st = point_in_left(tc, uvl[2 * i], uvl[2 * i + 1], uvr[2 * i], p);
    status[i] = (uint8_t)st;
    xyz[3 * i] = p[0]; xyz[3 * i + 1] = p[1]; xyz[3 * i + 2] = p[2];
}

// ------------------------------------------------------------------ tracking, stage 1
struct TrackConst {
    double T[12];     // rows 0..2 of WORLDtoLEFT
    double PL[12], PR[12];
    float tri_scale;  // 1 + motion scaling (CFundamentalMatcher.cpp:1363)
    float cutoff1;    // m_dMatchingDistanceCutoffTrackingStage1
    int stage1_match; // 0: only the field-of-view gate of :1416 (the caller asked for stage 2 without stage 1)
};
struct LandmarksDev {
    const double* xyz_w; const uint8_t* desc_l; const uint8_t* desc_r; const float* disparity; const float* size;
};
struct TrackOutDev {
    uint8_t* status; uint8_t* stage; float* uv_l; float* uv_r; double* xyz; uint8_t* desc_l; uint8_t* desc_r;
};

// CPinholeCamera::getProjectionRounded (src/vision/CPinholeCamera.h:202-210)
__device__ __forceinline__ void projection_rounded(const double* P, const double* p, float& u, float& v) {
    double h0 = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(P[0], p[0]), __dmul_rn(P[1], p[1])), __dmul_rn(P[2], p[2])), P[3]);
    double h1 = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(P[4], p[0]), __dmul_rn(P[5], p[1])), __dmul_rn(P[6], p[2])), P[7]);
    double h2 = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(P[8], p[0]), __dmul_rn(P[9], p[1])), __dmul_rn(P[10], p[2])), P[11]);
    u = round_half_away((float)__ddiv_rn(h0, h2));
    v = round_half_away((float)__ddiv_rn(h1, h2));
}

__global__ void __launch_bounds__(MATCH_WARPS * 32, 3)
track_stage1_kernel(const uint16_t* __restrict__ box_l, const uint16_t* __restrict__ box_r,
                    const __grid_constant__ CUtensorMap map_l, const __grid_constant__ CUtensorMap map_ls,
                    const __grid_constant__ CUtensorMap map_r, const __grid_constant__ CUtensorMap map_rs, FrameGeom g,
                    TriConst tc, TrackConst k, LandmarksDev lm, int n, TrackOutDev out) {
    extern __shared__ __align__(128) unsigned char match_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = blockIdx.x * MATCH_WARPS + warp;
    if (q >= n) return;
    PatchStage ps;
    patch_stage_init(ps, match_smem, &map_r, &map_rs, 0, warp, lane);
    const double wx = lm.xyz_w[3 * q], wy = lm.xyz_w[3 * q + 1], wz = lm.xyz_w[3 * q + 2];
    double p[3];
#pragma unroll
    for (int r = 0; r < 3; ++r)   // Isometry3d * Vector3d = linear * v + translation (:1404)
        p[r] = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(k.T[4 * r], wx), __dmul_rn(k.T[4 * r + 1], wy)), __dmul_rn(k.T[4 * r + 2], wz)), k.T[4 * r + 3]);
    float ul, vl, ur, vr;
    projection_rounded(k.PL, p, ul, vl);
    projection_rounded(k.PR, p, ur, vr);
    const float size = lm.size[q], half = 4.f * size;
    const float search = k.tri_scale * lm.disparity[q];
    int status = SVI_TRK_OUT_OF_FOV, stage = 0;
    SearchResult r;
    double xyz[3] = {0.0, 0.0, 0.0};
    uint32_t mine[kDescWords], last_l[kDescWords], last_r[kDescWords];
    float o_ul = 0.f, o_vl = 0.f, o_ur = 0.f, o_vr = 0.f;
    const bool in_fov = ul >= 28.f && ul < (float)(g.W - 28) && vl >= 28.f && vl < (float)(g.H - 28) &&
                        ur >= 28.f && ur < (float)(g.W - 28) && vr >= 28.f && vr < (float)(g.H - 28);
    // the single key-point (half, half) of the (8*size+1)^2 ROI must survive BRIEF's border filter
    const int roi_len = (int)(8.f * size + 1.f);
    const bool kp_ok = cv_round_f(half) >= kBriefBorder && cv_round_f(half) < roi_len - kBriefBorder;
    if (in_fov && !k.stage1_match) status = SVI_TRK_STAGE1_DIST;   // untracked, inside both fields of view
    if (in_fov && k.stage1_match) {
        load_desc(lm.desc_l + (size_t)q * 32, last_l);
        load_desc(lm.desc_r + (size_t)q * 32, last_r);
        // STAGE 1 LEFT :1419-1476 -- descriptor exactly at the projection, then search RIGHT
        {
            const float roi_x = ul - half, roi_y = vl - half;
            const bool roi_ok = (int)roi_x >= 0 && (int)roi_y >= 0 && (int)roi_x + roi_len <= g.W && (int)roi_y + roi_len <= g.H;
            if (kp_ok && roi_ok)
                brief_at_point(box_l, g.box_pitch, (int)roi_x + brief_centre(half), (int)roi_y + brief_centre(half), lane, mine);
            status = roi_ok ? SVI_TRK_STAGE1_DIST : SVI_TRI_BAD_ROI;
            if (kp_ok && roi_ok && k.cutoff1 > (float)hamming_words(last_l, mine)) {
                ps.map = &map_r; ps.map_s = &map_rs;
                triangulate_right_dev(g, tc, ps, fmaxf(0.f, roi_x - search), roi_y, size, roi_x + half, roi_y + half, mine,
                                      lane, r, xyz);
                status = r.status;
                if (status == SVI_OK) {
                    if (tc.depth_min > xyz[2] || tc.depth_max < xyz[2]) status = SVI_TRK_DEPTH;
                    else if (k.cutoff1 < (float)hamming_words(last_r, r.w)) status = SVI_TRK_TRI_DESC;
                    else { stage = 1; o_ul = ul; o_vl = vl; o_ur = r.u; o_vr = r.v; }
                }
            }
        }
        // STAGE 1 RIGHT :1480-1538
        if (stage == 0) {
            const float roi_x = ur - half, roi_y = vr - half;
            const bool roi_ok = (int)roi_x >= 0 && (int)roi_y >= 0 && (int)roi_x + roi_len <= g.W && (int)roi_y + roi_len <= g.H;
            if (kp_ok && roi_ok)
                brief_at_point(box_r, g.box_pitch, (int)roi_x + brief_centre(half), (int)roi_y + brief_centre(half), lane, mine);
            status = roi_ok ? SVI_TRK_STAGE1_DIST : SVI_TRI_BAD_ROI;
            if (kp_ok && roi_ok && k.cutoff1 > (float)hamming_words(last_r, mine)) {
                ps.map = &map_l; ps.map_s = &map_ls;
                triangulate_left_dev(g, tc, ps, search, roi_x, roi_y, size, roi_x + half, mine, lane, r, xyz);
                status = r.status;
                if (status == SVI_OK) {
                    if (tc.depth_min > xyz[2] || tc.depth_max < xyz[2]) status = SVI_TRK_DEPTH;
                    else if (k.cutoff1 < (float)hamming_words(last_l, r.w)) status = SVI_TRK_TRI_DESC;
                    else { stage = 2; o_ul = r.u; o_vl = r.v; o_ur = ur; o_vr = vr; }
                }
            }
        }
    }
    if (stage == 1) { store_desc(out.desc_l + (size_t)q * 32, mine, lane); store_desc(out.desc_r + (size_t)q * 32, r.w, lane); }
    if (stage == 2) { store_desc(out.desc_l + (size_t)q * 32, r.w, lane); store_desc(out.desc_r + (size_t)q * 32, mine, lane); }
    if (lane == 0) {
        out.status[q] = (uint8_t)status;
        out.stage[q] = (uint8_t)stage;
        if (stage) {
            out.uv_l[2 * q] = o_ul; out.uv_l[2 * q + 1] = o_vl;
            out.uv_r[2 * q] = o_ur; out.uv_r[2 * q + 1] = o_vr;
            out.xyz[3 * q] = xyz[0]; out.xyz[3 * q + 1] = xyz[1]; out.xyz[3 * q + 2] = xyz[2];
        }
    }
}

// ------------------------------------------------------------------ tracking, stage 2
// One work item = one landmark on one side (CFundamentalMatcher.cpp:1545-1665 LEFT, :1669-1785 RIGHT).
struct Stage2Item {
    int q;                 // landmark index (output slot)
    int gx, gy, gw, gh;    // window grown by 28 px and clamped (:1572-1575), as cv::Rect(Point2f, Point2f)
    float ul_x, ul_y;      // ptUpperLeft of the search window (Point2f)
    float search;          // fTriangulationScale * lastDisparity
    float size;            // dKeyPointSize
};

// After GFTT has run inside every item's window (harris/nms/select kernels in window mode): shift the
// corners by (+28,+28) (:1579), BRIEF on the grown window with its own border filter (:1580), 1 x K
// Hamming arg-min against the landmark's last descriptor (:1584), cut-off 50, then the scan-line
// triangulation in the other image, depth window and the other-side descriptor check (:1586-1637).
// One warp per item; lanes = corners for the K descriptors (box-sum gathers from global memory).
template <bool kLeft>
__global__ void __launch_bounds__(MATCH_WARPS * 32, 3)
track_stage2_kernel(const uint16_t* __restrict__ box_this, const __grid_constant__ CUtensorMap map_other,
                    const __grid_constant__ CUtensorMap map_other_s, FrameGeom g, TriConst tc, float cutoff2,
                    const Stage2Item* __restrict__ items, const int* __restrict__ n_items, const ushort2* __restrict__ det_xy,
                    const int* __restrict__ n_det, int max_corners, LandmarksDev lm, TrackOutDev out) {
    extern __shared__ __align__(128) unsigned char match_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int i = blockIdx.x * MATCH_WARPS + warp;
    if (i >= *n_items) return;   // the item list was compacted on the device
    const Stage2Item it = items[i];
    const int q = it.q;
    PatchStage ps;
    patch_stage_init(ps, match_smem, &map_other, &map_other_s, 0, warp, lane);
    const float half = 4.f * it.size;
    uint32_t last_this[kDescWords], last_other[kDescWords];
    load_desc((kLeft ? lm.desc_l : lm.desc_r) + (size_t)q * 32, last_this);
    load_desc((kLeft ? lm.desc_r : lm.desc_l) + (size_t)q * 32, last_other);

    int status = SVI_TRK_NO_FEATURES;
    const int nd = n_det[i];
    uint32_t best = 0xFFFFFFFFu;
    if (nd > 0) {
        status = SVI_TRK_NO_MATCHES;
        const ushort2* corners = det_xy + (size_t)i * max_corners;
        // lanes = corners: every lane describes its own corner (brief_at_point_lane), 32 corners per round
        SVI_CHECK(3, nd <= max_corners);
        for (int k0 = 0; k0 < nd; k0 += 32) {
            const int k = k0 + lane;
            uint32_t key = 0xFFFFFFFFu;
            if (k < nd) {
                const ushort2 c = corners[k];
                const float px = (float)c.x + half, py = (float)c.y + half;
                const int rx = cv_round_f(px), ry = cv_round_f(py), cx = brief_centre(px), cy = brief_centre(py);
                const bool keep = rx >= kBriefBorder && rx < it.gw - kBriefBorder && ry >= kBriefBorder && ry < it.gh - kBriefBorder &&
                                  cx >= kBriefBorder && cx < it.gw - kBriefBorder && cy >= kBriefBorder && cy < it.gh - kBriefBorder;
                if (keep) {
                    uint32_t w[kDescWords];
                    brief_at_point_lane(box_this, g.box_pitch, it.gx + cx, it.gy + cy, w);
                    key = ((uint32_t)hamming_words(w, last_this) << 16) | (uint32_t)k;
                }
            }
            best = min(best, warp_min_u32(key));   // smaller k wins ties: BFMatcher's first minimum in pool order
        }
    }
    SearchResult r;
    double xyz[3] = {0.0, 0.0, 0.0};
    uint32_t mine[kDescWords];
    float in_x = 0.f, in_y = 0.f;
    if (best != 0xFFFFFFFFu) {
        const int dist = (int)(best >> 16), k = (int)(best & 0xFFFFu);
        status = SVI_TRK_DESC;
        if (cutoff2 > (float)dist) {
            const ushort2 c = det_xy[(size_t)i * max_corners + k];
            const float px = (float)c.x + half, py = (float)c.y + half;
            in_x = (it.ul_x + px) - half;       // ptUpperLeft + ptBestMatch - ptOffsetKeyPointHalf (:1592)
            in_y = (it.ul_y + py) - half;
            brief_at_point(box_this, g.box_pitch, it.gx + brief_centre(px), it.gy + brief_centre(py), lane, mine);
            const float v_ref = in_y - half;
            status = SVI_TRK_RANGE;
            if (0.0f <= v_ref) {
                if (kLeft) triangulate_right_dev(g, tc, ps, fmaxf(0.f, (in_x - it.search) - half), v_ref, it.size, in_x, in_y, mine, lane, r, xyz);
                else triangulate_left_dev(g, tc, ps, it.search, fmaxf(0.f, in_x - half), v_ref, it.size, in_x, mine, lane, r, xyz);
                status = r.status;
                if (status == SVI_OK) {
                    if (tc.depth_min > xyz[2] || tc.depth_max < xyz[2]) status = SVI_TRK_DEPTH;
                    else if (!(cutoff2 > (float)hamming_words(last_other, r.w))) status = SVI_TRK_TRI_DESC;
                }
            }
        }
    }
    if (status == SVI_OK) {
        store_desc((kLeft ? out.desc_l : out.desc_r) + (size_t)q * 32, mine, lane);
        store_desc((kLeft ? out.desc_r : out.desc_l) + (size_t)q * 32, r.w, lane);
    }
    if (lane == 0) {
        out.status[q] = (uint8_t)status;
        if (status == SVI_OK) {
            out.stage[q] = kLeft ? 3 : 4;
            float* uv_this = kLeft ? out.uv_l : out.uv_r;
            float* uv_other = kLeft ? out.uv_r : out.uv_l;
            uv_this[2 * q] = in_x; uv_this[2 * q + 1] = in_y;
            uv_other[2 * q] = r.u; uv_other[2 * q + 1] = r.v;
            out.xyz[3 * q] = xyz[0]; out.xyz[3 * q + 1] = xyz[1]; out.xyz[3 * q + 2] = xyz[2];
        }
    }
}

// ------------------------------------------------------------------ tracking, stage 3 (epipolar line)
struct Stage3Item {
    int q;             // landmark index
    int along_u;       // 1: one sample per u, v from the line (:2142-2238); 0: one per v, u from the line (:2240-2334)
    int count;         // uDeltaU / uDeltaV
    float size, search;   // dKeyPointSize, (float)((1 + scaling) * lastDisparity)  (:2415)
    double start;      // dUMinimum / dVForUMinimum
    double c0, c1, c2; // line coefficients F * uvReference (:1818)
};

__device__ __forceinline__ void epipolar_sample(const Stage3Item& it, int i, double off, float& fx, float& fy) {
    if (it.along_u) {
        const double du = __dadd_rn(it.start, (double)i);
        const double dv = __dadd_rn(__ddiv_rn(-__dadd_rn(__dmul_rn(it.c0, du), it.c2), it.c1), off);   // _getCurveV + offset
        fx = (float)du; fy = (float)dv;
    } else {
        const double dv = __dadd_rn(it.start, (double)i);
        const double du = __dadd_rn(__ddiv_rn(-__dadd_rn(__dmul_rn(it.c1, dv), it.c2), it.c0), off);   // _getCurveU + offset
        fx = (float)du; fy = (float)dv;
    }
}

// _getMatchSampleRecursiveU/V + _getMatch (:2142-2397) and _addMeasurementToLandmarkLEFT (:2399-2453):
// the line geometry (coefficients, clipped range, sampling direction) comes from stage3_plan_kernel; one warp per item.
__global__ void __launch_bounds__(MATCH_WARPS * 32, 3)
track_stage3_kernel(const uint16_t* __restrict__ box_l, const __grid_constant__ CUtensorMap map_r,
                    const __grid_constant__ CUtensorMap map_rs, FrameGeom g, TriConst tc, float cutoff3, float cutoff_orig,
                    const Stage3Item* __restrict__ items, const int* __restrict__ n_items, const uint8_t* __restrict__ desc_orig,
                    LandmarksDev lm, TrackOutDev out) {
    extern __shared__ __align__(128) unsigned char match_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int idx = blockIdx.x * MATCH_WARPS + warp;
    if (idx >= *n_items) return;   // the item list was compacted on the device
    const Stage3Item it = items[idx];
    const int q = it.q, n = it.count;
    PatchStage ps;
    patch_stage_init(ps, match_smem, &map_r, &map_rs, 0, warp, lane);
    uint32_t last_l[kDescWords], orig_l[kDescWords], mine[kDescWords];
    load_desc(lm.desc_l + (size_t)q * 32, last_l);
    load_desc(desc_orig + (size_t)q * 32, orig_l);
    const float wf = (float)g.W, hf = (float)g.H;
    int status = SVI_EPI_POOL_EMPTY;
    float res_x = 0.f, res_y = 0.f;
    bool found = false;
    for (int attempt = 0; attempt < 2 && !found; ++attempt) {
        const double off = attempt ? 2.0 : 0.0;    // recursion depth 0, then 2 (limit 2, step 2)
        float ax, ay, bx, by, cx, cy;
        epipolar_sample(it, 0, off, ax, ay);
        epipolar_sample(it, n - 1, off, bx, by);
        epipolar_sample(it, n / 2, off, cx, cy);
        const float f_du = fabsf(ax - bx) + 16.f * it.size, f_dv = fabsf(ay - by) + 16.f * it.size;
        const float u_tl = fmaxf(cx - f_du / 2.f, 0.f), v_tl = fmaxf(cy - f_dv / 2.f, 0.f);
        const float width = fminf(f_du, wf - u_tl), height = fminf(f_dv, hf - v_tl);
        status = SVI_EPI_POOL_EMPTY;
        if (!(isfinite(u_tl) && isfinite(v_tl) && isfinite(width) && isfinite(height))) continue;
        const int rx = (int)u_tl, ry = (int)v_tl, rw = (int)width, rh = (int)height;   // cv::Rect(float...) truncates
        if (rw <= 0 || rh <= 0 || rx + rw > g.W || ry + rh > g.H) continue;
        uint32_t best = 0xFFFFFFFFu;
        for (int i0 = 0; i0 < n; i0 += 32) {
            const int i = i0 + lane;
            bool keep = false;
            int sx = 0, sy = 0;
            if (i < n) {
                float fx, fy;
                epipolar_sample(it, i, off, fx, fy);
                const float kx = fx - u_tl, ky = fy - v_tl;
                const int rnx = cv_round_f(kx), rny = cv_round_f(ky), ccx = brief_centre(kx), ccy = brief_centre(ky);
                keep = rnx >= kBriefBorder && rnx < rw - kBriefBorder && rny >= kBriefBorder && rny < rh - kBriefBorder &&
                       ccx >= kBriefBorder && ccx < rw - kBriefBorder && ccy >= kBriefBorder && ccy < rh - kBriefBorder;
                sx = rx + ccx;
                sy = ry + ccy;
            }
            uint32_t dist = 0;
            if (keep) {
                uint32_t w[kDescWords];
                brief_at_point_lane(box_l, g.box_pitch, sx, sy, w);
                dist = (uint32_t)hamming_words(w, last_l);
            }
            best = min(best, warp_min_u32(keep ? ((dist << 16) | (uint32_t)i) : 0xFFFFFFFFu));
        }
        if (best == 0xFFFFFFFFu) continue;                       // "empty key point pool"
        status = SVI_EPI_DIST;
        if (!(cutoff3 > (float)(best >> 16))) continue;
        float fx, fy;
        epipolar_sample(it, (int)(best & 0xFFFFu), off, fx, fy);
        const float kx = fx - u_tl, ky = fy - v_tl;
        brief_at_point(box_l, g.box_pitch, rx + brief_centre(kx), ry + brief_centre(ky), lane, mine);
        status = SVI_EPI_ORIG_DIST;
        if (!(cutoff_orig > (float)hamming_words(orig_l, mine))) continue;
        res_x = kx + u_tl;                                        // cKeyPointShifted.pt += p_ptOffsetROI
        res_y = ky + v_tl;
        found = true;
    }
    SearchResult r;
    double xyz[3] = {0.0, 0.0, 0.0};
    if (found) {
        triangulate_right_dev(g, tc, ps, fmaxf(0.f, (res_x - it.search) - 4.f * it.size), res_y - 4.f * it.size, it.size, res_x,
                              res_y, mine, lane, r, xyz);
        status = r.status;
        if (status == SVI_OK && (tc.depth_min > xyz[2] || tc.depth_max < xyz[2])) status = SVI_TRK_DEPTH;
    }
    if (status == SVI_OK) {
        store_desc(out.desc_l + (size_t)q * 32, mine, lane);
        store_desc(out.desc_r + (size_t)q * 32, r.w, lane);
    }
    if (lane == 0) {
        out.status[q] = (uint8_t)status;
        if (status == SVI_OK) {
            out.stage[q] = 5;
            out.uv_l[2 * q] = res_x; out.uv_l[2 * q + 1] = res_y;
            out.uv_r[2 * q] = r.u; out.uv_r[2 * q + 1] = r.v;
            out.xyz[3 * q] = xyz[0]; out.xyz[3 * q + 1] = xyz[1]; out.xyz[3 * q + 2] = xyz[2];
        }
    }
}

}  // namespace svi
