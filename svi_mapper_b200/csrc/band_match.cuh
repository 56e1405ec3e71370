// band_match.cuh -- key-point to key-point Hamming matching inside an epipolar row band (the sparse form of a stereo frame).
//
// What cv::BFMatcher(NORM_HAMMING).match(query, train, mask) computes with the band mask
//   mask(q, t) = |y_q - y_t| <= band_v  &&  min_disparity <= x_q - x_t <= max_disparity      (fp32, as written)
// plus the second-smallest admissible distance (for a ratio test in the caller).  Not a reference code path: the reference
// searches dense scan lines (brief_match.cuh); this is the second way of matching a stereo pair that BASELINE.json's C5 names.
//
// Work decomposition: a CTA owns BM_THREADS queries, one thread each, with the query's descriptor in registers.  The trains
// the CTA can reach form ONE contiguous range of the train list -- in a stereo frame both lists are sorted by image row
// (bin_keypoints_kernel with one-row bins), the CTA's queries are consecutive in row order, and the range is the rows
// [y_min - band, y_max + band]; for svi_match_epipolar it is the whole caller-ordered list.  That range streams through
// shared memory in double-buffered tiles (descriptor, coordinates, original index: one bulk async copy each), and every
// thread tests every train of a tile with broadcast reads: the admissibility test, 8 x XOR/POPC, then an update of its
// (distance << 32 | original index) minimum and its second-smallest distance.  Both reductions are order-independent, so the
// result is the brute-force scan's whatever the tiles and whatever the band (a band >= H streams the whole list).
//
// Three modes (BandMode):
//   BM_FRAME     svi_stereo_frames_sparse[_device]: LEFT queries against RIGHT trains; the same kernel finishes the LEFT slot:
//                cut-off, with `mutual` set the left-right check against `rev`, getPointInLEFT (point_in_left, fp64), outputs.
//   BM_REVERSE   the left-right check's reverse pass: RIGHT queries against LEFT trains (row-ordered descriptors gathered by
//                gather_rows_kernel) with the bounds mirrored to (-max_disparity, -min_disparity).  x_R - x_L == -(x_L - x_R)
//                exactly in IEEE fp32, so the test admits exactly the pairs BM_FRAME admits, NaNs included.  Writes only
//                the (distance << 32 | LEFT slot) minimum -- the first arg-min: lowest slot on ties -- into rev[f][original
//                RIGHT index] by 64-bit atomicMin (rev starts at ~0: no admissible LEFT key-point).  Few RIGHT queries against
//                many LEFT trains make few, long CTAs, so gridDim.z splits each query block's train range into that many
//                runs of tiles; the minimum is order-independent, so the result does not depend on the split.
//   BM_EPIPOLAR  svi_match_epipolar: caller-ordered float lists; writes index, distance and second.
#pragma once
#include <type_traits>

#include "brief_match.cuh"

namespace svi {

constexpr int BM_THREADS = 128;   // queries per CTA
constexpr int BM_TILE = 256;      // trains per shared tile (a multiple of 4: every bulk copy is a multiple of 16 bytes)
constexpr int BM_ALIGN = 4;       // the streamed range starts and ends on a multiple of 4 elements (16-byte copy addresses)

enum BandMode { BM_EPIPOLAR = 0, BM_FRAME = 1, BM_REVERSE = 2 };

// Tile layout: [descriptors | coordinates | original indices (row-sorted lists only)], twice, then two mbarriers.
// kFrame: the row-sorted lists of a stereo frame (BM_FRAME and BM_REVERSE).
template <bool kFrame>
struct BandTile {
    using XY = typename std::conditional<kFrame, ushort2, float2>::type;   // frame: integer corners; epipolar: caller's floats
    static constexpr int DESC = BM_TILE * 32;
    static constexpr int XYB = BM_TILE * (int)sizeof(XY);
    static constexpr int SLOTB = kFrame ? BM_TILE * 4 : 0;
    static constexpr int BUF = DESC + XYB + SLOTB;
    static constexpr int SMEM = 2 * BUF + 16;
};

struct BandArgs {
    float band_v, min_disp, max_disp;
    // queries.  Frame: LEFT key-points sorted by row ([f][max_corners]), their slots, per-frame counts; the descriptors are
    // out.desc_l at the slot.  Reverse: the same for RIGHT, descriptors in row order ([f][max_corners]).  Epipolar: nq
    // descriptors / coordinates in caller order.
    const ushort2* q_kp;
    const uint32_t* q_slot;
    const int* n_q;
    const uint8_t* q_desc;
    const float2* q_xy;
    int nq;
    // trains.  Frame: RIGHT key-points, slots and descriptors sorted by row ([f][max_corners]) and the row CSR ([f][H + 1]).
    // Reverse: the same for LEFT.  Epipolar: nt descriptors / coordinates in caller order.
    const ushort2* t_kp;
    const uint32_t* t_slot;
    const uint8_t* t_desc;
    const int* t_row;
    const float2* t_xy;
    int nt;
    int H, max_corners;
    // outputs.  Frame: the slot arrays of out (+ second at the same index).  Epipolar: index / distance / second per query.
    StereoOutDev out;
    int out_frame0;
    TriConst tc;
    int* index;
    int* distance;
    int* second;
    // left-right check.  Frame: `mutual` (CTA-uniform) applies it against rev, per-frame train counts n_t bound its index.
    // Reverse: the output, rev[f][original RIGHT index] ([f][max_corners]), (distance << 32 | LEFT slot) or ~0.
    unsigned long long* rev;
    const int* n_t;
    int mutual;
};

__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}

// The left-right check of LEFT slot `slot` matched to RIGHT key-point `idx`: is the reverse pass's arg-min of idx another slot?
__device__ __forceinline__ bool not_mutual(const BandArgs& a, size_t fbase, int f, int idx, uint32_t slot) {
    SVI_CHECK(12, idx < a.n_t[f] && idx < a.max_corners);
    return (uint32_t)a.rev[fbase + idx] != slot;
}

template <int kMode>
__global__ void __launch_bounds__(BM_THREADS)
band_match_kernel(const __grid_constant__ BandArgs a) {
    constexpr bool kFrame = kMode != BM_EPIPOLAR;   // row-sorted lists of a stereo frame
    using TL = BandTile<kFrame>;
    using XY = typename TL::XY;
    extern __shared__ __align__(128) unsigned char bm_smem[];
    const int tid = threadIdx.x, f = blockIdx.y;
    const int MC = a.max_corners;
    const size_t fbase = kFrame ? (size_t)f * MC : 0;   // first element of this frame's lists
    const int nq = kFrame ? min(a.n_q[f], MC) : a.nq;
    const int q0 = blockIdx.x * BM_THREADS;
    if (q0 >= nq) return;   // CTA-uniform
    const int q = q0 + tid;
    const bool live = q < nq;

    // ---- the query: coordinates and descriptor (raw words: XOR / popc do not care about the byte order)
    float xq = 0.f, yq = 0.f;
    uint32_t slot = (uint32_t)q;
    uint32_t ref[kDescWords] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (live) {
        const uint8_t* src;
        if constexpr (kFrame) {
            const ushort2 k = a.q_kp[fbase + q];
            xq = (float)k.x;
            yq = (float)k.y;
            slot = a.q_slot[fbase + q];
            if constexpr (kMode == BM_FRAME) {
                SVI_CHECK(12, slot < (uint32_t)MC && slot < (uint32_t)a.out.cap);
                src = a.out.desc_l + ((size_t)(a.out_frame0 + f) * a.out.cap + slot) * 32;
            } else {
                SVI_CHECK(12, slot < (uint32_t)MC);
                src = a.q_desc + (fbase + q) * 32;
            }
        } else {
            const float2 k = a.q_xy[q];
            xq = k.x;
            yq = k.y;
            src = a.q_desc + (size_t)q * 32;
        }
#pragma unroll
        for (int j = 0; j < kDescWords; ++j) ref[j] = __ldg(reinterpret_cast<const uint32_t*>(src) + j);
    }

    // ---- the CTA's train range [lo, hi) (element indices of the whole list)
    size_t lo = 0, hi = 0;
    if constexpr (kFrame) {
        const int y_min = a.q_kp[fbase + q0].y, y_max = a.q_kp[fbase + min(q0 + BM_THREADS, nq) - 1].y;
        const int* rows = a.t_row + (size_t)f * (a.H + 1);
        if (a.band_v >= 0.f) {
            // a superset of the rows the band reaches (one row more on each side); the exact fp32 test below decides
            const int r0 = (int)fmax(0.0, floor((double)y_min - (double)a.band_v) - 1.0);
            const int r1 = (int)fmin((double)(a.H - 1), ceil((double)y_max + (double)a.band_v) + 1.0);
            if (r0 <= r1) {
                lo = fbase + rows[r0];
                hi = fbase + rows[r1 + 1];
            }
        }
        SVI_CHECK(12, lo <= hi && hi <= fbase + (size_t)MC);
    } else {
        hi = (size_t)a.nt;
    }
    const size_t a0 = lo & ~size_t(BM_ALIGN - 1), a1 = (hi + BM_ALIGN - 1) & ~size_t(BM_ALIGN - 1);
    const int n_tiles = (int)((a1 - a0 + BM_TILE - 1) / BM_TILE);
    int k0 = 0, k1 = n_tiles;   // the tiles this CTA streams
    if constexpr (kMode == BM_REVERSE) {
        const int per = (n_tiles + (int)gridDim.z - 1) / (int)gridDim.z;
        k0 = min(n_tiles, (int)blockIdx.z * per);
        k1 = min(n_tiles, k0 + per);
        if (k0 >= k1) return;   // CTA-uniform; nothing to merge
    }

    const uint32_t bar0 = smem_u32(bm_smem + 2 * TL::BUF);
    if (tid == 0) {
        mbar_init(bar0, 1);
        mbar_init(bar0 + 8, 1);
        fence_barrier_init();
    }
    __syncthreads();
    const uint8_t* t_desc = a.t_desc;
    const XY* t_xy;
    if constexpr (kFrame) t_xy = a.t_kp;
    else t_xy = a.t_xy;
    auto issue = [&](int k) {   // thread 0: tile k into buffer k & 1
        const size_t e0 = a0 + (size_t)k * BM_TILE;
        const uint32_t cnt = (uint32_t)min((size_t)BM_TILE, a1 - e0);
        const uint32_t buf = smem_u32(bm_smem + (k & 1) * TL::BUF), bar = bar0 + 8 * (k & 1);
        fence_proxy_async();   // the generic-proxy reads of this buffer (ordered by the CTA barrier) come first
        mbar_expect_tx(bar, cnt * (32u + (uint32_t)sizeof(XY) + (kFrame ? 4u : 0u)));
        bulk_load(buf, t_desc + e0 * 32, cnt * 32u, bar);
        bulk_load(buf + TL::DESC, t_xy + e0, cnt * (uint32_t)sizeof(XY), bar);
        if constexpr (kFrame) bulk_load(buf + TL::DESC + TL::XYB, a.t_slot + e0, cnt * 4u, bar);
    };
    if (tid == 0) {
        if (k0 < k1) issue(k0);
        if (k0 + 1 < k1) issue(k0 + 1);
    }

    const float band_v = a.band_v, dmin = a.min_disp, dmax = a.max_disp;
    unsigned long long best = ~0ull;   // (distance << 32 | original index): the minimum is the first arg-min
    uint32_t second = 0xFFFFFFFFu;
    size_t best_pos = 0;               // element index of the best train (frame: its row-ordered descriptor and corner)
    uint32_t phase = 0u;               // bit b: parity of buffer b's next completion
    for (int k = k0; k < k1; ++k) {
        const int b = k & 1;
        mbar_wait(bar0 + 8 * b, (phase >> b) & 1u);
        phase ^= 1u << b;
        const size_t e0 = a0 + (size_t)k * BM_TILE;
        const unsigned char* buf = bm_smem + b * TL::BUF;
        const uint4* sd = reinterpret_cast<const uint4*>(buf);
        const XY* sxy = reinterpret_cast<const XY*>(buf + TL::DESC);
        const uint32_t* ss = reinterpret_cast<const uint32_t*>(buf + TL::DESC + TL::XYB);
        // the part of the tile inside [lo, hi): the alignment padding at both ends is not looked at
        const int i0 = lo > e0 ? (int)(lo - e0) : 0;
        const int i1 = (int)min((long long)BM_TILE, (long long)hi - (long long)e0);
        for (int i = i0; i < i1; ++i) {
            const uint4 u = sd[2 * i], v = sd[2 * i + 1];
            const XY t = sxy[i];
            const float d = xq - (float)t.x;
            const bool adm = fabsf(yq - (float)t.y) <= band_v && d >= dmin && d <= dmax;
            const uint32_t dist = __popc(ref[0] ^ u.x) + __popc(ref[1] ^ u.y) + __popc(ref[2] ^ u.z) + __popc(ref[3] ^ u.w) +
                                  __popc(ref[4] ^ v.x) + __popc(ref[5] ^ v.y) + __popc(ref[6] ^ v.z) + __popc(ref[7] ^ v.w);
            uint32_t orig;
            if constexpr (kFrame) orig = ss[i];
            else orig = (uint32_t)(e0 + i);
            const unsigned long long key = ((unsigned long long)dist << 32) | orig;
            if (adm) {
                if (key < best) {
                    second = min(second, (uint32_t)(best >> 32));
                    best = key;
                    best_pos = e0 + i;
                } else {
                    second = min(second, dist);
                }
            }
        }
        __syncthreads();   // every thread is done with buffer b
        if (tid == 0 && k + 2 < k1) issue(k + 2);
    }
    if (!live) return;

    const bool any = best != ~0ull;
    const int dist = any ? (int)(best >> 32) : -1;
    const int idx = any ? (int)(uint32_t)best : -1;
    const int sec = second != 0xFFFFFFFFu ? (int)second : -1;
    if constexpr (kMode == BM_REVERSE) {
        if (any) atomicMin(a.rev + fbase + slot, best);
    } else if constexpr (kMode == BM_EPIPOLAR) {
        a.index[q] = idx;
        a.distance[q] = dist;
        a.second[q] = sec;
    } else {
        const StereoOutDev& out = a.out;
        const size_t o = (size_t)(a.out_frame0 + f) * out.cap + slot;
        out.uv_l[o * 2] = xq;
        out.uv_l[o * 2 + 1] = yq;
        out.dist[o] = dist;
        out.idx[o] = idx;
        a.second[o] = sec;
        int st;
        if (!any) {
            st = SVI_TRI_NO_MATCH;
        } else if (!((float)dist < a.tc.match_cutoff)) {
            st = SVI_TRI_DISTANCE;
        } else if (a.mutual && not_mutual(a, fbase, f, idx, slot)) {
            st = SVI_SPARSE_NOT_MUTUAL;
        } else {
            SVI_CHECK(12, best_pos >= lo && best_pos < hi);
            const ushort2 t = a.t_kp[best_pos];
            double xyz[3] = {0.0, 0.0, 0.0};
            st = point_in_left(a.tc, xq, yq, (float)t.x, xyz);
            if (st == SVI_OK) {
                out.uv_r[o * 2] = (float)t.x;
                out.uv_r[o * 2 + 1] = (float)t.y;
                out.xyz[o * 3] = xyz[0];
                out.xyz[o * 3 + 1] = xyz[1];
                out.xyz[o * 3 + 2] = xyz[2];
                const uint32_t* ds = reinterpret_cast<const uint32_t*>(a.t_desc + best_pos * 32);
                uint32_t* dd = reinterpret_cast<uint32_t*>(out.desc_r + o * 32);
#pragma unroll
                for (int j = 0; j < kDescWords; ++j) dd[j] = __ldg(ds + j);
            }
        }
        out.status[o] = (uint8_t)st;
    }
}

// LEFT descriptors in row order for the reverse pass: dst[f][i] = desc[frame0 + f][slot[f][i]] for the frame's n[f] key-points,
// one thread per 16-byte half of a descriptor.
constexpr int GR_THREADS = 256;
__global__ void __launch_bounds__(GR_THREADS)
gather_rows_kernel(const uint8_t* desc, int cap, int frame0, const uint32_t* slot, const int* n, int max_corners, uint8_t* dst) {
    const int f = blockIdx.y, t = blockIdx.x * GR_THREADS + threadIdx.x, i = t >> 1;
    if (i >= min(n[f], max_corners)) return;
    const size_t e = (size_t)f * max_corners + i;
    const uint32_t s = slot[e];
    SVI_CHECK(12, s < (uint32_t)max_corners && s < (uint32_t)cap);
    reinterpret_cast<uint4*>(dst + e * 32)[t & 1] = __ldg(reinterpret_cast<const uint4*>(desc + ((size_t)(frame0 + f) * cap + s) * 32) + (t & 1));
}

}  // namespace svi
