// subpixel.cuh -- sub-pixel disparity of the new-landmark path's matches (optional mode: svi_params.subpixel_window > 0).
//
// Not a reference code path: ORB-SLAM2's Frame::ComputeStereoMatches refinement, specified step by step in include/svi_gpu.h
// (svi_params.subpixel_window) so that the CPU restatement the tests use and this kernel agree bit for bit.  It runs once
// per chunk after the matcher, on the matcher's outputs, and rewrites uv_right.x, xyz_left and status of the SVI_OK slots.
//
// Work decomposition: one warp per slot.  The warp stages the centred LEFT patch (int16) and the RIGHT strip of all 2L+1
// patches ((2w+1) rows x (2w+1+2L) bytes) in shared memory, then per offset k every lane sums |PL - PR(k)| over its share of
// the patch and __reduce_add_sync gives SAD(k) to every lane.  Integer arithmetic up to the parabola, no atomics: the
// result does not depend on the schedule.
#pragma once
#include "brief_match.cuh"

namespace svi {

constexpr int SP_WARPS = 4;                  // slots per CTA
constexpr int SP_MAX_REACH = kBriefBorder;   // w + L <= 28 (svi_create)
constexpr int SP_MAX_PATCH = 55 * 55;        // (2w+1)^2, w <= 27
constexpr int SP_MAX_STRIP = 55 * 57;        // (2w+1) x (2w+2L+1), w + L <= 28

struct SubpixelArgs {
    const uint8_t* left;    // the planes the detector read, g.img_pitch bytes per row, g.img_stride per frame
    const uint8_t* right;
    FrameGeom g;
    const int* n_kp;        // [chunk frame] LEFT key-points (slots) of the frame
    int max_corners;
    StereoOutDev out;
    int out_frame0;
    TriConst tc;
    int w, L;
};

__global__ void __launch_bounds__(SP_WARPS * 32) subpixel_refine_kernel(const SubpixelArgs a) {
    __shared__ int16_t s_pl[SP_WARPS][SP_MAX_PATCH];
    __shared__ uint8_t s_strip[SP_WARPS][SP_MAX_STRIP];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int f = blockIdx.y, slot = blockIdx.x * SP_WARPS + warp;
    if (slot >= min(a.n_kp[f], a.max_corners)) return;
    SVI_CHECK(13, slot < a.out.cap);
    const size_t o = (size_t)(a.out_frame0 + f) * a.out.cap + slot;
    if (a.out.status[o] != SVI_OK) return;   // warp-uniform
    const int w = a.w, L = a.L, D = 2 * w + 1, SW = D + 2 * L, P = D * D;
    const float xl_f = a.out.uv_l[o * 2], y_f = a.out.uv_l[o * 2 + 1], xr_f = a.out.uv_r[o * 2];
    const int xl = (int)xl_f, y = (int)y_f, xr = (int)xr_f;
    int st;
    float xr_new = 0.f;
    double xyz[3] = {0.0, 0.0, 0.0};
    // whole-pixel matches (the reference's geometry, every sparse match) are always inside; see the header for the others
    if (xr - w - L < 0 || xr + w + L >= a.g.W || xl - w < 0 || xl + w >= a.g.W || y - w < 0 || y + w >= a.g.H) {
        st = SVI_SUBPIXEL_REJECTED;
    } else {
        SVI_CHECK(13, w + L <= SP_MAX_REACH && P <= SP_MAX_PATCH && D * SW <= SP_MAX_STRIP);
        const uint8_t* il = a.left + (size_t)f * a.g.img_stride + (size_t)(y - w) * a.g.img_pitch + (xl - w);
        const uint8_t* ir = a.right + (size_t)f * a.g.img_stride + (size_t)(y - w) * a.g.img_pitch + (xr - w - L);
        int16_t* pl = s_pl[warp];
        uint8_t* strip = s_strip[warp];
        const int cl = __ldg(il + (size_t)w * a.g.img_pitch + w);
        for (int p = lane; p < P; p += 32) {
            const int dy = p / D, dx = p - dy * D;
            pl[p] = (int16_t)(__ldg(il + (size_t)dy * a.g.img_pitch + dx) - cl);
        }
        for (int p = lane; p < D * SW; p += 32) {
            const int r = p / SW, c = p - r * SW;
            strip[p] = __ldg(ir + (size_t)r * a.g.img_pitch + c);
        }
        __syncwarp();
        // (p + 0.5) / D lies at least 0.5 / D >= 1/110 away from an integer, far above the fp32 error: exact row of p
        const float inv_d = 1.f / (float)D;
        int best = 0x7FFFFFFF, kbest = -L, prev = 0, s1 = 0, s3 = 0;
        bool want_next = false;
        for (int k = -L; k <= L; ++k) {
            const int j = k + L;
            const int cr = strip[w * SW + w + j];
            int s = 0;
            for (int p = lane; p < P; p += 32) {
                const int dy = (int)(((float)p + 0.5f) * inv_d), dx = p - dy * D;
                SVI_CHECK(13, dx >= 0 && dx < D);
                s += abs((int)pl[p] - ((int)strip[dy * SW + dx + j] - cr));
            }
            s = (int)__reduce_add_sync(0xFFFFFFFFu, (unsigned)s);
            if (s < best) {          // strict: the first minimum in increasing k
                best = s; kbest = k; s1 = prev; want_next = true;
            } else if (want_next) {
                s3 = s; want_next = false;
            }
            prev = s;
        }
        if (kbest == -L || kbest == L) {
            st = SVI_SUBPIXEL_REJECTED;
        } else {
            const float delta = __fdiv_rn((float)(s1 - s3), 2.f * (float)(s1 + s3 - 2 * best));
            xr_new = __fadd_rn(__fadd_rn(xr_f, (float)kbest), delta);
            st = point_in_left(a.tc, xl_f, y_f, xr_new, xyz);
        }
    }
    if (lane == 0) {
        a.out.status[o] = (uint8_t)st;
        if (st == SVI_OK) {
            a.out.uv_r[o * 2] = xr_new;
            a.out.xyz[o * 3] = xyz[0]; a.out.xyz[o * 3 + 1] = xyz[1]; a.out.xyz[o * 3 + 2] = xyz[2];
        }
    }
}

}  // namespace svi
