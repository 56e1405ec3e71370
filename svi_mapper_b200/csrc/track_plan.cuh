// track_plan.cuh -- the per-landmark geometry of trackManual on the device, so that the whole cascade is one
// stream of kernels without host turn-arounds, and the detection mask of addNewLandmarks.
//
// Replaces (reference paths):
//   stage-2 search windows                      src/core/CFundamentalMatcher.cpp:1548-1575 (LEFT), :1672-1699 (RIGHT)
//   stage-3 epipolar line set-up                src/core/CFundamentalMatcher.cpp:1795-1947
//   CFundamentalMatcher::getMaskActiveLandmarks src/core/CFundamentalMatcher.cpp:2043-2073
// One thread per landmark; fp64 with every operation rounded on its own, in the order the CPU restatement
// the parity tests compare against uses -- the library is built with -fmad=false.
// Work items are compacted with an atomic counter: their order is arbitrary, every item writes only its own
// landmark's output slot, so the results do not depend on it.
#pragma once
#include "brief_match.cuh"

namespace svi {

struct TrackPlanConst {
    double T[12];          // rows 0..2 of WORLDtoLEFT
    double P[12];          // projection matrix of the side the plan is for
    double motion_scaling;
    int W, H;
    int block;             // m_uSearchBlockSizePoseOptimization = 15 (CFundamentalMatcher.h:95)
    double epi_base;       // m_dEpipolarLineBaseLength = 15 (CFundamentalMatcher.h:92)
};

__device__ __forceinline__ void world_to_camera(const double* T, const double* w, double* p) {
#pragma unroll
    for (int r = 0; r < 3; ++r)   // Isometry3d * Vector3d = linear * v + translation
        p[r] = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(T[4 * r], w[0]), __dmul_rn(T[4 * r + 1], w[1])), __dmul_rn(T[4 * r + 2], w[2])), T[4 * r + 3]);
}

// Stage-2 windows for the landmarks [q0, q1) that are still untracked: half sizes round(round(w + scaling) * 15)
// with w = sqrt|u - cx| / 10 (CPinholeCamera.h:220-227), corners clamped to the image, cv::Rect(Point2f, Point2f)
// (= cvRound of both corners), then the window grown by 4*size and clamped (:1572-1575).  plane: 0 = LEFT, 1 = RIGHT.
__global__ void stage2_plan_kernel(TrackPlanConst k, int plane, float tri_scale, LandmarksDev lm, int q0, int q1,
                                   TrackOutDev out, RoiItem* __restrict__ rois, Stage2Item* __restrict__ items,
                                   int* __restrict__ n_items) {
    const int q = q0 + blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= q1) return;
    if (out.stage[q] != 0 || out.status[q] == SVI_TRK_OUT_OF_FOV) return;
    const double w3[3] = {lm.xyz_w[3 * q], lm.xyz_w[3 * q + 1], lm.xyz_w[3 * q + 2]};
    double p[3];
    world_to_camera(k.T, w3, p);
    float u, v;
    projection_rounded(k.P, p, u, v);
    const float size = lm.size[q], half = 4.f * size;
    const double cx = k.P[2], cy = k.P[6];
    const double su = round(__dadd_rn(__ddiv_rn(__dsqrt_rn(fabs(__dsub_rn((double)u, cx))), 10.0), k.motion_scaling));
    const double sv = round(__dadd_rn(__ddiv_rn(__dsqrt_rn(fabs(__dsub_rn((double)v, cy))), 10.0), k.motion_scaling));
    const double hw = round(__dmul_rn(su, (double)k.block)), hh = round(__dmul_rn(sv, (double)k.block));
    const float ul_x = (float)fmax(__dsub_rn((double)u, hw), 0.0), ul_y = (float)fmax(__dsub_rn((double)v, hh), 0.0);
    const float lr_x = (float)fmin(__dadd_rn((double)u, hw), (double)k.W), lr_y = (float)fmin(__dadd_rn((double)v, hh), (double)k.H);
    const int rx = cv_round_f(ul_x), ry = cv_round_f(ul_y);
    const int rw = cv_round_f(lr_x) - rx, rh = cv_round_f(lr_y) - ry;
    if (rw <= 0 || rh <= 0 || rx < 0 || ry < 0 || rx + rw > k.W || ry + rh > k.H) {
        out.status[q] = SVI_TRK_NO_FEATURES;   // GFTT on an empty image finds nothing
        return;
    }
    const float g_ulx = fmaxf(__fsub_rn(ul_x, half), 0.0f), g_uly = fmaxf(__fsub_rn(ul_y, half), 0.0f);
    const float g_lrx = fminf(__fadd_rn(lr_x, half), (float)k.W), g_lry = fminf(__fadd_rn(lr_y, half), (float)k.H);
    Stage2Item it;
    it.q = q;
    it.gx = cv_round_f(g_ulx); it.gy = cv_round_f(g_uly);
    it.gw = cv_round_f(g_lrx) - it.gx; it.gh = cv_round_f(g_lry) - it.gy;
    it.ul_x = ul_x; it.ul_y = ul_y;
    it.search = __fmul_rn(tri_scale, lm.disparity[q]);
    it.size = size;
    const int slot = atomicAdd(n_items, 1);
    SVI_CHECK(4, slot >= 0 && slot < q1 - q0);
    items[slot] = it;
    rois[slot] = RoiItem{plane, rx, ry, rw, rh};
}

// ---- stage 3 geometry (:1795-1947)
__device__ __forceinline__ void mul3_dev(const double A[3][3], const double B[3][3], double C[3][3]) {
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j)
            C[i][j] = __dadd_rn(__dadd_rn(__dmul_rn(A[i][0], B[0][j]), __dmul_rn(A[i][1], B[1][j])), __dmul_rn(A[i][2], B[2][j]));
}
__device__ __forceinline__ double cof3_dev(const double m[3][3], int i, int j) {
    const int i1 = (i + 1) % 3, i2 = (i + 2) % 3, j1 = (j + 1) % 3, j2 = (j + 2) % 3;
    return __dsub_rn(__dmul_rn(m[i1][j1], m[i2][j2]), __dmul_rn(m[i1][j2], m[i2][j1]));
}

struct Stage3Extra {
    const double* uv_ref;   // [n*2] vecUVReferenceLEFT
    const double* T_det;    // [n*16] LEFTtoWORLD of the landmark's detection point
};

// Returns SVI_OK and fills `it`, or the svi_status of the failing check.
__device__ inline int epipolar_plan_dev(const TrackPlanConst& k, const double* Td, const double* uv_ref, const double* pw, Stage3Item& it) {
    const double* Tw = k.T;
    double R[3][3], t[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int j = 0; j < 3; ++j)
            R[i][j] = __dadd_rn(__dadd_rn(__dmul_rn(Tw[4 * i], Td[j]), __dmul_rn(Tw[4 * i + 1], Td[4 + j])), __dmul_rn(Tw[4 * i + 2], Td[8 + j]));
        t[i] = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(Tw[4 * i], Td[3]), __dmul_rn(Tw[4 * i + 1], Td[7])), __dmul_rn(Tw[4 * i + 2], Td[11])), Tw[4 * i + 3]);
    }
    if (!(0.0 < __dadd_rn(__dadd_rn(__dmul_rn(t[0], t[0]), __dmul_rn(t[1], t[1])), __dmul_rn(t[2], t[2])))) return SVI_EPI_NO_TRANSLATION;
    const double S[3][3] = {{0.0, -t[2], t[1]}, {t[2], 0.0, -t[0]}, {-t[1], t[0], 0.0}};   // CMiniVisionToolbox::getSkew
    double E[3][3], K[3][3], Ki[3][3], KiT[3][3], A[3][3], F[3][3];
    mul3_dev(R, S, E);                                                                      // :1800
    const double* P = k.P;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) K[i][j] = P[4 * i + j];
    {   // adjugate / determinant (Eigen's closed form for fixed 3x3)
        const double c0 = cof3_dev(K, 0, 0), c1 = cof3_dev(K, 1, 0), c2 = cof3_dev(K, 2, 0);
        const double det = __dadd_rn(__dadd_rn(__dmul_rn(c0, K[0][0]), __dmul_rn(c1, K[1][0])), __dmul_rn(c2, K[2][0]));
        const double inv_det = __ddiv_rn(1.0, det);
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) Ki[i][j] = __dmul_rn(cof3_dev(K, j, i), inv_det);
    }
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) KiT[i][j] = Ki[j][i];
    mul3_dev(KiT, E, A);
    mul3_dev(A, Ki, F);                                                                     // :1801
    double c[3];
#pragma unroll
    for (int i = 0; i < 3; ++i)
        c[i] = __dadd_rn(__dadd_rn(__dmul_rn(F[i][0], uv_ref[0]), __dmul_rn(F[i][1], uv_ref[1])), __dmul_rn(F[i][2], 1.0));   // :1818
    double p[3];
    world_to_camera(Tw, pw, p);
    float pu, pv;
    projection_rounded(P, p, pu, pv);                                                       // :1807
    if (!(pu >= 28.f && pu < (float)(k.W - 28) && pv >= 28.f && pv < (float)(k.H - 28))) return SVI_EPI_OUT_OF_SIGHT;
    const double W = (double)k.W, H = (double)k.H;
    const double half = __dmul_rn(10.0, k.motion_scaling);                                  // :1362
    const double wu = __ddiv_rn(__dsqrt_rn(fabs(__dsub_rn((double)pu, P[2]))), 10.0), wv = __ddiv_rn(__dsqrt_rn(fabs(__dsub_rn((double)pv, P[6]))), 10.0);
    const double hl_u = __dadd_rn(k.epi_base, __dmul_rn(wu, half)), hl_v = __dadd_rn(k.epi_base, __dmul_rn(wv, half));   // :1821-1822
    auto curve_v = [&](double u) { return __ddiv_rn(-__dadd_rn(__dmul_rn(c[0], u), c[2]), c[1]); };
    auto curve_u = [&](double v) { return __ddiv_rn(-__dadd_rn(__dmul_rn(c[1], v), c[2]), c[0]); };
    const double u_min_raw = fmax(__dsub_rn((double)pu, hl_u), 0.0), u_max_raw = fmin(__dadd_rn((double)pu, hl_u), W);
    const double v_min_raw = curve_v(u_min_raw), v_max_raw = curve_v(u_max_raw);
    if ((0.0 > v_min_raw && 0.0 > v_max_raw) || (H < v_min_raw && H < v_max_raw)) return SVI_EPI_VERTICAL;
    const double v_lim_min = fmax(__dsub_rn((double)pv, hl_v), 0.0), v_lim_max = fmin(__dadd_rn((double)pv, hl_v), H);
    double u_min = u_min_raw, u_max = u_max_raw, v_for_min, v_for_max;
    if (v_min_raw < v_max_raw) {
        if (v_lim_min > v_max_raw || v_lim_max < v_min_raw) return SVI_EPI_NEG_SLOPE;
        if (v_lim_min > v_min_raw) { v_for_min = v_lim_min; u_min = curve_u(v_for_min); } else v_for_min = v_min_raw;
        if (v_lim_max < v_max_raw) { v_for_max = v_lim_max; u_max = curve_u(v_for_max); } else v_for_max = v_max_raw;
    } else {
        if (v_lim_min > v_min_raw || v_lim_max < v_max_raw) return SVI_EPI_POS_SLOPE;
        if (v_lim_min > v_max_raw) { v_for_min = v_lim_min; u_max = curve_u(v_for_min); } else v_for_min = v_max_raw;
        if (v_lim_max < v_min_raw) { v_for_max = v_lim_max; u_min = curve_u(v_for_max); } else v_for_max = v_min_raw;
    }
    const double du = __dsub_rn(u_max, u_min), dv = __dsub_rn(v_for_max, v_for_min);
    // the reference converts these to uint32_t; negative / non-finite values are undefined there
    if (!(isfinite(du) && isfinite(dv)) || du < 0.0 || dv < 0.0 || du >= 65536.0 || dv >= 65536.0) return SVI_EPI_ZERO_LEN;
    const int delta_u = (int)du, delta_v = (int)dv;
    if (delta_u == 0 && delta_v == 0) return SVI_EPI_ZERO_LEN;
    it.along_u = delta_v < delta_u ? 1 : 0;
    it.count = it.along_u ? delta_u : delta_v;
    it.start = it.along_u ? u_min : v_for_min;
    it.c0 = c[0]; it.c1 = c[1]; it.c2 = c[2];
    return SVI_OK;
}

// n_dev (may be null): the item count when only the device knows it; n is then the capacity the grid covers
__global__ void stage3_plan_kernel(TrackPlanConst k, LandmarksDev lm, Stage3Extra ex, int n, const int* __restrict__ n_dev, TrackOutDev out,
                                   Stage3Item* __restrict__ items, int* __restrict__ n_items) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n || (n_dev && q >= *n_dev)) return;
    if (out.stage[q] != 0 || out.status[q] == SVI_TRK_OUT_OF_FOV) return;
    Stage3Item it;
    it.q = q;
    it.size = lm.size[q];
    it.search = (float)__dmul_rn(__dadd_rn(1.0, k.motion_scaling), (double)lm.disparity[q]);   // :2415
    double Td[16], uvr[2], pw[3];
#pragma unroll
    for (int i = 0; i < 12; ++i) Td[i] = ex.T_det[16 * (size_t)q + i];
    uvr[0] = ex.uv_ref[2 * (size_t)q]; uvr[1] = ex.uv_ref[2 * (size_t)q + 1];
    pw[0] = lm.xyz_w[3 * q]; pw[1] = lm.xyz_w[3 * q + 1]; pw[2] = lm.xyz_w[3 * q + 2];
    const int st = epipolar_plan_dev(k, Td, uvr, pw, it);
    if (st == SVI_OK) {
        const int slot = atomicAdd(n_items, 1);
        SVI_CHECK(4, slot >= 0 && slot < n);
        items[slot] = it;
    }
    else out.status[q] = (uint8_t)st;
}

// ---- getMaskActiveLandmarks (:2043-2073): the plane is 255, every centre stamps a filled radius-7 disc of zeros as
// cv::circle(mask, Point(cvRound(x), cvRound(y)), 7, 0, -1) draws it -- row widths 1,7,9,11,13,13,13,15,13,13,13,11,9,7,1
// (149 px, pinned against cv2.circle in tests/golden).  One thread per (centre, row).
__global__ void mask_fill_kernel(uint8_t* __restrict__ mask, size_t bytes) {
    const size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 16;
    if (i + 16 <= bytes) *reinterpret_cast<uint4*>(mask + i) = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
    else for (size_t j = i; j < bytes; ++j) mask[j] = 255;
}
__global__ void mask_discs_kernel(uint8_t* __restrict__ mask, int W, int H, int pitch, const float* __restrict__ centres, int n) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int c = t / 15, row = t - c * 15;
    if (c >= n) return;
    const float fx = centres[2 * c], fy = centres[2 * c + 1];
    if (!(fabsf(fx) < 1.0e6f && fabsf(fy) < 1.0e6f)) return;   // projections at infinity / NaN draw nothing
    const int cx = cv_round_f(fx), cy = cv_round_f(fy);
    const int y = cy + row - 7;
    if (y < 0 || y >= H) return;
    const int hw = row == 7 ? 7 : (row == 0 || row == 14) ? 0 : (row == 1 || row == 13) ? 3 : (row == 2 || row == 12) ? 4 : (row == 3 || row == 11) ? 5 : 6;
    const int xa = max(cx - hw, 0), xb = min(cx + hw, W - 1);
    uint8_t* r = mask + (size_t)y * pitch;
    SVI_CHECK(4, xa >= 0 && xb < W && xb < pitch);
    for (int x = xa; x <= xb; ++x) r[x] = 0;
}

}  // namespace svi
