// posit.cuh -- CSolverStereoPosit::getTransformationWORLDtoLEFT for one frame's stereo measurements in one launch.
//
// Replaces the per-frame CPU loop of the pose solve (reference src/optimization/CSolverStereoPosit.cpp:8-170, fed by
// CFundamentalMatcher::getPoseStereoPosit): robust Gauss-Newton on the four-dimensional stereo re-projection error of the
// WORLD->LEFT pose, six unknowns (translation, quaternion vector part of CMiniVisionToolbox::getTransformationFromVector),
// weights above m_dMaximumErrorInlierPixelsL2, at most 1000 iterations, convergence 1e-5 on the total weighted error, then the
// accuracy test, the translation clamp and the risk test against the prior.  The whole iteration loop runs inside the kernel.
// fp64, every operation rounded on its own (the library is built with -fmad=false), the host's operation order everywhere and
// every sum in measurement order: the result is bit-identical to the C++ host implementation of the same loop
// (svi_mapper_b200/host/CSolverStereoPosit.h), which the parity test uses as its checker.
#pragma once
#include "common.cuh"

namespace svi {

// CSolverStereoPosit.h:89-99
constexpr uint32_t kPositCapIterations = 1000;
constexpr uint32_t kPositMinimumInliers = 15;
constexpr double kPositMaximumErrorInlierPixelsL2 = 10.0;
constexpr double kPositMaximumErrorAveragePixelsL2 = 9.0;
constexpr double kPositMaximumRisk = 2.0;
constexpr double kPositConvergenceDelta = 1e-5;
constexpr double kPositMinimumTranslationMetersL2 = 0.001;
constexpr int kPositMinimumPoints = 25;   // solve when MORE than this many measurements exist

struct PositIn {
    const double* xyz_world;   // n x 3
    const float* uv_left;      // n x 2
    const float* uv_right;     // n x 2
    double P_left[12], P_right[12];   // row-major 3 x 4
    double T_estimate[16], T_last[16];  // row-major 4 x 4
    double t_imu[3];
};
struct PositOut {
    double T[16];
    double average_squared_error, risk;
    int iterations, inliers, outcome;   // outcome = svi_posit_outcome of include/svi_gpu.h
};

// ---- the host's Isometry3d / solver helpers, same operation order (host/Types.h, host/CSolverStereoPosit.h)
__device__ __forceinline__ void posit_from_vector(const double (&t)[6], double (&T)[16]) {
#pragma unroll
    for (int k = 0; k < 16; ++k) T[k] = (k % 5 == 0) ? 1.0 : 0.0;
    T[3] = t[0]; T[7] = t[1]; T[11] = t[2];
    const double x = t[3], y = t[4], z = t[5], n2 = x * x + y * y + z * z;
    if (1.0 > n2) {
        const double w = sqrt(1.0 - n2);
        T[0] = 1 - 2 * (y * y + z * z); T[1] = 2 * (x * y - z * w);     T[2] = 2 * (x * z + y * w);
        T[4] = 2 * (x * y + z * w);     T[5] = 1 - 2 * (x * x + z * z); T[6] = 2 * (y * z - x * w);
        T[8] = 2 * (x * z - y * w);     T[9] = 2 * (y * z + x * w);     T[10] = 1 - 2 * (x * x + y * y);
    }
}

// C = A * B for two isometries (operator*(Isometry3d, Isometry3d)): the bottom row of C stays (0 0 0 1)
__device__ __forceinline__ void posit_compose(const double (&A)[16], const double (&B)[16], double (&C)[16]) {
#pragma unroll
    for (int k = 0; k < 16; ++k) C[k] = (k % 5 == 0) ? 1.0 : 0.0;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < 3; ++k) s += A[4 * r + k] * B[4 * k + c];
            C[4 * r + c] = s + (c == 3 ? A[4 * r + 3] : 0.0);
        }
    }
}

// translation column of inverseIsometry(T): -(R^T t)
__device__ __forceinline__ void posit_inverse_translation(const double (&T)[16], double (&ti)[3]) {
#pragma unroll
    for (int r = 0; r < 3; ++r) ti[r] = -(T[r] * T[3] + T[4 + r] * T[7] + T[8 + r] * T[11]);
}

// rows of (d(u,v)/d(abc)) * P * Jt for one camera (fillRows)
__device__ __forceinline__ void posit_fill_rows(const double* P, const double (&a)[3], double c, const double (&Jt)[3][6], double* rowU, double* rowV) {
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        double PJ[3];
#pragma unroll
        for (int r = 0; r < 3; ++r) PJ[r] = P[4 * r] * Jt[0][k] + P[4 * r + 1] * Jt[1][k] + P[4 * r + 2] * Jt[2][k];
        rowU[k] = PJ[0] / c - a[0] / (c * c) * PJ[2];
        rowV[k] = PJ[1] / c - a[1] / (c * c) * PJ[2];
    }
}

// H x = -b: Gaussian elimination with partial pivoting (solveSymmetric)
__device__ __forceinline__ void posit_solve(const double (&H)[6][6], const double (&b)[6], double (&x)[6]) {
    double A[6][7];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
#pragma unroll
        for (int j = 0; j < 6; ++j) A[i][j] = H[i][j];
        A[i][6] = -b[i];
    }
#pragma unroll
    for (int c = 0; c < 6; ++c) {
        int piv = c;
        double best = fabs(A[c][c]);   // == fabs(A[piv][c]) throughout: the host's comparison without a run-time row index
#pragma unroll
        for (int r = c + 1; r < 6; ++r) { const double v = fabs(A[r][c]); if (v > best) { piv = r; best = v; } }
#pragma unroll
        for (int r = c + 1; r < 6; ++r) {   // std::swap of rows c and piv, by selects: A stays in registers
            const bool sw = r == piv;
#pragma unroll
            for (int j = 0; j < 7; ++j) { const double u = A[c][j], v = A[r][j]; A[c][j] = sw ? v : u; A[r][j] = sw ? u : v; }
        }
#pragma unroll
        for (int r = c + 1; r < 6; ++r) {
            const double f = A[r][c] / A[c][c];
#pragma unroll
            for (int j = c; j < 7; ++j) A[r][j] -= f * A[c][j];
        }
    }
#pragma unroll
    for (int r = 5; r >= 0; --r) {
        double s = A[r][6];
#pragma unroll
        for (int j = r + 1; j < 6; ++j) s -= A[r][j] * x[j];
        x[r] = s / A[r][r];
    }
}

// One CTA per solve.  An iteration walks the measurements in chunks of kPositThreads: thread t evaluates measurement c0 + t
// (transform, both projections, error, robust weight, the 4 x 6 Jacobian) and parks its 28 contributions -- the 21 distinct
// entries of the symmetric w * J^T J (J_i * J_j == J_j * J_i: the host's full 6 x 6 sum is symmetric bit for bit), the six of
// w * J^T e and w * e^2 -- in shared memory; then thread j < 28 adds contribution j of the chunk's measurements to its
// accumulator IN MEASUREMENT ORDER, skipping measurements behind the camera, which is exactly the sequence of additions the
// host loop performs on that entry.  Inliers are counted by the barrier that closes the chunk.  Thread 0 solves the 6 x 6
// system, updates and re-orthonormalises the pose and runs the convergence / accuracy / clamp / risk tests; the pose lives
// in shared memory.  optimize_landmarks_kernel uses the same scheme with a warp in place of the CTA.
constexpr int kPositThreads = 256;
constexpr int kPositTerms = 28;
constexpr int kPositTermPitch = 29;   // doubles per measurement slot: odd pitch, parked rows do not collide on one bank
constexpr size_t kPositSmemBytes = sizeof(double) * kPositThreads * kPositTermPitch;   // dynamic: the term slots

__global__ void __launch_bounds__(kPositThreads)
stereo_posit_kernel(PositIn in, int n, PositOut* out) {
    extern __shared__ double s_term[];          // [kPositThreads][kPositTermPitch]
    __shared__ double s_T[16];                  // current pose WORLD->LEFT
    __shared__ double s_sum[kPositTerms];       // H upper triangle row by row | b | total error
    __shared__ uint8_t s_valid[kPositThreads];  // measurement in front of the camera: its terms are summed
    __shared__ int s_state;                     // -1: iterate on, else the outcome
    const int tid = threadIdx.x;
    if (tid < 16) s_T[tid] = in.T_estimate[tid];
    if (tid == 0) s_state = -1;
    __syncthreads();
    double err_prev = 0.0;   // thread 0's
    for (uint32_t it = 0; it < kPositCapIterations; ++it) {
        double acc = 0.0;    // thread j < 28: entry j
        int inliers = 0;
        double T[12];
#pragma unroll
        for (int k = 0; k < 12; ++k) T[k] = s_T[k];
        for (int c0 = 0; c0 < n; c0 += kPositThreads) {
            const int m = c0 + tid;
            bool valid = false, inlier = false;
            if (m < n) {
                SVI_CHECK(10, m >= 0 && m < n);
                const double X = in.xyz_world[3 * (size_t)m], Y = in.xyz_world[3 * (size_t)m + 1], Z = in.xyz_world[3 * (size_t)m + 2];
                const double p[3] = {T[0] * X + T[1] * Y + T[2] * Z + T[3], T[4] * X + T[5] * Y + T[6] * Z + T[7],
                                     T[8] * X + T[9] * Y + T[10] * Z + T[11]};
                if (0.0 < p[2]) {
                    valid = true;
                    double aL[3], aR[3];
#pragma unroll
                    for (int r = 0; r < 3; ++r) {
                        aL[r] = in.P_left[4 * r] * p[0] + in.P_left[4 * r + 1] * p[1] + in.P_left[4 * r + 2] * p[2] + in.P_left[4 * r + 3];
                        aR[r] = in.P_right[4 * r] * p[0] + in.P_right[4 * r + 1] * p[1] + in.P_right[4 * r + 2] * p[2] + in.P_right[4 * r + 3];
                    }
                    const double cL = aL[2], cR = aR[2];
                    const double e[4] = {aL[0] / cL - (double)in.uv_left[2 * (size_t)m], aL[1] / cL - (double)in.uv_left[2 * (size_t)m + 1],
                                         aR[0] / cR - (double)in.uv_right[2 * (size_t)m], aR[1] / cR - (double)in.uv_right[2 * (size_t)m + 1]};
                    const double e2 = e[0] * e[0] + e[1] * e[1] + e[2] * e[2] + e[3] * e[3];
                    double w = 1.0;
                    if (kPositMaximumErrorInlierPixelsL2 < e2) w = kPositMaximumErrorInlierPixelsL2 / e2;
                    else inlier = true;
                    const double Jt[3][6] = {{1, 0, 0, 0, 2 * p[2], -2 * p[1]}, {0, 1, 0, -2 * p[2], 0, 2 * p[0]}, {0, 0, 1, 2 * p[1], -2 * p[0], 0}};
                    double J[4][6];
                    posit_fill_rows(in.P_left, aL, cL, Jt, J[0], J[1]);
                    posit_fill_rows(in.P_right, aR, cR, Jt, J[2], J[3]);
                    SVI_CHECK(10, tid >= 0 && tid < kPositThreads);
                    double* term = s_term + (size_t)tid * kPositTermPitch;
                    int t = 0;
#pragma unroll
                    for (int i = 0; i < 6; ++i)
#pragma unroll
                        for (int j = i; j < 6; ++j) term[t++] = w * (J[0][i] * J[0][j] + J[1][i] * J[1][j] + J[2][i] * J[2][j] + J[3][i] * J[3][j]);
#pragma unroll
                    for (int i = 0; i < 6; ++i) term[21 + i] = w * (J[0][i] * e[0] + J[1][i] * e[1] + J[2][i] * e[2] + J[3][i] * e[3]);
                    term[27] = w * e2;
                }
            }
            SVI_CHECK(10, tid < kPositThreads);
            s_valid[tid] = valid ? 1 : 0;
            inliers += __syncthreads_count(inlier);   // also the barrier behind the parked terms
            const int cnt = min(kPositThreads, n - c0);
            if (tid < kPositTerms)
                for (int k = 0; k < cnt; ++k) {   // in measurement order
                    SVI_CHECK(10, k < kPositThreads && k * kPositTermPitch + tid < kPositThreads * kPositTermPitch);
                    if (s_valid[k]) acc += s_term[k * kPositTermPitch + tid];
                }
            __syncthreads();
        }
        SVI_CHECK(10, kPositTerms <= kPositThreads);
        if (tid < kPositTerms) s_sum[tid] = acc;
        __syncthreads();
        if (tid == 0) {
            double H[6][6], b[6];
            int t = 0;
#pragma unroll
            for (int i = 0; i < 6; ++i)
#pragma unroll
                for (int j = i; j < 6; ++j) { H[i][j] = s_sum[t]; H[j][i] = s_sum[t]; ++t; }
#pragma unroll
            for (int i = 0; i < 6; ++i) b[i] = s_sum[21 + i];
            const double err_total = s_sum[27];
            double dx[6], D[16], Tcur[16], Tn[16];
            posit_solve(H, b, dx);
            posit_from_vector(dx, D);
#pragma unroll
            for (int k = 0; k < 16; ++k) Tcur[k] = s_T[k];
            posit_compose(D, Tcur, Tn);
            // enforce rotation symmetry: R -= 0.5 * R * (R^T R - I)
            double RtR[3][3], R[3][3];
#pragma unroll
            for (int i = 0; i < 3; ++i)
#pragma unroll
                for (int j = 0; j < 3; ++j) RtR[i][j] = Tn[i] * Tn[j] + Tn[4 + i] * Tn[4 + j] + Tn[8 + i] * Tn[8 + j] - (i == j ? 1.0 : 0.0);
#pragma unroll
            for (int i = 0; i < 3; ++i)
#pragma unroll
                for (int j = 0; j < 3; ++j) R[i][j] = Tn[4 * i + j] - 0.5 * (Tn[4 * i] * RtR[0][j] + Tn[4 * i + 1] * RtR[1][j] + Tn[4 * i + 2] * RtR[2][j]);
#pragma unroll
            for (int i = 0; i < 3; ++i)
#pragma unroll
                for (int j = 0; j < 3; ++j) Tn[4 * i + j] = R[i][j];
            out->iterations = (int)it + 1;
            out->inliers = inliers;
            if (kPositConvergenceDelta > fabs(err_prev - err_total)) {
                const double err_avg = err_total / (double)n;
                out->average_squared_error = err_avg;
                if (kPositMaximumErrorAveragePixelsL2 < err_avg && kPositMinimumInliers > (uint32_t)inliers) {
                    s_state = 2;   // SVI_POSIT_INACCURATE
                } else {
                    double d2 = 0.0;
#pragma unroll
                    for (int r = 0; r < 3; ++r) { const double d = Tn[4 * r + 3] - in.T_last[4 * r + 3]; d2 += d * d; }
                    if (kPositMinimumTranslationMetersL2 > d2)
#pragma unroll
                        for (int r = 0; r < 3; ++r) Tn[4 * r + 3] = in.T_last[4 * r + 3];   // don't integrate the translational part
                    double ti[3], te[3];
                    posit_inverse_translation(Tn, ti);
                    posit_inverse_translation(in.T_estimate, te);
                    double risk = 0.0;
#pragma unroll
                    for (int r = 0; r < 3; ++r) { const double d = ti[r] - te[r] - in.t_imu[r]; risk += d * d; }
                    out->risk = risk;
                    s_state = (kPositMaximumRisk < risk) ? 3 : 0;   // SVI_POSIT_HIGH_RISK : SVI_POSIT_OK
                }
            } else if (it + 1 == kPositCapIterations) {
                s_state = 4;   // SVI_POSIT_NOT_CONVERGED
            }
            err_prev = err_total;
#pragma unroll
            for (int k = 0; k < 16; ++k) s_T[k] = Tn[k];
        }
        __syncthreads();
        if (s_state >= 0) break;
    }
    if (tid == 0) {
        const bool ok = s_state == 0;
#pragma unroll
        for (int k = 0; k < 16; ++k) out->T[k] = ok ? s_T[k] : in.T_estimate[k];
        out->outcome = s_state;
    }
}

}  // namespace svi
