// CSolverStereoPosit -- pose refinement from the stereo measurements of one frame, the consumer of
// CFundamentalMatcher::getPoseStereoPosit.  Same interface, constants and exceptions as the reference's
// src/optimization/CSolverStereoPosit.{h,cpp} (:8-170): robust Gauss-Newton on the four-dimensional stereo
// reprojection error with the increment (translation, quaternion vector part) of
// CMiniVisionToolbox::getTransformationFromVector (src/vision/CMiniVisionToolbox.cpp:354-377): six unknowns and a few hundred
// to a few thousand measurements per frame; written on the POD types of Types.h, no Eigen.  Constructed with a CGpuContext,
// the solve is ONE library call (svi_solve_stereo_posit: the whole iteration loop in one launch, the arithmetic below in the
// same order, bit-identical); without one, or with SVI_HOST_POSIT=cpu, the CPU loop below runs (the checker of the parity test).
#ifndef SVI_HOST_CSOLVERSTEREOPOSIT_H
#define SVI_HOST_CSOLVERSTEREOPOSIT_H

#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "CTriangulator.h"
#include "Types.h"

// Pinned arithmetic: every product and sum below rounds on its own, in the written order (the GPU kernels and the CPU
// oracle do the same), whatever flags the including project uses -- the reference builds with -O3 -march=native
// (CMakeLists.txt:51), where GCC's default -ffp-contract=fast would fuse a*b + c into an FMA.
#if defined(__clang__)
#pragma clang fp contract(off)
#elif defined(__GNUC__)
#pragma GCC push_options
#pragma GCC optimize("fp-contract=off")
#endif

class CLandmark;

class CSolverStereoPosit {
public:
    struct CMatch {   // CSolverStereoPosit.h:19-49
        CLandmark* pLandmark;
        const CPoint3DWORLD vecPointXYZWORLD;
        const CPoint3DCAMERA vecPointXYZLEFT;
        const Point2f ptUVLEFT;
        const Point2f ptUVRIGHT;
        const CDescriptor matDescriptorLEFT;
        const CDescriptor matDescriptorRIGHT;
        CMatch(CLandmark* p_pLandmark, const CPoint3DWORLD& p_vecPointXYZWORLD, const CPoint3DCAMERA& p_vecPointXYZLEFT, const Point2f& p_ptUVLEFT,
               const Point2f& p_ptUVRIGHT, const CDescriptor& p_matDescriptorLEFT, const CDescriptor& p_matDescriptorRIGHT)
            : pLandmark(p_pLandmark), vecPointXYZWORLD(p_vecPointXYZWORLD), vecPointXYZLEFT(p_vecPointXYZLEFT), ptUVLEFT(p_ptUVLEFT),
              ptUVRIGHT(p_ptUVRIGHT), matDescriptorLEFT(p_matDescriptorLEFT), matDescriptorRIGHT(p_matDescriptorRIGHT) {}
    };

    // p_pGpu: solve on the GPU; its context must have been created for the cameras of these two projection matrices (the
    // library takes them from the context)
    CSolverStereoPosit(const MatrixProjection& p_matProjectionLEFT, const MatrixProjection& p_matProjectionRIGHT,
                       const std::shared_ptr<CGpuContext> p_pGpu = nullptr)
        : m_matProjectionLEFT(p_matProjectionLEFT), m_matProjectionRIGHT(p_matProjectionRIGHT), m_pGpu(p_pGpu) {}

    // increment vector -> transform: translation t[0..2], rotation from the unit quaternion (sqrt(1-|q|^2), q)
    static Isometry3d getTransformationFromVector(const double (&t)[6]) {
        Isometry3d T;
        T(0, 3) = t[0]; T(1, 3) = t[1]; T(2, 3) = t[2];
        const double x = t[3], y = t[4], z = t[5], n2 = x * x + y * y + z * z;
        if (1.0 > n2) {
            const double w = std::sqrt(1.0 - n2);
            T(0, 0) = 1 - 2 * (y * y + z * z); T(0, 1) = 2 * (x * y - z * w);     T(0, 2) = 2 * (x * z + y * w);
            T(1, 0) = 2 * (x * y + z * w);     T(1, 1) = 1 - 2 * (x * x + z * z); T(1, 2) = 2 * (y * z - x * w);
            T(2, 0) = 2 * (x * z - y * w);     T(2, 1) = 2 * (y * z + x * w);     T(2, 2) = 1 - 2 * (x * x + y * y);
        }
        return T;
    }

    const Isometry3d getTransformationWORLDtoLEFT(const Isometry3d& p_matTransformationWORLDtoLEFTLAST, const CPoint3D& p_vecTranslationIMU,
                                                  const Isometry3d& p_matTransformationWORLDtoLEFTESTIMATE,
                                                  const std::vector<CMatch>& p_vecMeasurements) {
        static const bool bCPU = [] { const char* e = std::getenv("SVI_HOST_POSIT"); return e && std::string(e) == "cpu"; }();
        const CTimer cTimer(m_dDurationSeconds);
        m_uIterationsLAST = 0;
        if (m_pGpu && !bCPU)
            return _getTransformationWORLDtoLEFTGPU(p_matTransformationWORLDtoLEFTLAST, p_vecTranslationIMU, p_matTransformationWORLDtoLEFTESTIMATE, p_vecMeasurements);
        try {
            return _getTransformationWORLDtoLEFTCPU(p_matTransformationWORLDtoLEFTLAST, p_vecTranslationIMU, p_matTransformationWORLDtoLEFTESTIMATE, p_vecMeasurements);
        } catch (const CExceptionPoseOptimization& e) {
            m_strFailureLAST = e.what();
            throw;
        }
    }
    // iterations of the last successful solve; wall time of all solves so far (failed ones included; the solves inside
    // svi_track_frame_stereo_only are not timed on their own)
    uint32_t getIterationsLAST() const { return m_uIterationsLAST; }
    double getDurationSeconds() const { return m_dDurationSeconds; }
    // what() of the last failed solve ("" while none has failed)
    const std::string& getFailureLAST() const { return m_strFailureLAST; }

    // The accounting of the solves that ran inside svi_track_frame_stereo_only, in their order, as the separate solves leave it:
    // the text of every failed one (the last stays), the iterations of a successful last one.
    void recordAttempts(const svi_sv_frame_result& p_cResult) {
        m_uIterationsLAST = 0;
        for (int a = 0; a < p_cResult.attempts && a < 2; ++a) {
            const svi_posit_result& cAttempt = p_cResult.attempt[a];
            if (SVI_POSIT_OK == cAttempt.outcome) m_uIterationsLAST = (uint32_t)cAttempt.iterations;
            else m_strFailureLAST = getFailureText(cAttempt, (size_t)p_cResult.measurements[a]);
        }
    }
    // the reference's exception text for a failed outcome of the library
    static std::string getFailureText(const svi_posit_result& p_cResult, const size_t p_uNumberOfMeasurements) {
        switch (p_cResult.outcome) {
            case SVI_POSIT_TOO_FEW_POINTS: return "insufficient number of points: " + std::to_string(p_uNumberOfMeasurements);
            case SVI_POSIT_INACCURATE:
                return "insufficient accuracy (average error: " + std::to_string(p_cResult.average_squared_error) + " inliers: " +
                       std::to_string((size_t)p_cResult.inliers) + ")";
            case SVI_POSIT_HIGH_RISK: return "inconsistent with prior (HIGH RISK: " + std::to_string(p_cResult.risk) + ")";
            default: return "system did not converge";
        }
    }

private:
    struct CTimer {
        double& dTotal;
        const std::chrono::steady_clock::time_point tStart = std::chrono::steady_clock::now();
        explicit CTimer(double& p_dTotal) : dTotal(p_dTotal) {}
        ~CTimer() { dTotal += std::chrono::duration<double>(std::chrono::steady_clock::now() - tStart).count(); }
    };

    // svi_solve_stereo_posit: the loop below on the device, the exceptions rebuilt from the numbers it returns
    const Isometry3d _getTransformationWORLDtoLEFTGPU(const Isometry3d& p_matTransformationWORLDtoLEFTLAST, const CPoint3D& p_vecTranslationIMU,
                                                      const Isometry3d& p_matTransformationWORLDtoLEFTESTIMATE,
                                                      const std::vector<CMatch>& p_vecMeasurements) {
        const size_t uNumberOfMeasurements = p_vecMeasurements.size();
        m_vecXYZWORLD.resize(3 * uNumberOfMeasurements);
        m_vecUVLEFT.resize(2 * uNumberOfMeasurements);
        m_vecUVRIGHT.resize(2 * uNumberOfMeasurements);
        for (size_t u = 0; u < uNumberOfMeasurements; ++u) {
            const CMatch& cMatch = p_vecMeasurements[u];
            for (int k = 0; k < 3; ++k) m_vecXYZWORLD[3 * u + k] = cMatch.vecPointXYZWORLD.v[k];
            m_vecUVLEFT[2 * u] = cMatch.ptUVLEFT.x; m_vecUVLEFT[2 * u + 1] = cMatch.ptUVLEFT.y;
            m_vecUVRIGHT[2 * u] = cMatch.ptUVRIGHT.x; m_vecUVRIGHT[2 * u + 1] = cMatch.ptUVRIGHT.y;
        }
        svi_posit_problem cIn{};
        cIn.n = (int32_t)uNumberOfMeasurements;
        cIn.xyz_world = m_vecXYZWORLD.data();
        cIn.uv_left = m_vecUVLEFT.data();
        cIn.uv_right = m_vecUVRIGHT.data();
        std::memcpy(cIn.T_estimate, p_matTransformationWORLDtoLEFTESTIMATE.m, sizeof(cIn.T_estimate));
        std::memcpy(cIn.T_last, p_matTransformationWORLDtoLEFTLAST.m, sizeof(cIn.T_last));
        for (int r = 0; r < 3; ++r) cIn.t_imu[r] = p_vecTranslationIMU(r);
        svi_posit_result cOut;
        m_pGpu->check(svi_solve_stereo_posit(m_pGpu->ctx, &cIn, &cOut));
        if (SVI_POSIT_OK != cOut.outcome) {
            m_strFailureLAST = getFailureText(cOut, uNumberOfMeasurements);
            throw CExceptionPoseOptimization(m_strFailureLAST);
        }
        m_uIterationsLAST = (uint32_t)cOut.iterations;
        Isometry3d T;
        std::memcpy(T.m, cOut.T_world_to_left, sizeof(T.m));
        return T;
    }

    const Isometry3d _getTransformationWORLDtoLEFTCPU(const Isometry3d& p_matTransformationWORLDtoLEFTLAST, const CPoint3D& p_vecTranslationIMU,
                                                      const Isometry3d& p_matTransformationWORLDtoLEFTESTIMATE,
                                                      const std::vector<CMatch>& p_vecMeasurements) {
        const size_t uNumberOfMeasurements = p_vecMeasurements.size();
        if (!(m_uMinimumPointsForPoseOptimization < uNumberOfMeasurements))
            throw CExceptionPoseOptimization("insufficient number of points: " + std::to_string(uNumberOfMeasurements));
        Isometry3d T(p_matTransformationWORLDtoLEFTESTIMATE);
        double dErrorPrevious = 0.0;
        for (uint32_t uLS = 0; uLS < m_uCapIterationsPoseOptimization; ++uLS) {
            double H[6][6] = {{0}}, b[6] = {0}, dErrorTotal = 0.0;
            size_t uInliers = 0;
            for (const CMatch& cMatch : p_vecMeasurements) {
                const CPoint3D p(T * cMatch.vecPointXYZWORLD);
                if (!(0.0 < p.z())) continue;
                double aL[3], aR[3];
                for (int r = 0; r < 3; ++r) {
                    aL[r] = m_matProjectionLEFT(r, 0) * p.x() + m_matProjectionLEFT(r, 1) * p.y() + m_matProjectionLEFT(r, 2) * p.z() + m_matProjectionLEFT(r, 3);
                    aR[r] = m_matProjectionRIGHT(r, 0) * p.x() + m_matProjectionRIGHT(r, 1) * p.y() + m_matProjectionRIGHT(r, 2) * p.z() + m_matProjectionRIGHT(r, 3);
                }
                const double cL = aL[2], cR = aR[2];
                const double e[4] = {aL[0] / cL - cMatch.ptUVLEFT.x, aL[1] / cL - cMatch.ptUVLEFT.y, aR[0] / cR - cMatch.ptUVRIGHT.x, aR[1] / cR - cMatch.ptUVRIGHT.y};
                const double e2 = e[0] * e[0] + e[1] * e[1] + e[2] * e[2] + e[3] * e[3];
                double w = 1.0;
                if (m_dMaximumErrorInlierPixelsL2 < e2) w = m_dMaximumErrorInlierPixelsL2 / e2;
                else ++uInliers;
                dErrorTotal += w * e2;
                // d(point)/d(increment) = [ I | -2 skew(p) ] (4th homogeneous row is zero)
                const double Jt[3][6] = {{1, 0, 0, 0, 2 * p.z(), -2 * p.y()}, {0, 1, 0, -2 * p.z(), 0, 2 * p.x()}, {0, 0, 1, 2 * p.y(), -2 * p.x(), 0}};
                double J[4][6];
                fillRows(m_matProjectionLEFT, aL, cL, Jt, J[0], J[1]);
                fillRows(m_matProjectionRIGHT, aR, cR, Jt, J[2], J[3]);
                for (int i = 0; i < 6; ++i) {
                    for (int j = 0; j < 6; ++j) H[i][j] += w * (J[0][i] * J[0][j] + J[1][i] * J[1][j] + J[2][i] * J[2][j] + J[3][i] * J[3][j]);
                    b[i] += w * (J[0][i] * e[0] + J[1][i] * e[1] + J[2][i] * e[2] + J[3][i] * e[3]);
                }
            }
            double dx[6];
            solveSymmetric(H, b, dx);
            T = getTransformationFromVector(dx) * T;
            // enforce rotation symmetry: R -= 0.5 * R * (R^T R - I)
            double RtR[3][3];
            for (int i = 0; i < 3; ++i)
                for (int j = 0; j < 3; ++j) RtR[i][j] = T(0, i) * T(0, j) + T(1, i) * T(1, j) + T(2, i) * T(2, j) - (i == j ? 1.0 : 0.0);
            double R[3][3];
            for (int i = 0; i < 3; ++i)
                for (int j = 0; j < 3; ++j) R[i][j] = T(i, j) - 0.5 * (T(i, 0) * RtR[0][j] + T(i, 1) * RtR[1][j] + T(i, 2) * RtR[2][j]);
            for (int i = 0; i < 3; ++i)
                for (int j = 0; j < 3; ++j) T(i, j) = R[i][j];
            if (m_dConvergenceDelta > std::fabs(dErrorPrevious - dErrorTotal)) {
                const double dErrorAverage = dErrorTotal / uNumberOfMeasurements;
                if (m_dMaximumErrorAveragePixelsL2 < dErrorAverage && m_uMinimumInliersPoseOptimization > uInliers)
                    throw CExceptionPoseOptimization("insufficient accuracy (average error: " + std::to_string(dErrorAverage) + " inliers: " + std::to_string(uInliers) + ")");
                double d2 = 0.0;
                for (int r = 0; r < 3; ++r) { const double d = T(r, 3) - p_matTransformationWORLDtoLEFTLAST(r, 3); d2 += d * d; }
                if (m_dMinimumTranslationMetersL2 > d2)
                    for (int r = 0; r < 3; ++r) T(r, 3) = p_matTransformationWORLDtoLEFTLAST(r, 3);   // don't integrate the translational part
                const Isometry3d Tinv(inverseIsometry(T)), TestInv(inverseIsometry(p_matTransformationWORLDtoLEFTESTIMATE));
                double dRisk = 0.0;
                for (int r = 0; r < 3; ++r) { const double d = Tinv(r, 3) - TestInv(r, 3) - p_vecTranslationIMU(r); dRisk += d * d; }
                if (m_dMaximumRISK < dRisk) throw CExceptionPoseOptimization("inconsistent with prior (HIGH RISK: " + std::to_string(dRisk) + ")");
                m_uIterationsLAST = uLS + 1;
                return T;
            }
            dErrorPrevious = dErrorTotal;
        }
        throw CExceptionPoseOptimization("system did not converge");
    }

    // rows of (d(u,v)/d(abc)) * P * Jt for one camera
    static void fillRows(const MatrixProjection& P, const double (&a)[3], double c, const double (&Jt)[3][6], double* rowU, double* rowV) {
        for (int k = 0; k < 6; ++k) {
            double PJ[3];
            for (int r = 0; r < 3; ++r) PJ[r] = P(r, 0) * Jt[0][k] + P(r, 1) * Jt[1][k] + P(r, 2) * Jt[2][k];
            rowU[k] = PJ[0] / c - a[0] / (c * c) * PJ[2];
            rowV[k] = PJ[1] / c - a[1] / (c * c) * PJ[2];
        }
    }
    // H x = -b for the symmetric 6x6 normal matrix: Gaussian elimination with partial pivoting
    static void solveSymmetric(const double (&H)[6][6], const double (&b)[6], double (&x)[6]) {
        double A[6][7];
        for (int i = 0; i < 6; ++i) { for (int j = 0; j < 6; ++j) A[i][j] = H[i][j]; A[i][6] = -b[i]; }
        for (int c = 0; c < 6; ++c) {
            int piv = c;
            for (int r = c + 1; r < 6; ++r) if (std::fabs(A[r][c]) > std::fabs(A[piv][c])) piv = r;
            if (piv != c) for (int j = 0; j < 7; ++j) std::swap(A[c][j], A[piv][j]);
            for (int r = c + 1; r < 6; ++r) {
                const double f = A[r][c] / A[c][c];
                for (int j = c; j < 7; ++j) A[r][j] -= f * A[c][j];
            }
        }
        for (int r = 5; r >= 0; --r) {
            double s = A[r][6];
            for (int j = r + 1; j < 6; ++j) s -= A[r][j] * x[j];
            x[r] = s / A[r][r];
        }
    }

    const MatrixProjection m_matProjectionLEFT, m_matProjectionRIGHT;
    const std::shared_ptr<CGpuContext> m_pGpu;
    std::vector<double> m_vecXYZWORLD;   // staging of the GPU call (kept between frames: no allocation once grown)
    std::vector<float> m_vecUVLEFT, m_vecUVRIGHT;
    uint32_t m_uIterationsLAST = 0;
    double m_dDurationSeconds = 0.0;
    std::string m_strFailureLAST;
    const uint32_t m_uMinimumPointsForPoseOptimization = 25;   // CSolverStereoPosit.h:89-99
    const uint32_t m_uMinimumInliersPoseOptimization = 15;
    const uint32_t m_uCapIterationsPoseOptimization = 1000;
    const double m_dMaximumErrorInlierPixelsL2 = 10.0;
    const double m_dMaximumErrorAveragePixelsL2 = 9.0;
    const double m_dMaximumRISK = 2.0;
    const double m_dConvergenceDelta = 1e-5;
    const double m_dMinimumTranslationMetersL2 = 0.001;
};

#if defined(__GNUC__) && !defined(__clang__)
#pragma GCC pop_options
#endif
#endif
