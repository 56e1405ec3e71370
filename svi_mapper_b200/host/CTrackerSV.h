// CTrackerSV -- the per-frame orchestration of the reference's stereo-only tracker (src/core/CTrackerSV.cpp:143-172 process,
// :234-552 _trackLandmarks) reduced to the calls that touch the stereo front-end and the pose: constant-velocity pose
// prior, getPoseStereoPosit with the reference's two-step fallback (raw prior, then the rotation-only "damped" prior, then
// the prior itself), trackEpipolar for what the pose stage did not see, landmark optimisation every tenth frame, the
// new-landmark trigger and addNewLandmarks.  Display, key-framing, loop closing (DBoW2 / BTree) and g2o are the reference's
// CPU side and are not part of this host layer.
#ifndef SVI_HOST_CTRACKERSV_H
#define SVI_HOST_CTRACKERSV_H

#include <chrono>

#include "CFundamentalMatcher.h"

// Pinned arithmetic: every product and sum below rounds on its own, in the written order (the GPU kernels and the CPU
// oracle do the same), whatever flags the including project uses -- the reference builds with -O3 -march=native
// (CMakeLists.txt:51), where GCC's default -ffp-contract=fast would fuse a*b + c into an FMA.
#if defined(__clang__)
#pragma clang fp contract(off)
#elif defined(__GNUC__)
#pragma GCC push_options
#pragma GCC optimize("fp-contract=off")
#endif

// cv::Rodrigues(R) for the motion-scaling term: rotation vector (axis * angle) of a rotation matrix
inline CPoint3D toOrientationRodrigues(const Isometry3d& T) {
    const double dTrace = T(0, 0) + T(1, 1) + T(2, 2);
    const double dCos = std::min(1.0, std::max(-1.0, (dTrace - 1.0) / 2.0));
    const double dAngle = std::acos(dCos);
    const double rx = T(2, 1) - T(1, 2), ry = T(0, 2) - T(2, 0), rz = T(1, 0) - T(0, 1);
    const double dSin2 = std::sqrt(rx * rx + ry * ry + rz * rz);   // 2 sin(angle)
    if (dSin2 < 1e-12) return CPoint3D(0.0, 0.0, 0.0);             // identity (the half-turn case does not occur between frames)
    const double k = dAngle / dSin2;
    return CPoint3D(k * rx, k * ry, k * rz);
}

class CTrackerSV {
public:
    CTrackerSV(const std::shared_ptr<CStereoCamera> p_pCameraSTEREO, const std::shared_ptr<CGpuContext> p_pGpu)
        : m_cMatcher(p_pCameraSTEREO, p_pGpu) {}

    // process :143-172 + _trackLandmarks :234-552 (no IMU: linear acceleration and angular velocity are zero in the SV tracker)
    void process(const ImageView& p_matImageLEFT, const ImageView& p_matImageRIGHT) {
        Isometry3d matRotationOnlyLEFTLASTtoLEFTNOW(m_matTransformationLEFTLASTtoLEFTNOW);
        for (int r = 0; r < 3; ++r) matRotationOnlyLEFTLASTtoLEFTNOW(r, 3) = 0.0;
        const CPoint3D vecRotationTotal(toOrientationRodrigues(m_matTransformationLEFTLASTtoLEFTNOW));
        const CPoint3D vecTranslationTotal(m_matTransformationLEFTLASTtoLEFTNOW(0, 3), m_matTransformationLEFTLASTtoLEFTNOW(1, 3),
                                           m_matTransformationLEFTLASTtoLEFTNOW(2, 3));
        const Isometry3d matEstimate(m_matTransformationLEFTLASTtoLEFTNOW * m_matTransformationWORLDtoLEFTLAST);
        const Isometry3d matEstimateParallel(matRotationOnlyLEFTLASTtoLEFTNOW * m_matTransformationWORLDtoLEFTLAST);
        auto norm = [](const CPoint3D& v) { return std::sqrt(v.x() * v.x() + v.y() * v.y() + v.z() * v.z()); };
        const double dMotionScaling = std::min(1.0 + (10.0 * norm(vecRotationTotal) + 0.5 * norm(vecTranslationTotal)), 5.0);   // :254

        const auto tStart = std::chrono::steady_clock::now();
        m_cMatcher.resetVisibilityActiveLandmarks();                                                                           // :257
        Isometry3d matTransformationWORLDtoLEFT(matEstimate);
        m_strPoseSource = "posit";
        try {
            matTransformationWORLDtoLEFT = m_cMatcher.getPoseStereoPosit(m_uFrameCount, p_matImageLEFT, p_matImageRIGHT, matEstimate,
                                                                         m_matTransformationWORLDtoLEFTLAST, vecRotationTotal, vecTranslationTotal,
                                                                         dMotionScaling);                                      // :268-279
            if (0 < m_uCountInstability) --m_uCountInstability;
        } catch (const CExceptionPoseOptimization&) {
            try {
                m_strPoseSource = "posit-damped";
                matTransformationWORLDtoLEFT = m_cMatcher.getPoseStereoPosit(m_uFrameCount, p_matImageLEFT, p_matImageRIGHT, matEstimateParallel,
                                                                             m_matTransformationWORLDtoLEFTLAST, vecRotationTotal,
                                                                             vecTranslationTotal, dMotionScaling);             // :291-302
            } catch (const CExceptionPoseOptimization&) {
                if (20 > m_uCountInstability) m_uCountInstability += 5;
                m_strPoseSource = "prior";
                matTransformationWORLDtoLEFT = matEstimateParallel;                                                            // :313
            }
        }
        const auto tPose = std::chrono::steady_clock::now();
        const Isometry3d matTransformationLEFTtoWORLD(inverseIsometry(matTransformationWORLDtoLEFT));
        m_cMatcher.trackEpipolar(m_uFrameCount, p_matImageLEFT, p_matImageRIGHT, matTransformationWORLDtoLEFT, matTransformationLEFTtoWORLD,
                                 dMotionScaling);                                                                              // :320-327
        const int64_t iVisible = (int64_t)m_cMatcher.getNumberOfVisibleLandmarks();
        if (0 < m_uNumberofVisibleLandmarksLAST &&
            0.75 < (double)((int64_t)m_uNumberofVisibleLandmarksLAST - iVisible) / (double)m_uNumberofVisibleLandmarksLAST && 20 > m_uCountInstability)
            m_uCountInstability += 5;                                                                                          // :333-349
        m_uNumberofVisibleLandmarksLAST = (uint64_t)iVisible;
        const auto tEpipolar = std::chrono::steady_clock::now();
        if (0 == m_uFrameCount % m_uLandmarkOptimizationEveryNFrames) m_cMatcher.optimizeActiveLandmarks(m_uFrameCount);       // :362-365
        const auto tOptimized = std::chrono::steady_clock::now();
        if (m_uVisibleLandmarksMinimum > m_uNumberofVisibleLandmarksLAST || m_uMaximumNumberOfFramesWithoutDetection < m_uNumberOfFramesWithoutDetection) {
            m_uNumberofVisibleLandmarksLAST = m_cMatcher.addNewLandmarks(p_matImageLEFT, p_matImageRIGHT, matTransformationWORLDtoLEFT,
                                                                         matTransformationLEFTtoWORLD, m_uFrameCount);         // :468-473
            m_uNumberOfFramesWithoutDetection = 0;
            ++m_uNumberOfDetections;
        } else {
            ++m_uNumberOfFramesWithoutDetection;
        }
        // the reference keeps such timers too (m_dDurationTotalSeconds*), see CTrackerGT
        const auto tEnd = std::chrono::steady_clock::now();
        m_dDurationPoseSeconds += std::chrono::duration<double>(tPose - tStart).count();
        m_dDurationTrackEpipolarSeconds += std::chrono::duration<double>(tEpipolar - tPose).count();
        m_dDurationOptimizationSeconds += std::chrono::duration<double>(tOptimized - tEpipolar).count();
        m_dDurationDetectionSeconds += std::chrono::duration<double>(tEnd - tOptimized).count();
        ++m_uFrameCount;
        m_matTransformationLEFTLASTtoLEFTNOW = matTransformationWORLDtoLEFT * inverseIsometry(m_matTransformationWORLDtoLEFTLAST);   // :547
        m_matTransformationWORLDtoLEFTLAST = matTransformationWORLDtoLEFT;                                                     // :548
    }

    // wall time: the pose stage (getPoseStereoPosit incl. its fallback: stages 1-2 tracking and the solves), the solves alone
    // (CSolverStereoPosit, failed ones included), trackEpipolar, landmark optimisation, re-detection
    double getDurationPoseSeconds() const { return m_dDurationPoseSeconds; }
    double getDurationPoseSolverSeconds() const { return m_cMatcher.getSolverStereoPosit().getDurationSeconds(); }
    double getDurationTrackEpipolarSeconds() const { return m_dDurationTrackEpipolarSeconds; }
    double getDurationOptimizationSeconds() const { return m_dDurationOptimizationSeconds; }
    double getDurationDetectionSeconds() const { return m_dDurationDetectionSeconds; }

    CFundamentalMatcher& getMatcher() { return m_cMatcher; }
    UIDFrame getFrameCount() const { return m_uFrameCount; }
    uint64_t getNumberOfVisibleLandmarksLAST() const { return m_uNumberofVisibleLandmarksLAST; }
    uint64_t getNumberOfDetections() const { return m_uNumberOfDetections; }
    uint8_t getCountInstability() const { return m_uCountInstability; }
    const std::string& getPoseSource() const { return m_strPoseSource; }
    const Isometry3d& getTransformationWORLDtoLEFT() const { return m_matTransformationWORLDtoLEFTLAST; }

private:
    CFundamentalMatcher m_cMatcher;
    Isometry3d m_matTransformationWORLDtoLEFTLAST, m_matTransformationLEFTLASTtoLEFTNOW;
    UIDFrame m_uFrameCount = 0;
    uint64_t m_uNumberofVisibleLandmarksLAST = 0, m_uNumberOfDetections = 0;
    uint8_t m_uCountInstability = 0;
    std::string m_strPoseSource;
    const uint64_t m_uVisibleLandmarksMinimum = 100;                 // CTrackerSV.cpp:33
    const UIDFrame m_uMaximumNumberOfFramesWithoutDetection = 2;     // CTrackerSV.h:62
    const uint8_t m_uLandmarkOptimizationEveryNFrames = 10;          // CTrackerSV.h:79
    UIDFrame m_uNumberOfFramesWithoutDetection = 0;
    double m_dDurationPoseSeconds = 0.0, m_dDurationTrackEpipolarSeconds = 0.0, m_dDurationOptimizationSeconds = 0.0, m_dDurationDetectionSeconds = 0.0;
};

#if defined(__GNUC__) && !defined(__clang__)
#pragma GCC pop_options
#endif
#endif
