// CFundamentalMatcher -- image-space half of the reference's src/core/CFundamentalMatcher.{h,cpp}
// (addNewLandmarks :83-193, trackManual :1334-2027 (all stages), getMaskActiveLandmarks :2043-2073,
// visibility bookkeeping :244-263, :2005-2009) with the per-key-point / per-landmark image work done by
// ONE batched GPU call per frame instead of one OpenCV call per item.  CLandmark keeps the fields the
// optimisation side reads (src/types/CLandmark.h:35-59) and the per-landmark position refinement
// CLandmark::optimize (src/types/CLandmark.cpp:281-296, :447-581; CPU, a 3-unknown robust Gauss-Newton); g2o
// stays with the caller.
#ifndef SVI_HOST_CFUNDAMENTALMATCHER_H
#define SVI_HOST_CFUNDAMENTALMATCHER_H

#include <cmath>
#include <cstdlib>
#include <string>

#include "CSolverStereoPosit.h"
#include "CTriangulator.h"

// Pinned arithmetic: every product and sum below rounds on its own, in the written order (the GPU kernels and the CPU
// oracle do the same), whatever flags the including project uses -- the reference builds with -O3 -march=native
// (CMakeLists.txt:51), where GCC's default -ffp-contract=fast would fuse a*b + c into an FMA.
#if defined(__clang__)
#pragma clang fp contract(off)
#elif defined(__GNUC__)
#pragma GCC push_options
#pragma GCC optimize("fp-contract=off")
#endif

class CLandmark {
public:
    CLandmark(const UIDLandmark& p_uID, const CDescriptor& p_matDescriptorLEFT, const CDescriptor& p_matDescriptorRIGHT, const double& p_dKeyPointSize,
              const Point2f& p_ptUVLEFT, const Point2f& p_ptUVRIGHT, const CPoint3DCAMERA& p_vecPointXYZLEFT,
              const Isometry3d& p_matTransformationLEFTtoWORLD, const Isometry3d& p_matTransformationWORLDtoLEFT,
              const MatrixProjection& p_matProjectionWORLDtoLEFT, const MatrixProjection& p_matProjectionWORLDtoRIGHT, const UIDFrame& p_uIDFrame)
        : uID(p_uID), matDescriptorReferenceLEFT(p_matDescriptorLEFT), matDescriptorReferenceRIGHT(p_matDescriptorRIGHT), dKeyPointSize(p_dKeyPointSize),
          uIDFrameAtCreation(p_uIDFrame), vecPointXYZInitial(p_matTransformationLEFTtoWORLD * p_vecPointXYZLEFT), vecPointXYZOptimized(vecPointXYZInitial),
          vecUVReferenceLEFT{(double)p_ptUVLEFT.x, (double)p_ptUVLEFT.y, 1.0}, vecPointXYZMean(vecPointXYZInitial) {
        addMeasurement(p_uIDFrame, p_ptUVLEFT, p_ptUVRIGHT, p_matDescriptorLEFT, p_matDescriptorRIGHT, p_vecPointXYZLEFT, p_matTransformationLEFTtoWORLD,
                       p_matTransformationWORLDtoLEFT, p_matProjectionWORLDtoLEFT, p_matProjectionWORLDtoRIGHT);
    }
    ~CLandmark() { for (const CMeasurementLandmark* p : m_vecMeasurements) delete p; }
    CLandmark(const CLandmark&) = delete;

    const UIDLandmark uID;
    const CDescriptor matDescriptorReferenceLEFT, matDescriptorReferenceRIGHT;
    const double dKeyPointSize;
    const UIDFrame uIDFrameAtCreation;
    const CPoint3DWORLD vecPointXYZInitial;
    CPoint3DWORLD vecPointXYZOptimized;
    const double vecUVReferenceLEFT[3];   // CPoint2DHomogenized (CLandmark.h:43)
    uint8_t uFailedSubsequentTrackings = 0;
    uint32_t uOptimizationsSuccessful = 0, uOptimizationsFailed = 0;
    bool bIsOptimal = false, bIsCurrentlyVisible = false;
    uint32_t uNumberOfKeyFramePresences = 0;
    std::vector<CDescriptor> vecDescriptorsLEFT, vecDescriptorsRIGHT;
    CPoint3DWORLD vecPointXYZMean;
    double dCurrentAverageSquaredError = 0.0;
    // CLandmark.h:90-98
    static constexpr uint32_t uCapIterations = 1000;
    static constexpr double dConvergenceDelta = 1e-5;
    static constexpr double dMinimumRatioInliersToOutliers = 0.5;
    static constexpr double dKernelMaximumErrorSquaredPixels = 10.0;
    static constexpr double dMaximumErrorSquaredAveragePixels = 9.0;
    static constexpr size_t uMinimumMeasurementsForOptimization = 5;

    // src/types/CLandmark.cpp:80-279 without the per-bit statistics (loop-closure data, out of scope)
    void addMeasurement(const UIDFrame& p_uFrame, const Point2f& p_ptUVLEFT, const Point2f& p_ptUVRIGHT, const CDescriptor& p_matDescriptorLEFT,
                        const CDescriptor& p_matDescriptorRIGHT, const CPoint3DCAMERA& p_vecXYZLEFT, const Isometry3d& p_matTransformationLEFTtoWORLD,
                        const Isometry3d& p_matTransformationWORLDtoLEFT, const MatrixProjection& p_matProjectionWORLDtoLEFT,
                        const MatrixProjection& p_matProjectionWORLDtoRIGHT) {
        vecDescriptorsLEFT.push_back(p_matDescriptorLEFT);
        vecDescriptorsRIGHT.push_back(p_matDescriptorRIGHT);
        const CPoint3DWORLD vecXYZWORLD(p_matTransformationLEFTtoWORLD * p_vecXYZLEFT);
        for (int k = 0; k < 3; ++k) vecPointXYZMean.v[k] = (vecPointXYZMean.v[k] + vecXYZWORLD.v[k]) / 2.0;   // :126
        m_vecMeasurements.push_back(new CMeasurementLandmark(uID, p_ptUVLEFT, p_ptUVRIGHT, p_vecXYZLEFT, vecXYZWORLD,
                                                             vecPointXYZOptimized, p_matTransformationWORLDtoLEFT, p_matProjectionWORLDtoLEFT,
                                                             p_matProjectionWORLDtoRIGHT, uOptimizationsSuccessful));
        m_vecMeasurementFrames.push_back(p_uFrame);   // every measurement of a frame carries the same projection pair
    }
    const Point2f getLastDetectionLEFT() const { return m_vecMeasurements.back()->ptUVLEFT; }
    const Point2f getLastDetectionRIGHT() const { return m_vecMeasurements.back()->ptUVRIGHT; }
    const CDescriptor getLastDescriptorLEFT() const { return vecDescriptorsLEFT.back(); }
    const CDescriptor getLastDescriptorRIGHT() const { return vecDescriptorsRIGHT.back(); }
    float getLastDisparity() const { return m_vecMeasurements.back()->fDisparity; }
    const CMeasurementLandmark* getLastMeasurement() const { return m_vecMeasurements.back(); }
    std::vector<CMeasurementLandmark*>::size_type getNumberOfMeasurements() const { return m_vecMeasurements.size(); }

    // optimize :281-296: refine the world position once more than uMinimumMeasurementsForOptimization measurements exist
    void optimize(const UIDFrame& p_uFrame) {
        bIsOptimal = false;
        if (uMinimumMeasurementsForOptimization < m_vecMeasurements.size()) vecPointXYZOptimized = _getOptimizedLandmarkSTEREOUV(p_uFrame, vecPointXYZOptimized);
        else bIsOptimal = true;
    }

    // ---- the batched form of optimize (svi_optimize_landmarks: one GPU thread per landmark, same arithmetic).
    // Table of the projection pairs of the frames the packed measurements were taken in: one row per frame id.
    struct CPoseTable {
        std::vector<double> vecProjectionsLEFT, vecProjectionsRIGHT;   // rows of 12
        std::vector<int32_t> vecRowOfFrame;                            // frame id -> row, -1 = not seen yet
        void clear() { vecProjectionsLEFT.clear(); vecProjectionsRIGHT.clear(); vecRowOfFrame.clear(); }
        int32_t getRow(const UIDFrame p_uFrame, const CMeasurementLandmark* p_pMeasurement) {
            if (vecRowOfFrame.size() <= p_uFrame) vecRowOfFrame.resize(p_uFrame + 1, -1);
            int32_t& iRow = vecRowOfFrame[p_uFrame];
            if (0 > iRow) {
                iRow = (int32_t)(vecProjectionsLEFT.size() / 12);
                vecProjectionsLEFT.insert(vecProjectionsLEFT.end(), p_pMeasurement->matProjectionWORLDtoLEFT.m, p_pMeasurement->matProjectionWORLDtoLEFT.m + 12);
                vecProjectionsRIGHT.insert(vecProjectionsRIGHT.end(), p_pMeasurement->matProjectionWORLDtoRIGHT.m, p_pMeasurement->matProjectionWORLDtoRIGHT.m + 12);
            }
            return iRow;
        }
    };
    // appends this landmark's measurements (pose row, uv LEFT, uv RIGHT) to the packed arrays of a batch
    void packMeasurements(CPoseTable& p_cPoses, std::vector<int32_t>& p_vecPoseIndex, std::vector<float>& p_vecUVLEFT, std::vector<float>& p_vecUVRIGHT) const {
        for (size_t u = 0; u < m_vecMeasurements.size(); ++u) {
            const CMeasurementLandmark* pMeasurement = m_vecMeasurements[u];
            p_vecPoseIndex.push_back(p_cPoses.getRow(m_vecMeasurementFrames[u], pMeasurement));
            p_vecUVLEFT.push_back(pMeasurement->ptUVLEFT.x); p_vecUVLEFT.push_back(pMeasurement->ptUVLEFT.y);
            p_vecUVRIGHT.push_back(pMeasurement->ptUVRIGHT.x); p_vecUVRIGHT.push_back(pMeasurement->ptUVRIGHT.y);
        }
    }
    // the state changes of optimize / _getOptimizedLandmarkSTEREOUV for an outcome computed by the library
    void applyOptimization(const uint8_t p_uOutcome, const double* p_pXYZ, const double p_dAverageSquaredError) {
        bIsOptimal = false;
        m_bLastOptimizationFailed = false;
        switch (p_uOutcome) {
            case SVI_OPT_SKIPPED: bIsOptimal = true; break;
            case SVI_OPT_OPTIMAL: bIsOptimal = true;   // fall through
            case SVI_OPT_CONVERGED:
                ++uOptimizationsSuccessful;
                dCurrentAverageSquaredError = p_dAverageSquaredError;
                vecPointXYZOptimized = CPoint3DWORLD(p_pXYZ[0], p_pXYZ[1], p_pXYZ[2]);
                break;
            default:   // SVI_OPT_REJECTED, SVI_OPT_NOT_CONVERGED: position kept
                ++uOptimizationsFailed;
                m_bLastOptimizationFailed = true;
                m_uMeasurementsAtFailedOptimization = m_vecMeasurements.size();
                m_vecGuessAtFailedOptimization = vecPointXYZOptimized;
                break;
        }
    }
    // A failed optimisation leaves the landmark as it was, and trackManual never tracks it again (:1375-1384: no new
    // measurements), yet optimizeActiveLandmarks visits it in every later frame: the same measurements from the same guess
    // through a deterministic iteration -- the same failure, typically after all 1000 iterations.  When nothing the
    // optimisation reads has changed since it last failed, its outcome is repeated instead of recomputed.
    bool isRepeatOfFailedOptimization() const {
        return m_bLastOptimizationFailed && m_uMeasurementsAtFailedOptimization == m_vecMeasurements.size() &&
               m_vecGuessAtFailedOptimization.v[0] == vecPointXYZOptimized.v[0] && m_vecGuessAtFailedOptimization.v[1] == vecPointXYZOptimized.v[1] &&
               m_vecGuessAtFailedOptimization.v[2] == vecPointXYZOptimized.v[2];
    }
    void repeatFailedOptimization() { bIsOptimal = false; ++uOptimizationsFailed; }

private:
    // _getOptimizedLandmarkSTEREOUV :447-581: Gauss-Newton on the stereo reprojection error over all measurements, robust
    // weights above dKernelMaximumErrorSquaredPixels, the homogeneous coordinate held fixed (4x3 least-squares step)
    const CPoint3DWORLD _getOptimizedLandmarkSTEREOUV(const UIDFrame&, const CPoint3DWORLD& p_vecInitialGuess) {
        double X[4] = {p_vecInitialGuess.v[0], p_vecInitialGuess.v[1], p_vecInitialGuess.v[2], 1.0};
        double dErrorPrevious = 0.0;
        for (uint32_t uIteration = 0; uIteration < uCapIterations; ++uIteration) {
            double H[4][4] = {{0}}, b[4] = {0}, dErrorTotal = 0.0;
            uint32_t uInliers = 0;
            for (const CMeasurementLandmark* pMeasurement : m_vecMeasurements) {
                double J[4][4], e[4];
                const MatrixProjection* P[2] = {&pMeasurement->matProjectionWORLDtoLEFT, &pMeasurement->matProjectionWORLDtoRIGHT};
                const Point2f uv[2] = {pMeasurement->ptUVLEFT, pMeasurement->ptUVRIGHT};
                for (int s = 0; s < 2; ++s) {
                    double a[3];
                    for (int r = 0; r < 3; ++r) a[r] = (*P[s])(r, 0) * X[0] + (*P[s])(r, 1) * X[1] + (*P[s])(r, 2) * X[2] + (*P[s])(r, 3) * X[3];
                    const double c = a[2];
                    e[2 * s] = a[0] / c - uv[s].x;
                    e[2 * s + 1] = a[1] / c - uv[s].y;
                    for (int k = 0; k < 4; ++k) {
                        J[2 * s][k] = (*P[s])(0, k) / c - a[0] / (c * c) * (*P[s])(2, k);
                        J[2 * s + 1][k] = (*P[s])(1, k) / c - a[1] / (c * c) * (*P[s])(2, k);
                    }
                }
                const double e2 = e[0] * e[0] + e[1] * e[1] + e[2] * e[2] + e[3] * e[3];
                double w = 1.0;
                if (dKernelMaximumErrorSquaredPixels < e2) w = dKernelMaximumErrorSquaredPixels / e2;
                else ++uInliers;
                dErrorTotal += w * e2;
                for (int i = 0; i < 4; ++i) {
                    for (int j = 0; j < 4; ++j) H[i][j] += w * (J[0][i] * J[0][j] + J[1][i] * J[1][j] + J[2][i] * J[2][j] + J[3][i] * J[3][j]);
                    b[i] += w * (J[0][i] * e[0] + J[1][i] * e[1] + J[2][i] * e[2] + J[3][i] * e[3]);
                }
            }
            double dx[3];
            solveLeastSquares4x3(H, b, dx);   // H.block<4,3>(0,0).householderQr().solve(-b)
            for (int k = 0; k < 3; ++k) X[k] += dx[k];
            if (dConvergenceDelta > std::fabs(dErrorPrevious - dErrorTotal)) {
                const double dErrorAverage = dErrorTotal / m_vecMeasurements.size();
                if (dMinimumRatioInliersToOutliers < static_cast<double>(uInliers) / m_vecMeasurements.size()) {
                    ++uOptimizationsSuccessful;
                    dCurrentAverageSquaredError = dErrorAverage;
                    if (dMaximumErrorSquaredAveragePixels > dErrorAverage) bIsOptimal = true;
                    return CPoint3DWORLD(X[0], X[1], X[2]);
                }
                ++uOptimizationsFailed;
                return p_vecInitialGuess;
            }
            dErrorPrevious = dErrorTotal;
        }
        ++uOptimizationsFailed;
        return p_vecInitialGuess;
    }
    // min || A x + b || for the 4x3 matrix A = first three columns of H, by Householder reflections
    static void solveLeastSquares4x3(const double (&H)[4][4], const double (&b)[4], double (&x)[3]) {
        double A[4][3], y[4];
        for (int i = 0; i < 4; ++i) { for (int j = 0; j < 3; ++j) A[i][j] = H[i][j]; y[i] = -b[i]; }
        for (int c = 0; c < 3; ++c) {
            double norm = 0.0;
            for (int r = c; r < 4; ++r) norm += A[r][c] * A[r][c];
            norm = std::sqrt(norm);
            if (0.0 == norm) continue;
            const double alpha = A[c][c] > 0.0 ? -norm : norm;
            double v[4] = {0, 0, 0, 0};
            v[c] = A[c][c] - alpha;
            for (int r = c + 1; r < 4; ++r) v[r] = A[r][c];
            double vv = 0.0;
            for (int r = c; r < 4; ++r) vv += v[r] * v[r];
            if (0.0 == vv) continue;
            for (int j = c; j < 3; ++j) {
                double d = 0.0;
                for (int r = c; r < 4; ++r) d += v[r] * A[r][j];
                for (int r = c; r < 4; ++r) A[r][j] -= 2.0 * d / vv * v[r];
            }
            double d = 0.0;
            for (int r = c; r < 4; ++r) d += v[r] * y[r];
            for (int r = c; r < 4; ++r) y[r] -= 2.0 * d / vv * v[r];
        }
        for (int r = 2; r >= 0; --r) {
            double s2 = y[r];
            for (int j = r + 1; j < 3; ++j) s2 -= A[r][j] * x[j];
            x[r] = (0.0 != A[r][r]) ? s2 / A[r][r] : 0.0;
        }
    }

    std::vector<CMeasurementLandmark*> m_vecMeasurements;
    std::vector<UIDFrame> m_vecMeasurementFrames;
    bool m_bLastOptimizationFailed = false;
    size_t m_uMeasurementsAtFailedOptimization = 0;
    CPoint3DWORLD m_vecGuessAtFailedOptimization;
};

class CFundamentalMatcher {
    struct CDetectionPoint {
        UIDDetectionPoint uID;
        Isometry3d matTransformationLEFTtoWORLD;
        std::shared_ptr<std::vector<CLandmark*>> vecLandmarks;
    };

public:
    CFundamentalMatcher(const std::shared_ptr<CStereoCamera> p_pCameraSTEREO, const std::shared_ptr<CGpuContext> p_pGpu)
        : m_pGpu(p_pGpu), m_pTriangulator(std::make_shared<CTriangulator>(p_pCameraSTEREO, p_pGpu)), m_pCameraLEFT(p_pCameraSTEREO->m_pCameraLEFT),
          m_pCameraRIGHT(p_pCameraSTEREO->m_pCameraRIGHT), m_pCameraSTEREO(p_pCameraSTEREO), m_dMinimumDepthMeters(m_pTriangulator->dDepthMinimumMeters),
          m_dMaximumDepthMeters(m_pTriangulator->dDepthMaximumMeters),
          m_cSolverSterePosit(p_pCameraSTEREO->m_pCameraLEFT->m_matProjection, p_pCameraSTEREO->m_pCameraRIGHT->m_matProjection, p_pGpu) {}
    ~CFundamentalMatcher() { for (CLandmark* p : m_vecLandmarksWINDOW) delete p; }

    const std::shared_ptr<CTriangulator> getTriangulator() const { return m_pTriangulator; }
    std::vector<CLandmark*>::size_type getNumberOfVisibleLandmarks() const { return m_vecVisibleLandmarks.size(); }
    UIDLandmark getNumberOfLandmarksTotal() const { return m_uAvailableLandmarkID; }
    UIDLandmark getNumberOfTracksStage1() const { return m_uNumberOfTracksStage1; }
    UIDLandmark getNumberOfTracksStage2_1() const { return m_uNumberOfTracksStage2_1; }
    UIDLandmark getNumberOfTracksStage3() const { return m_uNumberOfTracksStage3; }
    const std::vector<CLandmark*>& getLandmarksWINDOW() const { return m_vecLandmarksWINDOW; }
    // the landmarks of the active detection points, in the order trackManual walks them
    std::vector<const CLandmark*> getActiveLandmarks() const {
        std::vector<const CLandmark*> v;
        for (const CDetectionPoint& d : m_vecDetectionPointsActive) v.insert(v.end(), d.vecLandmarks->begin(), d.vecLandmarks->end());
        return v;
    }
    size_t getNumberOfActiveLandmarks() const {
        size_t n = 0;
        for (const CDetectionPoint& d : m_vecDetectionPointsActive) n += d.vecLandmarks->size();
        return n;
    }

    // optimizeActiveLandmarks :265-277: CLandmark::optimize for every active landmark -- ONE library call (one GPU thread per
    // landmark, the arithmetic of CLandmark::_getOptimizedLandmarkSTEREOUV in the same order) instead of the per-landmark
    // CPU loop, which is the largest item of the host's frame time (SVI_HOST_OPTIMIZE=cpu keeps that loop: the checker of
    // the parity test)
    void optimizeActiveLandmarks(const UIDFrame& p_uFrame) {
        static const bool bCPU = [] { const char* e = std::getenv("SVI_HOST_OPTIMIZE"); return e && std::string(e) == "cpu"; }();
        if (bCPU) {
            for (const CDetectionPoint& cDetectionPoint : m_vecDetectionPointsActive)
                for (CLandmark* pLandmark : *cDetectionPoint.vecLandmarks) pLandmark->optimize(p_uFrame);
            return;
        }
        m_vecOptLandmarks.clear(); m_vecOptGuess.clear(); m_vecOptFirst.clear(); m_vecOptPoseIndex.clear(); m_vecOptUVLEFT.clear(); m_vecOptUVRIGHT.clear();
        m_cOptPoses.clear();
        m_vecOptFirst.push_back(0);
        for (const CDetectionPoint& cDetectionPoint : m_vecDetectionPointsActive)
            for (CLandmark* pLandmark : *cDetectionPoint.vecLandmarks) {
                if (pLandmark->isRepeatOfFailedOptimization()) { pLandmark->repeatFailedOptimization(); continue; }
                m_vecOptLandmarks.push_back(pLandmark);
                for (int k = 0; k < 3; ++k) m_vecOptGuess.push_back(pLandmark->vecPointXYZOptimized.v[k]);
                pLandmark->packMeasurements(m_cOptPoses, m_vecOptPoseIndex, m_vecOptUVLEFT, m_vecOptUVRIGHT);
                m_vecOptFirst.push_back((int32_t)m_vecOptPoseIndex.size());
            }
        const int n = (int)m_vecOptLandmarks.size();
        if (0 == n) return;
        m_vecOptXYZ.resize(3 * (size_t)n); m_vecOptOutcome.resize(n); m_vecOptError.resize(n);
        svi_landmark_measurements cIn{m_vecOptGuess.data(), m_vecOptFirst.data(), m_vecOptPoseIndex.data(), m_vecOptUVLEFT.data(), m_vecOptUVRIGHT.data(),
                                      m_cOptPoses.vecProjectionsLEFT.data(), m_cOptPoses.vecProjectionsRIGHT.data(),
                                      (int32_t)(m_cOptPoses.vecProjectionsLEFT.size() / 12)};
        svi_optimize_result cOut{m_vecOptXYZ.data(), m_vecOptOutcome.data(), m_vecOptError.data(), nullptr};
        m_pGpu->check(svi_optimize_landmarks(m_pGpu->ctx, &cIn, n, &cOut));
        for (int i = 0; i < n; ++i) m_vecOptLandmarks[i]->applyOptimization(m_vecOptOutcome[i], &m_vecOptXYZ[3 * (size_t)i], m_vecOptError[i]);
    }

    // :244-254
    void resetVisibilityActiveLandmarks() {
        for (CLandmark* pLandmark : m_vecVisibleLandmarks) pLandmark->bIsCurrentlyVisible = false;
        m_vecVisibleLandmarks.clear();
    }
    // :321-335
    const std::vector<const CMeasurementLandmark*> getMeasurementsForVisibleLandmarks() {
        m_vecMeasurementsVisible.clear();
        for (CLandmark* pLandmark : m_vecVisibleLandmarks) m_vecMeasurementsVisible.push_back(pLandmark->getLastMeasurement());
        return m_vecMeasurementsVisible;
    }

    // The centres getMaskActiveLandmarks :2043-2073 draws its discs at: the last LEFT detection of a visible landmark
    // (:2057), the projection of an invisible one (getUV, :2062-2065).
    std::vector<Point2f> getMaskCentres(const Isometry3d& p_matTransformationWORLDtoLEFT) const {
        std::vector<Point2f> vecCentres;
        for (const CDetectionPoint& cDetectionPoint : m_vecDetectionPointsActive)
            for (const CLandmark* pLandmark : *cDetectionPoint.vecLandmarks) {
                if (pLandmark->bIsCurrentlyVisible) vecCentres.push_back(pLandmark->getLastDetectionLEFT());
                else {
                    const CPoint3DCAMERA p(p_matTransformationWORLDtoLEFT * pLandmark->vecPointXYZOptimized);
                    const MatrixProjection& P = m_pCameraLEFT->m_matProjection;
                    const double w = P(2, 0) * p.x() + P(2, 1) * p.y() + P(2, 2) * p.z() + P(2, 3);
                    vecCentres.push_back(Point2f((float)((P(0, 0) * p.x() + P(0, 1) * p.y() + P(0, 2) * p.z() + P(0, 3)) / w),
                                                 (float)((P(1, 0) * p.x() + P(1, 1) * p.y() + P(1, 2) * p.z() + P(1, 3)) / w)));
                }
            }
        return vecCentres;
    }
    // 255 everywhere, filled radius-7 zero discs (cv::circle, m_uFeatureRadiusForMask): stamped on the GPU
    // (svi_mask_active_landmarks); the plane only comes back for callers that want to look at it
    std::vector<uint8_t> getMaskForCentres(const std::vector<Point2f>& p_vecCentres) const {
        const int W = m_pCameraSTEREO->m_uPixelWidth, H = m_pCameraSTEREO->m_uPixelHeight;
        std::vector<uint8_t> matMaskDetection((size_t)W * H, 255);
        static_assert(sizeof(Point2f) == 2 * sizeof(float), "Point2f is two packed floats");
        m_pGpu->check(svi_mask_active_landmarks(m_pGpu->ctx, p_vecCentres.empty() ? nullptr : &p_vecCentres[0].x, (int)p_vecCentres.size(),
                                                matMaskDetection.data(), (size_t)W));
        return matMaskDetection;
    }
    std::vector<uint8_t> getMaskActiveLandmarks(const Isometry3d& p_matTransformationWORLDtoLEFT) const {
        return getMaskForCentres(getMaskCentres(p_matTransformationWORLDtoLEFT));
    }

    // addNewLandmarks :83-193: mask -> detect -> describe -> per-key-point scan-line triangulation, one GPU call; the
    // mask is built on the device from the landmark centres (8 bytes per landmark instead of a W x H plane upload)
    std::vector<CLandmark*>::size_type addNewLandmarks(const ImageView& p_matImageLEFT, const ImageView& p_matImageRIGHT,
                                                       const Isometry3d& p_matTransformationWORLDtoLEFT,
                                                       const Isometry3d& p_matTransformationLEFTtoWORLD, const UIDFrame& p_uIDFrame) {
        const MatrixProjection matProjectionWORLDtoLEFT(m_pCameraLEFT->m_matProjection * p_matTransformationWORLDtoLEFT);
        const MatrixProjection matProjectionWORLDtoRIGHT(m_pCameraRIGHT->m_matProjection * p_matTransformationWORLDtoLEFT);
        const std::vector<Point2f> vecCentres(getMaskCentres(p_matTransformationWORLDtoLEFT));
        const int cap = m_pGpu->params.max_corners;
        int32_t nKeyPoints = 0, nDetected = 0;
        std::vector<float> uvL(2 * cap), uvR(2 * cap);
        std::vector<double> xyz(3 * cap);
        std::vector<uint8_t> dL(32 * cap), dR(32 * cap), st(cap);
        std::vector<int32_t> dist(cap), idx(cap);
        svi_stereo_result r{cap, &nKeyPoints, &nDetected, uvL.data(), uvR.data(), xyz.data(), dL.data(), dR.data(), dist.data(), idx.data(), st.data()};
        m_pGpu->check(svi_stereo_frame_masked(m_pGpu->ctx, p_matImageLEFT.data, p_matImageRIGHT.data, p_matImageLEFT.pitch,
                                              vecCentres.empty() ? nullptr : &vecCentres[0].x, (int)vecCentres.size(), &r));

        std::shared_ptr<std::vector<CLandmark*>> vecLandmarksNEW(std::make_shared<std::vector<CLandmark*>>());
        for (int32_t u = 0; u < nKeyPoints; ++u) {
            if (SVI_OK != st[u]) continue;   // catch( CExceptionNoMatchFound ) { continue; }  :170-174
            CDescriptor matDescriptorLEFT, matDescriptorRIGHT;
            std::memcpy(matDescriptorLEFT.data(), &dL[32 * u], 32);
            std::memcpy(matDescriptorRIGHT.data(), &dR[32 * u], 32);
            CLandmark* pLandmarkNEW = new CLandmark(m_uAvailableLandmarkID, matDescriptorLEFT, matDescriptorRIGHT, m_pGpu->params.keypoint_size,
                                                    Point2f(uvL[2 * u], uvL[2 * u + 1]), Point2f(uvR[2 * u], uvR[2 * u + 1]),
                                                    CPoint3DCAMERA(xyz[3 * u], xyz[3 * u + 1], xyz[3 * u + 2]), p_matTransformationLEFTtoWORLD,
                                                    p_matTransformationWORLDtoLEFT, matProjectionWORLDtoLEFT, matProjectionWORLDtoRIGHT, p_uIDFrame);
            pLandmarkNEW->bIsOptimal = true;   // :147
            vecLandmarksNEW->push_back(pLandmarkNEW);
            ++m_uAvailableLandmarkID;
        }
        if (vecLandmarksNEW->empty()) return 0;
        m_vecDetectionPointsActive.push_back(CDetectionPoint{m_uAvailableDetectionPointID++, p_matTransformationLEFTtoWORLD, vecLandmarksNEW});
        m_vecLandmarksWINDOW.insert(m_vecLandmarksWINDOW.end(), vecLandmarksNEW->begin(), vecLandmarksNEW->end());
        return vecLandmarksNEW->size();
    }

    // trackManual :1334-2027: the whole first-success cascade (stage 1 L/R, stage 2 L/R, stage 3) for ALL active
    // landmarks in ONE GPU call; the visibility / failed-tracking bookkeeping of :1980-2009 follows.
    void trackManual(const UIDFrame p_uFrame, const ImageView& p_matImageLEFT, const ImageView& p_matImageRIGHT,
                     const Isometry3d& p_matTransformationWORLDtoLEFT, const Isometry3d& p_matTransformationLEFTtoWORLD,
                     const double& p_dMotionScaling) {
        m_uNumberOfTracksStage1 = m_uNumberOfTracksStage2_1 = m_uNumberOfTracksStage3 = 0;
        const MatrixProjection matProjectionWORLDtoLEFT(m_pCameraLEFT->m_matProjection * p_matTransformationWORLDtoLEFT);
        const MatrixProjection matProjectionWORLDtoRIGHT(m_pCameraRIGHT->m_matProjection * p_matTransformationWORLDtoLEFT);
        std::vector<CLandmark*> vecCandidates;
        std::vector<const CDetectionPoint*> vecDetectionPointOf;
        for (const CDetectionPoint& cDetectionPoint : m_vecDetectionPointsActive)
            for (CLandmark* pLandmark : *cDetectionPoint.vecLandmarks) {
                if (0 < pLandmark->uOptimizationsFailed) { pLandmark->bIsCurrentlyVisible = false; pLandmark->bIsOptimal = false; }   // :1375-1384
                else if (0 < pLandmark->uOptimizationsSuccessful && !pLandmark->bIsOptimal) pLandmark->bIsCurrentlyVisible = false;      // :1387-1395
                else { vecCandidates.push_back(pLandmark); vecDetectionPointOf.push_back(&cDetectionPoint); }
            }
        const int n = (int)vecCandidates.size();
        if (0 < n) {
            std::vector<double> xyzW(3 * n), xyz(3 * n), uvRef(2 * n), Tdet(16 * n);
            std::vector<uint8_t> dL(32 * n), dR(32 * n), dRef(32 * n), oL(32 * n), oR(32 * n), st(n), stage(n);
            std::vector<float> disp(n), size(n), uvL(2 * n), uvR(2 * n);
            for (int i = 0; i < n; ++i) {
                const CLandmark* p = vecCandidates[i];
                for (int k = 0; k < 3; ++k) xyzW[3 * i + k] = p->vecPointXYZOptimized.v[k];
                std::memcpy(&dL[32 * i], p->getLastDescriptorLEFT().data(), 32);
                std::memcpy(&dR[32 * i], p->getLastDescriptorRIGHT().data(), 32);
                std::memcpy(&dRef[32 * i], p->matDescriptorReferenceLEFT.data(), 32);
                disp[i] = p->getLastDisparity();
                size[i] = (float)p->dKeyPointSize;
                uvRef[2 * i] = p->vecUVReferenceLEFT[0];
                uvRef[2 * i + 1] = p->vecUVReferenceLEFT[1];
                std::memcpy(&Tdet[16 * i], vecDetectionPointOf[i]->matTransformationLEFTtoWORLD.m, sizeof(double) * 16);
            }
            svi_landmarks lm{xyzW.data(), dL.data(), dR.data(), disp.data(), size.data(), uvRef.data(), dRef.data(), Tdet.data()};
            svi_track_result r{st.data(), stage.data(), uvL.data(), uvR.data(), xyz.data(), oL.data(), oR.data()};
            m_pGpu->check(svi_track_landmarks(m_pGpu->ctx, p_matImageLEFT.data, p_matImageRIGHT.data, p_matImageLEFT.pitch,
                                              p_matTransformationWORLDtoLEFT.m, &lm, n, p_dMotionScaling, &r));
            for (int i = 0; i < n; ++i) {
                CLandmark* pLandmark = vecCandidates[i];
                if (0 < stage[i]) {   // _addMeasurementToLandmarkSTEREO :2487-2524
                    CDescriptor a, b;
                    std::memcpy(a.data(), &oL[32 * i], 32);
                    std::memcpy(b.data(), &oR[32 * i], 32);
                    pLandmark->bIsCurrentlyVisible = true;
                    pLandmark->uFailedSubsequentTrackings = 0;
                    pLandmark->addMeasurement(p_uFrame, Point2f(uvL[2 * i], uvL[2 * i + 1]), Point2f(uvR[2 * i], uvR[2 * i + 1]), a, b,
                                              CPoint3DCAMERA(xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]), p_matTransformationLEFTtoWORLD,
                                              p_matTransformationWORLDtoLEFT, matProjectionWORLDtoLEFT, matProjectionWORLDtoRIGHT);
                    m_vecVisibleLandmarks.push_back(pLandmark);
                    if (stage[i] <= 2) ++m_uNumberOfTracksStage1;
                    else if (stage[i] <= 4) ++m_uNumberOfTracksStage2_1;
                    else ++m_uNumberOfTracksStage3;
                } else if (SVI_EPI_NO_TRANSLATION != st[i]) {
                    ++pLandmark->uFailedSubsequentTrackings;   // :1980-1987, :1996-2001
                    pLandmark->bIsCurrentlyVisible = false;
                }   // no translation since detection: the reference neither tracks nor penalises the landmark (:1804)
            }
        }
        // keep landmarks while failed trackings stay below the limit :2005-2009
        for (CDetectionPoint& cDetectionPoint : m_vecDetectionPointsActive) {
            std::vector<CLandmark*>& v = *cDetectionPoint.vecLandmarks;
            v.erase(std::remove_if(v.begin(), v.end(), [this](CLandmark* p) { return p->uFailedSubsequentTrackings >= m_uMaximumFailedSubsequentTrackingsPerLandmark; }), v.end());
        }
        m_vecDetectionPointsActive.erase(std::remove_if(m_vecDetectionPointsActive.begin(), m_vecDetectionPointsActive.end(),
                                                        [](const CDetectionPoint& d) { return d.vecLandmarks->empty(); }),
                                         m_vecDetectionPointsActive.end());
    }

    // Gathers what svi_track_landmarks[_stages] reads of a set of landmarks, runs the requested stages in ONE GPU call
    // and returns the per-landmark verdicts.
    struct CTrackBatch {
        std::vector<double> xyz;
        std::vector<uint8_t> oL, oR, st, stage;
        std::vector<float> uvL, uvR;
    };
    CTrackBatch trackStages(const std::vector<CLandmark*>& p_vecLandmarks, const std::vector<const CDetectionPoint*>& p_vecDetectionPointOf,
                            const ImageView& p_matImageLEFT, const ImageView& p_matImageRIGHT, const Isometry3d& p_matTransformationWORLDtoLEFT,
                            const double& p_dMotionScaling, const uint32_t p_uStageMask) const {
        const int n = (int)p_vecLandmarks.size();
        CTrackBatch c;
        c.xyz.resize(3 * n); c.oL.resize(32 * n); c.oR.resize(32 * n); c.st.resize(n); c.stage.resize(n); c.uvL.resize(2 * n); c.uvR.resize(2 * n);
        if (0 == n) return c;
        std::vector<double> xyzW(3 * n), uvRef(2 * n), Tdet(16 * n);
        std::vector<uint8_t> dL(32 * n), dR(32 * n), dRef(32 * n);
        std::vector<float> disp(n), size(n);
        for (int i = 0; i < n; ++i) {
            const CLandmark* p = p_vecLandmarks[i];
            for (int k = 0; k < 3; ++k) xyzW[3 * i + k] = p->vecPointXYZOptimized.v[k];
            std::memcpy(&dL[32 * i], p->getLastDescriptorLEFT().data(), 32);
            std::memcpy(&dR[32 * i], p->getLastDescriptorRIGHT().data(), 32);
            std::memcpy(&dRef[32 * i], p->matDescriptorReferenceLEFT.data(), 32);
            disp[i] = p->getLastDisparity();
            size[i] = (float)p->dKeyPointSize;
            uvRef[2 * i] = p->vecUVReferenceLEFT[0];
            uvRef[2 * i + 1] = p->vecUVReferenceLEFT[1];
            std::memcpy(&Tdet[16 * i], p_vecDetectionPointOf[i]->matTransformationLEFTtoWORLD.m, sizeof(double) * 16);
        }
        const bool bStage3 = 0 != (p_uStageMask & SVI_STAGE_3);
        svi_landmarks lm{xyzW.data(), dL.data(), dR.data(), disp.data(), size.data(), bStage3 ? uvRef.data() : nullptr,
                         bStage3 ? dRef.data() : nullptr, bStage3 ? Tdet.data() : nullptr};
        svi_track_result r{c.st.data(), c.stage.data(), c.uvL.data(), c.uvR.data(), c.xyz.data(), c.oL.data(), c.oR.data()};
        m_pGpu->check(svi_track_landmarks_stages(m_pGpu->ctx, p_matImageLEFT.data, p_matImageRIGHT.data, p_matImageLEFT.pitch,
                                                 p_matTransformationWORLDtoLEFT.m, &lm, n, p_dMotionScaling, p_uStageMask, &r));
        return c;
    }

    // _addMeasurementToLandmarkSTEREO :2487-2524
    void _addMeasurementToLandmarkSTEREO(const UIDFrame p_uFrame, CLandmark* p_pLandmark, const Point2f& p_ptUVLEFT, const Point2f& p_ptUVRIGHT,
                                         const CPoint3DCAMERA& p_vecPointXYZLEFT, const CDescriptor& p_matDescriptorLEFT,
                                         const CDescriptor& p_matDescriptorRIGHT, const Isometry3d& p_matTransformationLEFTtoWORLD,
                                         const Isometry3d& p_matTransformationWORLDtoLEFT, const MatrixProjection& p_matProjectionWORLDtoLEFT,
                                         const MatrixProjection& p_matProjectionWORLDtoRIGHT) {
        p_pLandmark->bIsCurrentlyVisible = true;
        p_pLandmark->uFailedSubsequentTrackings = 0;
        p_pLandmark->addMeasurement(p_uFrame, p_ptUVLEFT, p_ptUVRIGHT, p_matDescriptorLEFT, p_matDescriptorRIGHT, p_vecPointXYZLEFT,
                                    p_matTransformationLEFTtoWORLD, p_matTransformationWORLDtoLEFT, p_matProjectionWORLDtoLEFT, p_matProjectionWORLDtoRIGHT);
        m_vecVisibleLandmarks.push_back(p_pLandmark);
    }

    // getPoseStereoPosit :338-757: stages 1 and 2 on every OPTIMAL landmark around the pose estimate (one GPU call), the
    // measurements go to CSolverStereoPosit (one more GPU call; CExceptionPoseOptimization on failure, as in the reference), then the
    // landmarks receive their measurement under the optimised pose.
    const Isometry3d getPoseStereoPosit(const UIDFrame p_uFrame, const ImageView& p_matImageLEFT, const ImageView& p_matImageRIGHT,
                                        const Isometry3d& p_matTransformationEstimateWORLDtoLEFT, const Isometry3d& p_matTransformationWORLDtoLEFTLAST,
                                        const CPoint3D& /*p_vecRotationIMU*/, const CPoint3D& p_vecTranslationIMU, const double& p_dMotionScaling) {
        m_uNumberOfTracksStage1 = m_uNumberOfTracksStage2_1 = 0;
        std::vector<CLandmark*> vecCandidates;
        std::vector<const CDetectionPoint*> vecDetectionPointOf;
        for (const CDetectionPoint& cDetectionPoint : m_vecDetectionPointsActive)
            for (CLandmark* pLandmark : *cDetectionPoint.vecLandmarks)
                if (pLandmark->bIsOptimal) { vecCandidates.push_back(pLandmark); vecDetectionPointOf.push_back(&cDetectionPoint); }
        const CTrackBatch c(trackStages(vecCandidates, vecDetectionPointOf, p_matImageLEFT, p_matImageRIGHT, p_matTransformationEstimateWORLDtoLEFT,
                                        p_dMotionScaling, SVI_STAGE_1 | SVI_STAGE_2));
        std::vector<CSolverStereoPosit::CMatch> vecMeasurementsForStereoPosit;
        for (size_t i = 0; i < vecCandidates.size(); ++i) {
            if (0 == c.stage[i]) continue;
            CDescriptor a, b;
            std::memcpy(a.data(), &c.oL[32 * i], 32);
            std::memcpy(b.data(), &c.oR[32 * i], 32);
            vecMeasurementsForStereoPosit.push_back(CSolverStereoPosit::CMatch(vecCandidates[i], vecCandidates[i]->vecPointXYZOptimized,
                                                                               CPoint3DCAMERA(c.xyz[3 * i], c.xyz[3 * i + 1], c.xyz[3 * i + 2]),
                                                                               Point2f(c.uvL[2 * i], c.uvL[2 * i + 1]), Point2f(c.uvR[2 * i], c.uvR[2 * i + 1]), a, b));
            if (c.stage[i] <= 2) ++m_uNumberOfTracksStage1; else ++m_uNumberOfTracksStage2_1;
        }
        const Isometry3d matTransformationWORLDtoLEFT(m_cSolverSterePosit.getTransformationWORLDtoLEFT(
            p_matTransformationWORLDtoLEFTLAST, p_vecTranslationIMU, p_matTransformationEstimateWORLDtoLEFT, vecMeasurementsForStereoPosit));
        const MatrixProjection matProjectionWORLDtoLEFT(m_pCameraLEFT->m_matProjection * matTransformationWORLDtoLEFT);
        const MatrixProjection matProjectionWORLDtoRIGHT(m_pCameraRIGHT->m_matProjection * matTransformationWORLDtoLEFT);
        const Isometry3d matTransformationLEFTtoWORLD(inverseIsometry(matTransformationWORLDtoLEFT));
        for (const CSolverStereoPosit::CMatch& cMatchSTEREO : vecMeasurementsForStereoPosit)
            _addMeasurementToLandmarkSTEREO(p_uFrame, cMatchSTEREO.pLandmark, cMatchSTEREO.ptUVLEFT, cMatchSTEREO.ptUVRIGHT, cMatchSTEREO.vecPointXYZLEFT,
                                            cMatchSTEREO.matDescriptorLEFT, cMatchSTEREO.matDescriptorRIGHT, matTransformationLEFTtoWORLD,
                                            matTransformationWORLDtoLEFT, matProjectionWORLDtoLEFT, matProjectionWORLDtoRIGHT);
        m_vecMeasurementsStereoPositLAST.swap(vecMeasurementsForStereoPosit);
        return matTransformationWORLDtoLEFT;
    }
    const std::vector<CSolverStereoPosit::CMatch>& getMeasurementsStereoPositLAST() const { return m_vecMeasurementsStereoPositLAST; }
    const CSolverStereoPosit& getSolverStereoPosit() const { return m_cSolverSterePosit; }

    // trackEpipolar :760-1332: the landmarks getPoseStereoPosit did not see.  Where the camera has moved since the
    // landmark's detection: the epipolar search (stage 3) alone; otherwise: the regional search (stage 2) behind the
    // field-of-view gate.  Two GPU calls for the whole frame, then the reference's activity bookkeeping.
    void trackEpipolar(const UIDFrame p_uFrame, const ImageView& p_matImageLEFT, const ImageView& p_matImageRIGHT,
                       const Isometry3d& p_matTransformationWORLDtoLEFT, const Isometry3d& p_matTransformationLEFTtoWORLD, const double& p_dMotionScaling) {
        const MatrixProjection matProjectionWORLDtoLEFT(m_pCameraLEFT->m_matProjection * p_matTransformationWORLDtoLEFT);
        const MatrixProjection matProjectionWORLDtoRIGHT(m_pCameraRIGHT->m_matProjection * p_matTransformationWORLDtoLEFT);
        m_uNumberOfTracksStage3 = m_uNumberOfTracksStage2_2 = 0;
        std::vector<CLandmark*> vecEpipolar, vecRegional, vecDropped;
        std::vector<const CDetectionPoint*> vecDetectionPointOfEpipolar, vecDetectionPointOfRegional;
        for (const CDetectionPoint& cDetectionPoint : m_vecDetectionPointsActive) {
            const Isometry3d matTransformationToNow(p_matTransformationWORLDtoLEFT * cDetectionPoint.matTransformationLEFTtoWORLD);   // :800
            const double dTranslationSquaredNorm = matTransformationToNow(0, 3) * matTransformationToNow(0, 3) + matTransformationToNow(1, 3) * matTransformationToNow(1, 3) +
                                                   matTransformationToNow(2, 3) * matTransformationToNow(2, 3);
            for (CLandmark* pLandmark : *cDetectionPoint.vecLandmarks) {
                if (0 < pLandmark->uOptimizationsFailed) { pLandmark->bIsCurrentlyVisible = false; vecDropped.push_back(pLandmark); }                                   // :808-815
                else if (0 < pLandmark->uOptimizationsSuccessful && !pLandmark->bIsOptimal) { pLandmark->bIsCurrentlyVisible = false; vecDropped.push_back(pLandmark); } // :818-825
                else if (pLandmark->bIsCurrentlyVisible) continue;                                                                                                       // :830-833
                else if (0.0 < dTranslationSquaredNorm) { vecEpipolar.push_back(pLandmark); vecDetectionPointOfEpipolar.push_back(&cDetectionPoint); }
                else { vecRegional.push_back(pLandmark); vecDetectionPointOfRegional.push_back(&cDetectionPoint); }
            }
        }
        auto apply = [&](const std::vector<CLandmark*>& p_vecLandmarks, const CTrackBatch& c, UIDLandmark& p_uCounter) {
            for (size_t i = 0; i < p_vecLandmarks.size(); ++i) {
                CLandmark* pLandmark = p_vecLandmarks[i];
                if (0 < c.stage[i]) {
                    CDescriptor a, b;
                    std::memcpy(a.data(), &c.oL[32 * i], 32);
                    std::memcpy(b.data(), &c.oR[32 * i], 32);
                    _addMeasurementToLandmarkSTEREO(p_uFrame, pLandmark, Point2f(c.uvL[2 * i], c.uvL[2 * i + 1]), Point2f(c.uvR[2 * i], c.uvR[2 * i + 1]),
                                                    CPoint3DCAMERA(c.xyz[3 * i], c.xyz[3 * i + 1], c.xyz[3 * i + 2]), a, b, p_matTransformationLEFTtoWORLD,
                                                    p_matTransformationWORLDtoLEFT, matProjectionWORLDtoLEFT, matProjectionWORLDtoRIGHT);
                    ++p_uCounter;
                } else {
                    ++pLandmark->uFailedSubsequentTrackings;   // :1014-1023, :1281-1289
                    pLandmark->bIsCurrentlyVisible = false;
                }
            }
        };
        {
            const CTrackBatch c(trackStages(vecEpipolar, vecDetectionPointOfEpipolar, p_matImageLEFT, p_matImageRIGHT, p_matTransformationWORLDtoLEFT,
                                            p_dMotionScaling, SVI_STAGE_3));
            // the library decides "no translation" on its own product of the two transforms: follow its verdict
            std::vector<CLandmark*> vecMoved;
            CTrackBatch m;
            for (size_t i = 0; i < vecEpipolar.size(); ++i) {
                if (SVI_EPI_NO_TRANSLATION == c.st[i]) { vecRegional.push_back(vecEpipolar[i]); vecDetectionPointOfRegional.push_back(vecDetectionPointOfEpipolar[i]); continue; }
                vecMoved.push_back(vecEpipolar[i]);
                m.st.push_back(c.st[i]); m.stage.push_back(c.stage[i]);
                m.uvL.insert(m.uvL.end(), &c.uvL[2 * i], &c.uvL[2 * i] + 2); m.uvR.insert(m.uvR.end(), &c.uvR[2 * i], &c.uvR[2 * i] + 2);
                m.xyz.insert(m.xyz.end(), &c.xyz[3 * i], &c.xyz[3 * i] + 3);
                m.oL.insert(m.oL.end(), &c.oL[32 * i], &c.oL[32 * i] + 32); m.oR.insert(m.oR.end(), &c.oR[32 * i], &c.oR[32 * i] + 32);
            }
            apply(vecMoved, m, m_uNumberOfTracksStage3);
        }
        apply(vecRegional, trackStages(vecRegional, vecDetectionPointOfRegional, p_matImageLEFT, p_matImageRIGHT, p_matTransformationWORLDtoLEFT,
                                       p_dMotionScaling, SVI_STAGE_2), m_uNumberOfTracksStage2_2);
        // activity :1291-1312: landmarks with a failed / invalid optimisation leave, the others stay while their failed trackings are below the limit
        for (CDetectionPoint& cDetectionPoint : m_vecDetectionPointsActive) {
            std::vector<CLandmark*>& v = *cDetectionPoint.vecLandmarks;
            v.erase(std::remove_if(v.begin(), v.end(), [&](CLandmark* p) {
                        return p->uFailedSubsequentTrackings >= m_uMaximumFailedSubsequentTrackingsPerLandmark ||
                               std::find(vecDropped.begin(), vecDropped.end(), p) != vecDropped.end(); }), v.end());
        }
        m_vecDetectionPointsActive.erase(std::remove_if(m_vecDetectionPointsActive.begin(), m_vecDetectionPointsActive.end(),
                                                        [](const CDetectionPoint& d) { return d.vecLandmarks->empty(); }),
                                         m_vecDetectionPointsActive.end());
    }
    UIDLandmark getNumberOfTracksStage2_2() const { return m_uNumberOfTracksStage2_2; }

private:
    const std::shared_ptr<CGpuContext> m_pGpu;
    std::shared_ptr<CTriangulator> m_pTriangulator;
    const std::shared_ptr<CPinholeCamera> m_pCameraLEFT, m_pCameraRIGHT;
    const std::shared_ptr<CStereoCamera> m_pCameraSTEREO;
    const double m_dMinimumDepthMeters, m_dMaximumDepthMeters;
    const uint8_t m_uMaximumFailedSubsequentTrackingsPerLandmark = 5;   // CFundamentalMatcher.h:83
    UIDDetectionPoint m_uAvailableDetectionPointID = 0;
    std::vector<CDetectionPoint> m_vecDetectionPointsActive;
    std::vector<CLandmark*> m_vecVisibleLandmarks, m_vecLandmarksWINDOW;
    std::vector<const CMeasurementLandmark*> m_vecMeasurementsVisible;
    UIDLandmark m_uAvailableLandmarkID = 0, m_uNumberOfTracksStage1 = 0, m_uNumberOfTracksStage2_1 = 0, m_uNumberOfTracksStage2_2 = 0, m_uNumberOfTracksStage3 = 0;
    CSolverStereoPosit m_cSolverSterePosit;
    std::vector<CSolverStereoPosit::CMatch> m_vecMeasurementsStereoPositLAST;
    // packed arrays of optimizeActiveLandmarks (kept between frames: no allocation once they have grown)
    std::vector<CLandmark*> m_vecOptLandmarks;
    std::vector<double> m_vecOptGuess, m_vecOptXYZ, m_vecOptError;
    std::vector<int32_t> m_vecOptFirst, m_vecOptPoseIndex;
    std::vector<float> m_vecOptUVLEFT, m_vecOptUVRIGHT;
    std::vector<uint8_t> m_vecOptOutcome;
    CLandmark::CPoseTable m_cOptPoses;
};

#if defined(__GNUC__) && !defined(__clang__)
#pragma GCC pop_options
#endif
#endif
