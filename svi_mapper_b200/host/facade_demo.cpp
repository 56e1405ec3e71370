// facade_demo -- drives the C++ host facade the way CTrackerGT::_trackLandmarks drives the reference
// (src/core/CTrackerGT.cpp:160-174, 305-319): addNewLandmarks on frame 0, trackManual on frame 1.
// Usage: facade_demo <left_calib> <right_calib> <W> <H> <L0.raw> <R0.raw> <L1.raw> <R1.raw> <out.txt>
// Writes one line per landmark of frame 0 and one per tracked landmark of frame 1 (parsed by the tests), then
// drives the SV/SVI entry points getPoseStereoPosit and trackEpipolar (src/core/CTrackerSV.cpp:274,324).
//        facade_demo --solver <left_calib> <right_calib> <matches.txt>
// CSolverStereoPosit alone (no GPU work): matches.txt holds "x y z uL vL uR vR" per line, the pose goes to stdout.
//        facade_demo --posit <left_calib> <right_calib> <problem.txt>
// CSolverStereoPosit with arbitrary priors, on the GPU (SVI_HOST_POSIT=cpu: the CPU loop, no GPU needed): problem.txt holds
// T_estimate (16 numbers), T_last (16), t_imu (3), then "x y z uL vL uR vR" per line; prints the 12 pose numbers and the
// iteration count, or FAILED <what()>.
//        facade_demo --sequence-sv <left_calib> <right_calib> <n> <L.raw> <R.raw> <max_corners> <out.txt>
// CTrackerSV::process over n frames without any pose given (see sequenceSVMain).
//        facade_demo --landmark <measurements.txt>
// CLandmark::optimize alone (no GPU work): first line "x y z" = first triangulation in the camera frame of measurement 0,
// then per line 16 numbers of LEFTtoWORLD... see landmarkMain; prints "x y z optimal successful failed".
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <string>
#include <vector>

#include "CGraphFile.h"
#include "CKeyFrameCloud.h"
#include "CTrackerGT.h"
#include "CTrackerSV.h"

static std::vector<uint8_t> readRaw(const char* path, size_t n) {
    std::vector<uint8_t> v(n);
    std::ifstream f(path, std::ios::binary);
    if (!f.read(reinterpret_cast<char*>(v.data()), (std::streamsize)n)) { std::fprintf(stderr, "cannot read %s\n", path); std::exit(2); }
    return v;
}

static int solverMain(char** argv) {
    try {
        CParameterBase::loadCameraLEFT(argv[2]);
        CParameterBase::loadCameraRIGHT(argv[3]);
        CSolverStereoPosit cSolver(CParameterBase::pCameraLEFT->m_matProjection, CParameterBase::pCameraRIGHT->m_matProjection);
        std::vector<CSolverStereoPosit::CMatch> vecMatches;
        std::ifstream f(argv[4]);
        double x, y, z;
        float uL, vL, uR, vR;
        while (f >> x >> y >> z >> uL >> vL >> uR >> vR)
            vecMatches.push_back(CSolverStereoPosit::CMatch(nullptr, CPoint3D(x, y, z), CPoint3D(), Point2f(uL, vL), Point2f(uR, vR), CDescriptor(), CDescriptor()));
        const Isometry3d matIdentity;
        const Isometry3d T(cSolver.getTransformationWORLDtoLEFT(matIdentity, CPoint3D(), matIdentity, vecMatches));
        for (int i = 0; i < 12; ++i) std::printf("%.17g%c", T.m[i], i == 11 ? '\n' : ' ');
    } catch (const CExceptionPoseOptimization& e) {
        std::printf("FAILED %s\n", e.what());
    } catch (const std::exception& e) {
        std::fprintf(stderr, "facade_demo failed: %s\n", e.what());
        return 1;
    }
    return 0;
}

static int positMain(char** argv) {
    try {
        CParameterBase::loadCameraLEFT(argv[2]);
        CParameterBase::loadCameraRIGHT(argv[3]);
        CParameterBase::constructCameraSTEREO(CPoint3D(-0.54, 0.0, 0.0));
        const char* e = std::getenv("SVI_HOST_POSIT");
        const bool bCPU = e && std::string(e) == "cpu";
        const std::shared_ptr<CGpuContext> pGpu(bCPU ? nullptr : std::make_shared<CGpuContext>(CParameterBase::pCameraSTEREO));
        CSolverStereoPosit cSolver(CParameterBase::pCameraLEFT->m_matProjection, CParameterBase::pCameraRIGHT->m_matProjection, pGpu);
        std::ifstream f(argv[4]);
        Isometry3d matEstimate, matLast;
        CPoint3D vecTranslationIMU;
        for (double& d : matEstimate.m) f >> d;
        for (double& d : matLast.m) f >> d;
        for (double& d : vecTranslationIMU.v) f >> d;
        if (!f) throw std::invalid_argument("malformed problem file");
        std::vector<CSolverStereoPosit::CMatch> vecMatches;
        double x, y, z;
        float uL, vL, uR, vR;
        while (f >> x >> y >> z >> uL >> vL >> uR >> vR)
            vecMatches.push_back(CSolverStereoPosit::CMatch(nullptr, CPoint3D(x, y, z), CPoint3D(), Point2f(uL, vL), Point2f(uR, vR), CDescriptor(), CDescriptor()));
        try {
            const Isometry3d T(cSolver.getTransformationWORLDtoLEFT(matLast, vecTranslationIMU, matEstimate, vecMatches));
            for (int i = 0; i < 12; ++i) std::printf("%.17g ", T.m[i]);
            std::printf("%u\n", cSolver.getIterationsLAST());
        } catch (const CExceptionPoseOptimization& e) {
            std::printf("FAILED %s\n", e.what());
        }
        if (const char* pTiming = std::getenv("SVI_DEMO_TIMING")) {   // the same solve SVI_DEMO_TIMING more times: median wall time of one call
            std::vector<double> vecMicroseconds;
            for (int k = std::max(1, std::atoi(pTiming)); k > 0; --k) {
                const auto t0 = std::chrono::steady_clock::now();
                try { cSolver.getTransformationWORLDtoLEFT(matLast, vecTranslationIMU, matEstimate, vecMatches); } catch (const CExceptionPoseOptimization&) {}
                vecMicroseconds.push_back(std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count());
            }
            std::sort(vecMicroseconds.begin(), vecMicroseconds.end());
            std::printf("{\"calls\": %zu, \"median_us\": %.3f, \"min_us\": %.3f}\n", vecMicroseconds.size(), vecMicroseconds[vecMicroseconds.size() / 2], vecMicroseconds[0]);
        }
    } catch (const std::exception& e) {
        std::fprintf(stderr, "facade_demo failed: %s\n", e.what());
        return 1;
    }
    return 0;
}

// --cloud <in.cloud> <out.cloud> <poses.txt>: read a key-frame cloud and write it back; print the relative motions of a
// KITTI pose file the way tracker_gt.cpp feeds them to the tracker (no GPU work)
static int cloudMain(char** argv) {
    try {
        Isometry3d T;
        const std::vector<CDescriptorVectorPoint3DWORLD> vecCloud(getCloudFromFile(argv[2], T));
        saveCloudToFile(argv[3], T, vecCloud);
        std::printf("POINTS %zu\n", vecCloud.size());
        const std::vector<Isometry3d> vecPoses(readPosesKITTI(argv[4]));
        for (size_t i = 0; i < vecPoses.size(); ++i) {
            const Isometry3d M(i ? getTransformationLEFTLASTtoLEFTNOW(vecPoses[i], vecPoses[i - 1]) : Isometry3d());
            std::printf("MOTION");
            for (int k = 0; k < 12; ++k) std::printf(" %.17g", M.m[k]);
            std::printf("\n");
        }
    } catch (const std::exception& e) {
        std::printf("FAILED %s\n", e.what());
    }
    return 0;
}

// --graph <in.txt> <out.g2o>: the g2o graph file of a hand-off described by a plain text file (no GPU work):
//   CAMERAS fxL fyL cxL cyL fxR fyR cxR cyR baseline | SHIFT x y z | LANDMARK id x y z |
//   KEYFRAME id <16 numbers LEFTtoWORLD> ax ay az | MEASUREMENT id uL vL uR vR x y z (belongs to the last KEYFRAME)
static int graphMain(char** argv) {
    try {
        std::ifstream ifIn(argv[2]);
        if (!ifIn.is_open()) throw std::invalid_argument("invalid graph description");
        CGraphCameras cCameras;
        CPoint3D vecShift;
        std::vector<CGraphKeyFrame> vecKeyFrames;
        std::vector<CGraphLandmark> vecLandmarks;
        std::string strTag;
        while (ifIn >> strTag) {
            if (strTag == "CAMERAS") {
                for (double& d : cCameras.dLEFT) ifIn >> d;
                for (double& d : cCameras.dRIGHT) ifIn >> d;
                ifIn >> cCameras.dBaselineMeters;
            } else if (strTag == "SHIFT") {
                ifIn >> vecShift.v[0] >> vecShift.v[1] >> vecShift.v[2];
            } else if (strTag == "LANDMARK") {
                CGraphLandmark l;
                ifIn >> l.uID >> l.vecPointXYZOptimized.v[0] >> l.vecPointXYZOptimized.v[1] >> l.vecPointXYZOptimized.v[2];
                vecLandmarks.push_back(l);
            } else if (strTag == "KEYFRAME") {
                CGraphKeyFrame k;
                ifIn >> k.uID;
                for (double& d : k.matTransformationLEFTtoWORLD.m) ifIn >> d;
                ifIn >> k.vecLinearAccelerationNormalized.v[0] >> k.vecLinearAccelerationNormalized.v[1] >> k.vecLinearAccelerationNormalized.v[2];
                vecKeyFrames.push_back(k);
            } else if (strTag == "MEASUREMENT" && !vecKeyFrames.empty()) {
                CGraphMeasurement m;
                ifIn >> m.uID >> m.ptUVLEFT.x >> m.ptUVLEFT.y >> m.ptUVRIGHT.x >> m.ptUVRIGHT.y >> m.vecPointXYZLEFT.v[0] >> m.vecPointXYZLEFT.v[1] >> m.vecPointXYZLEFT.v[2];
                vecKeyFrames.back().vecMeasurements.push_back(m);
            } else {
                throw std::invalid_argument("unknown tag " + strTag);
            }
            if (!ifIn) throw std::invalid_argument("malformed graph description");
        }
        saveGraphToFile(argv[3], cCameras, vecKeyFrames, vecLandmarks, vecShift);
        std::printf("GRAPH %zu keyframes %zu landmarks\n", vecKeyFrames.size(), vecLandmarks.size());
    } catch (const std::exception& e) {
        std::printf("FAILED %s\n", e.what());
    }
    return 0;
}

// measurements.txt: per line  P_WORLDtoLEFT (12) P_WORLDtoRIGHT (12) uL vL uR vR ; the first line is preceded by the initial
// world position "x y z".  The landmark is created at identity pose with that position, every line is one addMeasurement.
static int landmarkMain(char** argv) {
    std::ifstream f(argv[2]);
    double x, y, z;
    f >> x >> y >> z;
    const Isometry3d matIdentity;
    CLandmark* pLandmark = nullptr;
    MatrixProjection PL, PR;
    float uL, vL, uR, vR;
    while (true) {
        for (int i = 0; i < 12; ++i) f >> PL.m[i];
        for (int i = 0; i < 12; ++i) f >> PR.m[i];
        if (!(f >> uL >> vL >> uR >> vR)) break;
        if (!pLandmark) pLandmark = new CLandmark(0, CDescriptor(), CDescriptor(), 7.0, Point2f(uL, vL), Point2f(uR, vR), CPoint3D(x, y, z), matIdentity, matIdentity, PL, PR, 0);
        else pLandmark->addMeasurement(0, Point2f(uL, vL), Point2f(uR, vR), CDescriptor(), CDescriptor(), CPoint3D(x, y, z), matIdentity, matIdentity, PL, PR);
    }
    if (!pLandmark) return 2;
    pLandmark->optimize(0);
    if (std::getenv("SVI_DEMO_REPEAT")) {
        // host bookkeeping of the batched refinement, without the GPU: feed the CPU verdict through applyOptimization the way
        // optimizeActiveLandmarks does, and check when a failed optimisation may be repeated instead of recomputed
        const bool bFailed = 0 < pLandmark->uOptimizationsFailed;
        const uint8_t uOutcome = bFailed ? (uint8_t)SVI_OPT_NOT_CONVERGED : (pLandmark->bIsOptimal ? (0 < pLandmark->uOptimizationsSuccessful ? (uint8_t)SVI_OPT_OPTIMAL : (uint8_t)SVI_OPT_SKIPPED) : (uint8_t)SVI_OPT_CONVERGED);
        const double arrXYZ[3] = {pLandmark->vecPointXYZOptimized.x(), pLandmark->vecPointXYZOptimized.y(), pLandmark->vecPointXYZOptimized.z()};
        const uint32_t uFailedBefore = pLandmark->uOptimizationsFailed;
        if (bFailed) --pLandmark->uOptimizationsFailed; else if (0 < pLandmark->uOptimizationsSuccessful) --pLandmark->uOptimizationsSuccessful;
        pLandmark->applyOptimization(uOutcome, arrXYZ, pLandmark->dCurrentAverageSquaredError);
        const bool bRepeatAfterVerdict = pLandmark->isRepeatOfFailedOptimization();
        bool bCountersAgree = pLandmark->uOptimizationsFailed == uFailedBefore;
        if (bRepeatAfterVerdict) {
            pLandmark->repeatFailedOptimization();
            const uint32_t uAfterRepeat = pLandmark->uOptimizationsFailed;
            --pLandmark->uOptimizationsFailed;
            pLandmark->optimize(1);   // what the reference does in the next frame: the same failure again
            bCountersAgree = bCountersAgree && uAfterRepeat == pLandmark->uOptimizationsFailed && !pLandmark->bIsOptimal;
        }
        pLandmark->addMeasurement(1, Point2f(uL, vL), Point2f(uR, vR), CDescriptor(), CDescriptor(), CPoint3D(x, y, z), matIdentity, matIdentity, PL, PR);
        std::printf("REPEAT failed=%d repeat_after_verdict=%d counters_agree=%d repeat_after_new_measurement=%d\n", (int)bFailed, (int)bRepeatAfterVerdict,
                    (int)bCountersAgree, (int)pLandmark->isRepeatOfFailedOptimization());
        delete pLandmark;
        return 0;
    }
    std::printf("%.17g %.17g %.17g %d %u %u\n", pLandmark->vecPointXYZOptimized.x(), pLandmark->vecPointXYZOptimized.y(), pLandmark->vecPointXYZOptimized.z(),
                (int)pLandmark->bIsOptimal, pLandmark->uOptimizationsSuccessful, pLandmark->uOptimizationsFailed);
    delete pLandmark;
    return 0;
}

// --mask <left_calib> <right_calib> <centres.txt> <out.raw>: the detection mask of getMaskActiveLandmarks for the given
// centres ("x y" per line), written as a W x H u8 plane -- pinned against cv2.circle golden data by the tests
static int maskMain(char** argv) {
    try {
        CParameterBase::loadCameraLEFT(argv[2]);
        CParameterBase::loadCameraRIGHT(argv[3]);
        CParameterBase::constructCameraSTEREO(CPoint3D(-0.54, 0.0, 0.0));
        auto pGpu = std::make_shared<CGpuContext>(CParameterBase::pCameraSTEREO);
        CFundamentalMatcher cMatcher(CParameterBase::pCameraSTEREO, pGpu);
        std::vector<Point2f> vecCentres;
        std::ifstream f(argv[4]);
        float x, y;
        while (f >> x >> y) vecCentres.push_back(Point2f(x, y));
        const std::vector<uint8_t> matMask(cMatcher.getMaskForCentres(vecCentres));
        std::ofstream o(argv[5], std::ios::binary);
        o.write(reinterpret_cast<const char*>(matMask.data()), (std::streamsize)matMask.size());
    } catch (const std::exception& e) {
        std::fprintf(stderr, "facade_demo failed: %s\n", e.what());
        return 1;
    }
    return 0;
}

// --sequence <left_calib> <right_calib> <n> <L.raw> <R.raw> <motions.txt> <max_corners> <out.txt>: n frames (concatenated W x H
// planes) through CTrackerGT::process (track -> optimise -> re-detect), the per-frame relative motion LEFTLAST->LEFTNOW as
// 12 numbers + the rotation norm per line.  Prints, per frame, the counters, every visible landmark's measurement and the
// state of every active landmark after the frame -- compared line by line with the CPU restatement of the same loop.
// --sequence --rectify <left_calib> ...: the frames are RAW camera images, rectified on the GPU (CGpuContext::setRectification).
// With SVI_DEMO_TIMING set the per-frame dump is skipped and ONE line goes to stdout instead: the wall time of every
// process() call (frames after the first three), split into trackManual / landmark optimisation / re-detection.
static int sequenceMain(char** argv, bool p_bRectify) {
    try {
        CParameterBase::loadCameraLEFT(argv[2]);
        CParameterBase::loadCameraRIGHT(argv[3]);
        CParameterBase::constructCameraSTEREO(CPoint3D(-0.54, 0.0, 0.0));
        const int W = (int)CParameterBase::pCameraLEFT->m_uWidthPixel, H = (int)CParameterBase::pCameraLEFT->m_uHeightPixel;
        const int n = std::atoi(argv[4]);
        const std::vector<uint8_t> L = readRaw(argv[5], (size_t)n * W * H), R = readRaw(argv[6], (size_t)n * W * H);
        std::ifstream fm(argv[7]);
        svi_params p;
        svi_params_default(&p);
        p.max_corners = std::atoi(argv[8]);
        auto pGpu = std::make_shared<CGpuContext>(CParameterBase::pCameraSTEREO, &p);
        if (p_bRectify) pGpu->setRectification(*CParameterBase::pCameraSTEREO);
        CTrackerGT cTracker(CParameterBase::pCameraSTEREO, pGpu);
        const bool bTiming = std::getenv("SVI_DEMO_TIMING") != nullptr;
        std::FILE* out = bTiming ? nullptr : std::fopen(argv[9], "w");
        std::vector<double> vecFrameMilliseconds;
        double dWarmTracking = 0.0, dWarmOptimization = 0.0, dWarmDetection = 0.0;
        size_t uLandmarksTracked = 0;
        for (int t = 0; t < n; ++t) {
            Isometry3d M;
            double dRotationNorm = 0.0;
            for (int i = 0; i < 12; ++i) fm >> M.m[i];
            fm >> dRotationNorm;
            if (t == 3) {
                dWarmTracking = cTracker.getDurationTrackingSeconds();
                dWarmOptimization = cTracker.getDurationOptimizationSeconds();
                dWarmDetection = cTracker.getDurationDetectionSeconds();
            }
            const size_t uActiveBefore = cTracker.getMatcher().getNumberOfActiveLandmarks();
            const auto t0 = std::chrono::steady_clock::now();
            cTracker.process(ImageView(L.data() + (size_t)t * W * H, W, H), ImageView(R.data() + (size_t)t * W * H, W, H), M, dRotationNorm);
            if (t >= 3) {
                vecFrameMilliseconds.push_back(std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
                uLandmarksTracked += uActiveBefore;
            }
            if (bTiming) continue;
            CFundamentalMatcher& m = cTracker.getMatcher();
            std::fprintf(out, "F %d VISIBLE %lu ACTIVE %zu S1 %lu S2 %lu S3 %lu DETECTIONS %lu\n", t, (unsigned long)cTracker.getNumberOfVisibleLandmarksLAST(),
                         m.getNumberOfActiveLandmarks(), (unsigned long)m.getNumberOfTracksStage1(), (unsigned long)m.getNumberOfTracksStage2_1(),
                         (unsigned long)m.getNumberOfTracksStage3(), (unsigned long)cTracker.getNumberOfDetections());
            for (const CMeasurementLandmark* q : m.getMeasurementsForVisibleLandmarks())
                std::fprintf(out, "M %lu %.9g %.9g %.9g %.9g %.17g %.17g %.17g\n", (unsigned long)q->uID, q->ptUVLEFT.x, q->ptUVLEFT.y, q->ptUVRIGHT.x,
                             q->ptUVRIGHT.y, q->vecPointXYZLEFT.x(), q->vecPointXYZLEFT.y(), q->vecPointXYZLEFT.z());
            for (const CLandmark* q : m.getActiveLandmarks())
                std::fprintf(out, "A %lu %.17g %.17g %.17g %d %d %u %u %u %zu\n", (unsigned long)q->uID, q->vecPointXYZOptimized.x(), q->vecPointXYZOptimized.y(),
                             q->vecPointXYZOptimized.z(), (int)q->bIsOptimal, (int)q->bIsCurrentlyVisible, q->uOptimizationsSuccessful, q->uOptimizationsFailed,
                             (unsigned)q->uFailedSubsequentTrackings, q->getNumberOfMeasurements());
        }
        if (out) std::fclose(out);
        if (bTiming && !vecFrameMilliseconds.empty()) {
            double dTotal = 0.0;
            for (const double d : vecFrameMilliseconds) dTotal += d;
            std::vector<double> vecSorted(vecFrameMilliseconds);
            std::sort(vecSorted.begin(), vecSorted.end());
            std::printf("{\"frames\": %zu, \"total_ms\": %.4f, \"median_ms\": %.4f, \"track_manual_ms\": %.4f, \"optimize_ms\": %.4f, "
                        "\"add_new_landmarks_ms\": %.4f, \"landmarks_tracked\": %zu, \"detections\": %lu}\n",
                        vecFrameMilliseconds.size(), dTotal, vecSorted[vecSorted.size() / 2],
                        1e3 * (cTracker.getDurationTrackingSeconds() - dWarmTracking), 1e3 * (cTracker.getDurationOptimizationSeconds() - dWarmOptimization),
                        1e3 * (cTracker.getDurationDetectionSeconds() - dWarmDetection), uLandmarksTracked, (unsigned long)cTracker.getNumberOfDetections());
        }
    } catch (const std::exception& e) {
        std::fprintf(stderr, "facade_demo failed: %s\n", e.what());
        return 1;
    }
    return 0;
}

// --sequence-sv <left_calib> <right_calib> <n> <L.raw> <R.raw> <max_corners> <out.txt>: n frames through CTrackerSV::process --
// the stereo-only tracker, no pose given: each frame's pose comes from getPoseStereoPosit (CSolverStereoPosit on the GPU;
// SVI_HOST_POSIT=cpu: the CPU loop).  Prints, per frame, the pose source, the counters and the 12 numbers of T_WORLDtoLEFT,
// then the M / A lines of --sequence.  With SVI_DEMO_TIMING set ONE line goes to stdout instead: the wall time of every
// process() call (frames after the first three), split into pose stage (tracking + solves), solves alone, trackEpipolar,
// landmark optimisation and re-detection.
static int sequenceSVMain(char** argv) {
    try {
        CParameterBase::loadCameraLEFT(argv[2]);
        CParameterBase::loadCameraRIGHT(argv[3]);
        CParameterBase::constructCameraSTEREO(CPoint3D(-0.54, 0.0, 0.0));
        const int W = (int)CParameterBase::pCameraLEFT->m_uWidthPixel, H = (int)CParameterBase::pCameraLEFT->m_uHeightPixel;
        const int n = std::atoi(argv[4]);
        const std::vector<uint8_t> L = readRaw(argv[5], (size_t)n * W * H), R = readRaw(argv[6], (size_t)n * W * H);
        svi_params p;
        svi_params_default(&p);
        p.max_corners = std::atoi(argv[7]);
        auto pGpu = std::make_shared<CGpuContext>(CParameterBase::pCameraSTEREO, &p);
        CTrackerSV cTracker(CParameterBase::pCameraSTEREO, pGpu);
        const bool bTiming = std::getenv("SVI_DEMO_TIMING") != nullptr;
        std::FILE* out = bTiming ? nullptr : std::fopen(argv[8], "w");
        std::vector<double> vecFrameMilliseconds;
        double dWarm[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
        auto durations = [&cTracker](double (&d)[5]) {
            d[0] = cTracker.getDurationPoseSeconds(); d[1] = cTracker.getDurationPoseSolverSeconds(); d[2] = cTracker.getDurationTrackEpipolarSeconds();
            d[3] = cTracker.getDurationOptimizationSeconds(); d[4] = cTracker.getDurationDetectionSeconds();
        };
        size_t uMeasurementsPosit = 0, uFramesPosit = 0;
        for (int t = 0; t < n; ++t) {
            if (t == 3) durations(dWarm);
            const auto t0 = std::chrono::steady_clock::now();
            cTracker.process(ImageView(L.data() + (size_t)t * W * H, W, H), ImageView(R.data() + (size_t)t * W * H, W, H));
            CFundamentalMatcher& m = cTracker.getMatcher();
            if (t >= 3) {
                vecFrameMilliseconds.push_back(std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
                uMeasurementsPosit += m.getMeasurementsStereoPositLAST().size();
                ++uFramesPosit;
            }
            if (bTiming) continue;
            const Isometry3d& T = cTracker.getTransformationWORLDtoLEFT();
            std::fprintf(out, "F %d POSE %s VISIBLE %lu ACTIVE %zu S1 %lu S2 %lu S3 %lu S22 %lu DETECTIONS %lu INSTABILITY %d POSIT %zu T", t,
                         cTracker.getPoseSource().c_str(), (unsigned long)cTracker.getNumberOfVisibleLandmarksLAST(), m.getNumberOfActiveLandmarks(),
                         (unsigned long)m.getNumberOfTracksStage1(), (unsigned long)m.getNumberOfTracksStage2_1(), (unsigned long)m.getNumberOfTracksStage3(),
                         (unsigned long)m.getNumberOfTracksStage2_2(), (unsigned long)cTracker.getNumberOfDetections(), (int)cTracker.getCountInstability(),
                         m.getMeasurementsStereoPositLAST().size());
            for (int i = 0; i < 12; ++i) std::fprintf(out, " %.17g", T.m[i]);
            std::fprintf(out, "\n");
            for (const CMeasurementLandmark* q : m.getMeasurementsForVisibleLandmarks())
                std::fprintf(out, "M %lu %.9g %.9g %.9g %.9g %.17g %.17g %.17g\n", (unsigned long)q->uID, q->ptUVLEFT.x, q->ptUVLEFT.y, q->ptUVRIGHT.x,
                             q->ptUVRIGHT.y, q->vecPointXYZLEFT.x(), q->vecPointXYZLEFT.y(), q->vecPointXYZLEFT.z());
            for (const CLandmark* q : m.getActiveLandmarks())
                std::fprintf(out, "A %lu %.17g %.17g %.17g %d %d %u %u %u %zu\n", (unsigned long)q->uID, q->vecPointXYZOptimized.x(), q->vecPointXYZOptimized.y(),
                             q->vecPointXYZOptimized.z(), (int)q->bIsOptimal, (int)q->bIsCurrentlyVisible, q->uOptimizationsSuccessful, q->uOptimizationsFailed,
                             (unsigned)q->uFailedSubsequentTrackings, q->getNumberOfMeasurements());
        }
        if (out) std::fclose(out);
        if (bTiming && !vecFrameMilliseconds.empty()) {
            double dTotal = 0.0, dNow[5];
            for (const double d : vecFrameMilliseconds) dTotal += d;
            std::vector<double> vecSorted(vecFrameMilliseconds);
            std::sort(vecSorted.begin(), vecSorted.end());
            durations(dNow);
            std::printf("{\"frames\": %zu, \"total_ms\": %.4f, \"median_ms\": %.4f, \"pose_ms\": %.4f, \"pose_solver_ms\": %.4f, \"track_epipolar_ms\": %.4f, "
                        "\"optimize_ms\": %.4f, \"add_new_landmarks_ms\": %.4f, \"posit_measurements_mean\": %.1f, \"detections\": %lu}\n",
                        vecFrameMilliseconds.size(), dTotal, vecSorted[vecSorted.size() / 2], 1e3 * (dNow[0] - dWarm[0]), 1e3 * (dNow[1] - dWarm[1]),
                        1e3 * (dNow[2] - dWarm[2]), 1e3 * (dNow[3] - dWarm[3]), 1e3 * (dNow[4] - dWarm[4]),
                        (double)uMeasurementsPosit / (double)std::max<size_t>(1, uFramesPosit), (unsigned long)cTracker.getNumberOfDetections());
        }
    } catch (const std::exception& e) {
        std::fprintf(stderr, "facade_demo failed: %s\n", e.what());
        return 1;
    }
    return 0;
}

int main(int argc, char** argv) {
    if (argc == 10 && std::string(argv[1]) == "--sequence") return sequenceMain(argv, false);
    if (argc == 11 && std::string(argv[1]) == "--sequence" && std::string(argv[2]) == "--rectify") {
        return sequenceMain(argv + 1, true);   // the remaining arguments keep their positions
    }
    if (argc == 5 && std::string(argv[1]) == "--solver") return solverMain(argv);
    if (argc == 5 && std::string(argv[1]) == "--posit") return positMain(argv);
    if (argc == 9 && std::string(argv[1]) == "--sequence-sv") return sequenceSVMain(argv);
    if (argc == 6 && std::string(argv[1]) == "--mask") return maskMain(argv);
    if (argc == 3 && std::string(argv[1]) == "--landmark") return landmarkMain(argv);
    if (argc == 5 && std::string(argv[1]) == "--cloud") return cloudMain(argv);
    if (argc == 4 && std::string(argv[1]) == "--graph") return graphMain(argv);
    if (argc < 10) { std::fprintf(stderr, "usage: see source\n"); return 2; }
    try {
        CParameterBase::loadCameraLEFT(argv[1]);
        CParameterBase::loadCameraRIGHT(argv[2]);
        CParameterBase::constructCameraSTEREO(CPoint3D(-0.54, 0.0, 0.0));   // tracker_gt.cpp:123
        const int W = std::atoi(argv[3]), H = std::atoi(argv[4]);
        if (W != (int)CParameterBase::pCameraLEFT->m_uWidthPixel || H != (int)CParameterBase::pCameraLEFT->m_uHeightPixel) {
            std::fprintf(stderr, "image size does not match the calibration\n");
            return 2;
        }
        const std::vector<uint8_t> L0 = readRaw(argv[5], (size_t)W * H), R0 = readRaw(argv[6], (size_t)W * H);
        const std::vector<uint8_t> L1 = readRaw(argv[7], (size_t)W * H), R1 = readRaw(argv[8], (size_t)W * H);
        auto pGpu = std::make_shared<CGpuContext>(CParameterBase::pCameraSTEREO);
        CFundamentalMatcher cMatcher(CParameterBase::pCameraSTEREO, pGpu);
        const Isometry3d matIdentity;
        std::FILE* out = std::fopen(argv[9], "w");
        const size_t n = cMatcher.addNewLandmarks(ImageView(L0.data(), W, H), ImageView(R0.data(), W, H), matIdentity, matIdentity, 0);
        std::fprintf(out, "NEW %zu\n", n);
        for (const CLandmark* p : cMatcher.getLandmarksWINDOW()) {
            const CMeasurementLandmark* m = p->getLastMeasurement();
            std::fprintf(out, "L %lu %.1f %.1f %.1f %.1f %.17g %.17g %.17g\n", (unsigned long)p->uID, m->ptUVLEFT.x, m->ptUVLEFT.y, m->ptUVRIGHT.x,
                         m->ptUVRIGHT.y, m->vecPointXYZLEFT.x(), m->vecPointXYZLEFT.y(), m->vecPointXYZLEFT.z());
        }
        cMatcher.resetVisibilityActiveLandmarks();
        cMatcher.trackManual(1, ImageView(L1.data(), W, H), ImageView(R1.data(), W, H), matIdentity, matIdentity, 1.0);
        std::fprintf(out, "TRACKED %lu STAGE2 %lu STAGE3 %lu VISIBLE %zu\n", (unsigned long)cMatcher.getNumberOfTracksStage1(),
                     (unsigned long)cMatcher.getNumberOfTracksStage2_1(), (unsigned long)cMatcher.getNumberOfTracksStage3(),
                     cMatcher.getNumberOfVisibleLandmarks());
        for (const CMeasurementLandmark* m : cMatcher.getMeasurementsForVisibleLandmarks())
            std::fprintf(out, "T %lu %.1f %.1f %.1f %.1f %.17g\n", (unsigned long)m->uID, m->ptUVLEFT.x, m->ptUVLEFT.y, m->ptUVRIGHT.x, m->ptUVRIGHT.y,
                         m->vecPointXYZLEFT.z());
        // scalar CTriangulator calls with exception semantics
        const auto tri = cMatcher.getTriangulator();
        try {
            tri->getPointInLEFT(Point2f(100.f, 50.f), Point2f(100.f, 50.f));
            std::fprintf(out, "EXC none\n");
        } catch (const CExceptionNoMatchFound& e) {
            std::fprintf(out, "EXC %s\n", e.what());
        }
        // a short sequence through the CTrackerGT orchestration: the same pair shown 6 times while the camera is
        // reported to move 1 cm per frame along x (tracker_gt.cpp feeds ground-truth poses the same way)
        CTrackerGT cTracker(CParameterBase::pCameraSTEREO, pGpu);
        Isometry3d matStep;
        matStep(0, 3) = 0.01;
        for (int uFrame = 0; uFrame < 6; ++uFrame) {
            cTracker.process(ImageView(L0.data(), W, H), ImageView(R0.data(), W, H), uFrame ? matStep : matIdentity);
            std::fprintf(out, "SEQ %d VISIBLE %lu TOTAL %lu S1 %lu S2 %lu S3 %lu DETECTIONS %lu\n", uFrame,
                         (unsigned long)cTracker.getNumberOfVisibleLandmarksLAST(), (unsigned long)cTracker.getMatcher().getNumberOfLandmarksTotal(),
                         (unsigned long)cTracker.getMatcher().getNumberOfTracksStage1(), (unsigned long)cTracker.getMatcher().getNumberOfTracksStage2_1(),
                         (unsigned long)cTracker.getMatcher().getNumberOfTracksStage3(), (unsigned long)cTracker.getNumberOfDetections());
        }
        if (argc > 10) {   // key-frame cloud of what the sequence tracker sees now (CKeyFrame::saveCloudToFile)
            std::vector<CLandmark*> vecVisible;
            for (CLandmark* p : cTracker.getMatcher().getLandmarksWINDOW()) if (p->bIsCurrentlyVisible) vecVisible.push_back(p);
            saveCloudToFile(argv[10], cTracker.getTransformationLEFTtoWORLD(), getCloudForVisibleOptimizedLandmarks(vecVisible));
        }
        // the SV/SVI entry points on a fresh matcher: frame 1 = pose from the stereo measurements of stages 1-2, frame 2 =
        // nothing seen yet and the camera 2 cm away from the detection pose (epipolar branch), frame 3 = nothing seen
        // yet at the detection pose (regional branch)
        CFundamentalMatcher cMatcherSV(CParameterBase::pCameraSTEREO, pGpu);
        cMatcherSV.addNewLandmarks(ImageView(L0.data(), W, H), ImageView(R0.data(), W, H), matIdentity, matIdentity, 0);
        cMatcherSV.resetVisibilityActiveLandmarks();
        try {
            const Isometry3d T(cMatcherSV.getPoseStereoPosit(1, ImageView(L1.data(), W, H), ImageView(R1.data(), W, H), matIdentity, matIdentity, CPoint3D(), CPoint3D(), 1.0));
            std::fprintf(out, "POSIT %zu S1 %lu S2 %lu VISIBLE %zu POSE", cMatcherSV.getMeasurementsStereoPositLAST().size(), (unsigned long)cMatcherSV.getNumberOfTracksStage1(),
                         (unsigned long)cMatcherSV.getNumberOfTracksStage2_1(), cMatcherSV.getNumberOfVisibleLandmarks());
            for (int i = 0; i < 12; ++i) std::fprintf(out, " %.17g", T.m[i]);
            std::fprintf(out, "\n");
        } catch (const CExceptionPoseOptimization& e) {
            std::fprintf(out, "POSIT_FAILED %s\n", e.what());
        }
        Isometry3d matMoved;
        matMoved(0, 3) = 0.02;
        cMatcherSV.resetVisibilityActiveLandmarks();
        cMatcherSV.trackEpipolar(2, ImageView(L1.data(), W, H), ImageView(R1.data(), W, H), matMoved, inverseIsometry(matMoved), 1.5);
        std::fprintf(out, "EPI 2 S3 %lu S22 %lu VISIBLE %zu\n", (unsigned long)cMatcherSV.getNumberOfTracksStage3(), (unsigned long)cMatcherSV.getNumberOfTracksStage2_2(),
                     cMatcherSV.getNumberOfVisibleLandmarks());
        cMatcherSV.resetVisibilityActiveLandmarks();
        cMatcherSV.trackEpipolar(3, ImageView(L1.data(), W, H), ImageView(R1.data(), W, H), matIdentity, matIdentity, 1.0);
        std::fprintf(out, "EPI 3 S3 %lu S22 %lu VISIBLE %zu\n", (unsigned long)cMatcherSV.getNumberOfTracksStage3(), (unsigned long)cMatcherSV.getNumberOfTracksStage2_2(),
                     cMatcherSV.getNumberOfVisibleLandmarks());
        // the stereo-only tracker: no ground truth, the pose comes from the stereo measurements.  The scene is static (the
        // same pair every frame), so the recovered pose has to stay at the origin while landmarks are detected, tracked,
        // optimised and re-detected.
        CTrackerSV cTrackerSV(CParameterBase::pCameraSTEREO, pGpu);
        for (int uFrame = 0; uFrame < 12; ++uFrame) {
            cTrackerSV.process(ImageView(L0.data(), W, H), ImageView(R0.data(), W, H));
            const Isometry3d& T = cTrackerSV.getTransformationWORLDtoLEFT();
            std::fprintf(out, "SV %d VISIBLE %lu TOTAL %lu S1 %lu S2 %lu S3 %lu S22 %lu DETECTIONS %lu POSE %s T %.9g %.9g %.9g\n", uFrame,
                         (unsigned long)cTrackerSV.getNumberOfVisibleLandmarksLAST(), (unsigned long)cTrackerSV.getMatcher().getNumberOfLandmarksTotal(),
                         (unsigned long)cTrackerSV.getMatcher().getNumberOfTracksStage1(), (unsigned long)cTrackerSV.getMatcher().getNumberOfTracksStage2_1(),
                         (unsigned long)cTrackerSV.getMatcher().getNumberOfTracksStage3(), (unsigned long)cTrackerSV.getMatcher().getNumberOfTracksStage2_2(),
                         (unsigned long)cTrackerSV.getNumberOfDetections(), cTrackerSV.getPoseSource().c_str(), T(0, 3), T(1, 3), T(2, 3));
        }
        std::fclose(out);
    } catch (const std::exception& e) {
        std::fprintf(stderr, "facade_demo failed: %s\n", e.what());
        return 1;
    }
    return 0;
}
