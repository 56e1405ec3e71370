// CTriangulator -- same public interface as the reference's src/core/CTriangulator.h:54-81, with the
// OpenCV BRIEF / BFMatcher work done on the GPU behind the C-ABI of include/svi_gpu.h.
// Per-item failures come back as svi_status and are re-thrown as CExceptionNoMatchFound with the
// reference's what() text, so callers' catch blocks behave as before.  The cv::Mat& display
// parameters of the reference are dropped (documented deviation: no drawing).
#ifndef SVI_HOST_CTRIANGULATOR_H
#define SVI_HOST_CTRIANGULATOR_H

#include <memory>
#include <stdexcept>

#include "../../include/svi_gpu.h"
#include "CPinholeCamera.h"

// Pinned arithmetic: every product and sum below rounds on its own, in the written order (the GPU kernels and the CPU
// oracle do the same), whatever flags the including project uses -- the reference builds with -O3 -march=native
// (CMakeLists.txt:51), where GCC's default -ffp-contract=fast would fuse a*b + c into an FMA.
#if defined(__clang__)
#pragma clang fp contract(off)
#elif defined(__GNUC__)
#pragma GCC push_options
#pragma GCC optimize("fp-contract=off")
#endif

class CGpuContext {   // owns one svi_ctx (one per host thread and GPU)
public:
    CGpuContext(const std::shared_ptr<CStereoCamera> p_pStereoCamera, const svi_params* p_pParams = nullptr, int p_iDevice = 0) {
        svi_camera cL, cR;
        fill(cL, *p_pStereoCamera->m_pCameraLEFT);
        fill(cR, *p_pStereoCamera->m_pCameraRIGHT);
        if (p_pParams) params = *p_pParams; else svi_params_default(&params);
        if (SVI_SUCCESS != svi_create(&cL, &cR, &params, p_iDevice, &ctx))
            throw std::runtime_error(std::string("svi_create: ") + svi_last_error(nullptr));
    }
    ~CGpuContext() { svi_destroy(ctx); }
    CGpuContext(const CGpuContext&) = delete;
    CGpuContext& operator=(const CGpuContext&) = delete;
    void check(int rc) const { if (SVI_SUCCESS != rc) throw std::runtime_error(std::string("libsvi_gpu: ") + svi_last_error(ctx)); }
    // CStereoCamera.h:102-107: from here on every image handed to the library is a RAW camera image, undistorted and
    // rectified on the GPU with the maps cv::initUndistortRectifyMap builds from the members CPinholeCamera holds
    // (m_matIntrinsic, m_vecDistortionCoefficients, m_matRectification; new camera matrix m_matProjection).
    // p_bFloatMaps: the CV_32FC1 maps instead of CV_16SC2.
    void setRectification(const CStereoCamera& p_cCamera, bool p_bFloatMaps = false) {
        svi_rectification rL, rR;
        fill(rL, *p_cCamera.m_pCameraLEFT, p_bFloatMaps);
        fill(rR, *p_cCamera.m_pCameraRIGHT, p_bFloatMaps);
        check(svi_set_rectification(ctx, &rL, &rR));
    }
    void clearRectification() { check(svi_set_rectification(ctx, nullptr, nullptr)); }
    svi_ctx* ctx = nullptr;
    svi_params params;
private:
    static void fill(svi_camera& c, const CPinholeCamera& cam) {
        c.width = cam.m_uWidthPixel;
        c.height = cam.m_uHeightPixel;
        for (int i = 0; i < 12; ++i) c.P[i] = cam.m_matProjection.m[i];
    }
    static void fill(svi_rectification& r, const CPinholeCamera& cam, bool p_bFloatMaps) {
        for (int i = 0; i < 9; ++i) r.K[i] = cam.m_matIntrinsic.m[i];
        for (int i = 0; i < 4; ++i) r.D[i] = cam.m_vecDistortionCoefficients.v[i];
        for (int i = 0; i < 9; ++i) r.R[i] = cam.m_matRectification.m[i];
        r.float_maps = p_bFloatMaps ? 1 : 0;
    }
};

class CTriangulator {
public:
    CTriangulator(const std::shared_ptr<CStereoCamera> p_pStereoCamera, const std::shared_ptr<CGpuContext> p_pGpu)
        : m_pCameraSTEREO(p_pStereoCamera), m_pCameraLEFT(p_pStereoCamera->m_pCameraLEFT), m_pCameraRIGHT(p_pStereoCamera->m_pCameraRIGHT),
          m_pGpu(p_pGpu), m_fMatchingDistanceCutoff(p_pGpu->params.match_cutoff), m_dF(m_pCameraLEFT->m_matProjection(0, 0)), m_dFInverse(1 / m_dF),
          m_dPu(m_pCameraLEFT->m_matProjection(0, 2)), m_dPv(m_pCameraLEFT->m_matProjection(1, 2)), m_dDuR(m_pCameraRIGHT->m_matProjection(0, 3)),
          m_dDuRFlipped(-m_dDuR), dDepthMinimumMeters(m_dDuRFlipped / m_pCameraSTEREO->m_uPixelWidth),
          dDepthMaximumMeters(m_dDuRFlipped / CTriangulator::dMinimumDisparityPixels) {}

    static constexpr float fMinimumSearchRangePixels = 60.0;
    static constexpr double dMinimumDisparityPixels = 0.01;

    const std::shared_ptr<CStereoCamera> m_pCameraSTEREO;
    const std::shared_ptr<CPinholeCamera> m_pCameraLEFT, m_pCameraRIGHT;
    const std::shared_ptr<CGpuContext> m_pGpu;
    const float m_fMatchingDistanceCutoff;
    const double m_dF, m_dFInverse, m_dPu, m_dPv, m_dDuR, m_dDuRFlipped;
    const double dDepthMinimumMeters, dDepthMaximumMeters;

    // src/core/CTriangulator.cpp:185-253 (and the ...Full variant :51-119, identical without the display)
    const CMatchTriangulation getPointTriangulatedInRIGHT(const ImageView& p_matImageRIGHT, const float& p_fUTopLeft, const float& p_fVTopLeft,
                                                          const float& p_fKeyPointSizePixels, const Point2f& p_ptUVLEFT,
                                                          const CDescriptor& p_matReferenceDescriptorLEFT) const {
        const float tl[2] = {p_fUTopLeft, p_fVTopLeft}, uv[2] = {p_ptUVLEFT.x, p_ptUVLEFT.y};
        Out o;
        svi_tri_result r = o.result();
        m_pGpu->check(svi_triangulate_right(m_pGpu->ctx, p_matImageRIGHT.data, p_matImageRIGHT.pitch, 1, tl, uv, p_matReferenceDescriptorLEFT.data(),
                                            p_fKeyPointSizePixels, &r));
        return o.unwrap(false);
    }
    const CMatchTriangulation getPointTriangulatedInRIGHTFull(const ImageView& p_matImageRIGHT, const float& p_fUTopLeft, const float& p_fVTopLeft,
                                                              const float& p_fKeyPointSizePixels, const Point2f& p_ptUVLEFT,
                                                              const CDescriptor& p_matReferenceDescriptorLEFT) const {
        return getPointTriangulatedInRIGHT(p_matImageRIGHT, p_fUTopLeft, p_fVTopLeft, p_fKeyPointSizePixels, p_ptUVLEFT, p_matReferenceDescriptorLEFT);
    }
    // src/core/CTriangulator.cpp:255-324
    const CMatchTriangulation getPointTriangulatedInLEFT(const ImageView& p_matImageLEFT, const float& p_fSearchRange, const float& p_fUTopLeft,
                                                         const float& p_fVTopLeft, const float& p_fKeyPointSizePixels, const Point2f& p_ptUVRIGHT,
                                                         const CDescriptor& p_matReferenceDescriptorRIGHT) const {
        const float tl[2] = {p_fUTopLeft, p_fVTopLeft}, uv[2] = {p_ptUVRIGHT.x, p_ptUVRIGHT.y};
        Out o;
        svi_tri_result r = o.result();
        m_pGpu->check(svi_triangulate_left(m_pGpu->ctx, p_matImageLEFT.data, p_matImageLEFT.pitch, 1, &p_fSearchRange, tl, uv,
                                           p_matReferenceDescriptorRIGHT.data(), p_fKeyPointSizePixels, &r));
        return o.unwrap(true);
    }
    // src/core/CTriangulator.cpp:326-356
    const CPoint3DCAMERA getPointInLEFT(const Point2f& p_ptUVLEFT, const Point2f& p_ptUVRIGHT) const {
        const float l[2] = {p_ptUVLEFT.x, p_ptUVLEFT.y}, r[2] = {p_ptUVRIGHT.x, p_ptUVRIGHT.y};
        double xyz[3];
        uint8_t st;
        m_pGpu->check(svi_point_in_left(m_pGpu->ctx, 1, l, r, xyz, &st));
        if (SVI_OK != st) throw CExceptionNoMatchFound(svi_status_text(st), st);
        return CPoint3DCAMERA(xyz[0], xyz[1], xyz[2]);
    }

private:
    struct Out {
        float uv[2] = {0, 0};
        double xyz[3] = {0, 0, 0};
        CDescriptor desc{};
        int32_t dist = -1, idx = -1;
        uint8_t status = 0;
        svi_tri_result result() { return svi_tri_result{uv, xyz, desc.data(), &dist, &idx, &status}; }
        CMatchTriangulation unwrap(bool p_bLeft) const {
            if (SVI_OK != status) {
                std::string strText(svi_status_text(status));
                if (p_bLeft) {   // the LEFT variants throw the same texts with "InLEFT" (CTriangulator.cpp:270-322)
                    const std::string::size_type u = strText.find("InRIGHT");
                    if (std::string::npos != u) strText.replace(u, 7, "InLEFT");
                }
                throw CExceptionNoMatchFound(strText, status);
            }
            return CMatchTriangulation(CPoint3DCAMERA(xyz[0], xyz[1], xyz[2]), Point2f(uv[0], uv[1]), desc);
        }
    };
};

#if defined(__GNUC__) && !defined(__clang__)
#pragma GCC pop_options
#endif
#endif
