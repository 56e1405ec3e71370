// rectify.cuh -- undistortion + rectification of raw camera images on the device: cv::remap(raw, out, map1, map2,
// INTER_LINEAR, BORDER_CONSTANT 0) on u8 with the CV_16SC2 maps of cv::initUndistortRectifyMap, bit for bit
// (CStereoCamera.h:102-107 of the reference; DESIGN.md section 2 has the pins).
//
// Arithmetic (OpenCV's fixed-point bilinear path): a map entry is an integer source pixel (sx, sy) plus 5-bit fractions
// (fx, fy); the four tap weights are rint(float32(1 - ty or ty) * float32(1 - tx or tx) * 32768) of initInterTab2D --
// with 5-bit fractions every product is exact, so the weights are the integers (32 - fy or fy) * (32 - fx or fx) * 32 and
// always sum to 32768 (no fix-up) -- and the result is (sum of tap * weight + 2^14) >> 15.  A tap outside the image reads
// the border value 0; the other taps still count.
//
// Layout: a CTA owns RECT_THREADS * 4 consecutive output pixels of the dense W x H plane (flat index, rows wrap) and walks
// up to RECT_FRAMES frames of the chunk, so each map entry is read once per 16 frames; blockIdx.y selects the camera,
// blockIdx.z the group of frames.  The map is 6 bytes per pixel (short2 source + uint16 fractions), padded to a multiple
// of 8 pixels so a thread reads its 4 entries with one 16-byte and one 8-byte load; the taps are gathered through L1
// (neighbouring outputs share them).
#pragma once
#include "common.cuh"

namespace svi {

constexpr int RECT_THREADS = 256;
constexpr int RECT_PX = 4;   // output pixels per thread: one 32-bit store per frame
constexpr int RECT_FRAMES = 16;   // frames a CTA walks: its map entries are read once per 16 frames of the chunk

struct RectifySide {
    const short2* xy;        // [n_pad] integer source column / row
    const uint16_t* frac;    // [n_pad] fy * 32 + fx
    const uint8_t* src;      // raw frame 0 (src_pitch bytes per row, src_stride bytes per frame)
    uint8_t* dst;            // rectified frame 0 (W bytes per row, dst_stride bytes per frame)
};

struct RectifyArgs {
    RectifySide cam[2];
    int W, H, n_pix, n_pad, nf;
    size_t src_pitch, src_stride, dst_stride;
};

__device__ __forceinline__ uint32_t rect_tap(const uint8_t* img, int x, int y, int W, int H, size_t pitch) {
    if ((unsigned)x >= (unsigned)W || (unsigned)y >= (unsigned)H) return 0u;   // BORDER_CONSTANT 0
    SVI_CHECK(9, (size_t)x < pitch);
    return __ldg(img + (size_t)y * pitch + x);
}

// grid: (quads of the plane / RECT_THREADS, cameras, frame groups of RECT_FRAMES)
__global__ void __launch_bounds__(RECT_THREADS) rectify_kernel(const RectifyArgs a) {
    // every field in registers (indexing the parameter struct with blockIdx.y would copy it to local memory)
    const int W = a.W, H = a.H, n_pix = a.n_pix;
    const size_t pitch = a.src_pitch, src_stride = a.src_stride, dst_stride = a.dst_stride;
    const RectifySide cam = blockIdx.y ? a.cam[1] : a.cam[0];
    const int p0 = (blockIdx.x * RECT_THREADS + threadIdx.x) * RECT_PX;
    const int f_begin = blockIdx.z * RECT_FRAMES, f_end = min(a.nf, f_begin + RECT_FRAMES);
    if (p0 >= n_pix) return;
    SVI_CHECK(9, p0 + RECT_PX <= a.n_pad);
    const int4 xy4 = __ldg(reinterpret_cast<const int4*>(cam.xy + p0));
    const uint2 fr2 = __ldg(reinterpret_cast<const uint2*>(cam.frac + p0));
    const uint32_t xyw[4] = {(uint32_t)xy4.x, (uint32_t)xy4.y, (uint32_t)xy4.z, (uint32_t)xy4.w};
    const uint32_t frw[4] = {fr2.x & 0xFFFFu, fr2.x >> 16, fr2.y & 0xFFFFu, fr2.y >> 16};
    int sx[RECT_PX], sy[RECT_PX];
    uint32_t w00[RECT_PX], w01[RECT_PX], w10[RECT_PX], w11[RECT_PX];
#pragma unroll
    for (int k = 0; k < RECT_PX; ++k) {
        sx[k] = (int)(int16_t)(xyw[k] & 0xFFFFu);
        sy[k] = (int)(int16_t)(xyw[k] >> 16);
        const uint32_t fx = frw[k] & 31u, fy = (frw[k] >> 5) & 31u;
        w00[k] = (32u - fy) * (32u - fx) * 32u;
        w01[k] = (32u - fy) * fx * 32u;
        w10[k] = fy * (32u - fx) * 32u;
        w11[k] = fy * fx * 32u;
    }
    const int live = min(RECT_PX, n_pix - p0);
    SVI_CHECK(9, p0 + live <= n_pix);
#pragma unroll 4
    for (int f = f_begin; f < f_end; ++f) {
        const uint8_t* img = cam.src + (size_t)f * src_stride;
        uint32_t packed = 0;
#pragma unroll
        for (int k = 0; k < RECT_PX; ++k) {
            const uint32_t acc = rect_tap(img, sx[k], sy[k], W, H, pitch) * w00[k] + rect_tap(img, sx[k] + 1, sy[k], W, H, pitch) * w01[k] +
                                 rect_tap(img, sx[k], sy[k] + 1, W, H, pitch) * w10[k] + rect_tap(img, sx[k] + 1, sy[k] + 1, W, H, pitch) * w11[k];
            packed |= ((acc + (1u << 14)) >> 15) << (8 * k);
        }
        uint8_t* out = cam.dst + (size_t)f * dst_stride + p0;
        if (live == RECT_PX && (reinterpret_cast<uintptr_t>(out) & 3u) == 0) {
            *reinterpret_cast<uint32_t*>(out) = packed;
        } else {
            for (int k = 0; k < live; ++k) out[k] = (uint8_t)(packed >> (8 * k));
        }
    }
}

}  // namespace svi
