// sv_frame.cuh -- the device-side routing of one stereo-only tracking frame (svi_track_frame_stereo_only).
//
// The reference runs CTrackerSV::process as separate passes over the active landmarks: getPoseStereoPosit (stages 1 and 2 on the
// optimal landmarks, CSolverStereoPosit on their hits, once more with the damped prior if that fails) and trackEpipolar (stage 3
// where the camera moved since the landmark's detection, the regional stage 2 otherwise).  Here every such subset is an index list
// built on the device by an order-preserving compaction; the landmarks of a subset are gathered into the cascade's input arrays,
// the unchanged cascade kernels run on them, and their results are scattered back to full-n arrays.  The cascade kernels are
// per landmark, so the order of a subset only matters where the reference sums in it: the pose problem is assembled in candidate
// order, which is the measurement order of the solver's ordered sums.
#pragma once
#include "posit.cuh"
#include "track_plan.cuh"

namespace svi {

// route of a landmark (svi_sv_route of include/svi_gpu.h)
enum : uint8_t { kRoutePose = 1, kRouteEpipolar = 2, kRouteRegional = 3, kRouteRegionalNoTranslation = 4, kRouteDropped = 5 };

// The fields of the landmarks the cascade reads (svi_landmarks), for the whole frame or for a gathered subset.
struct SvLandmarksDev {
    double* xyz_w; uint8_t* desc_l; uint8_t* desc_r; float* disparity; float* size; double* uv_ref; uint8_t* desc_ref; double* T_det;
};

// Order-preserving compaction, one CTA: idx[0 .. *count) = the i in [0, n) with bit key[i] of `accept` set, ascending.  A block
// scan of warp ballots per chunk of kCompactThreads keys -- no atomics, the list is the same in every run.
constexpr int kCompactThreads = 1024;
__global__ void __launch_bounds__(kCompactThreads)
sv_compact_kernel(const uint8_t* __restrict__ key, int n, uint32_t accept, int* __restrict__ idx, int* __restrict__ count) {
    __shared__ int s_warp[kCompactThreads / 32];
    __shared__ int s_base;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int c0 = 0; c0 < n; c0 += kCompactThreads) {
        const int i = c0 + tid;
        bool take = false;
        if (i < n) {
            SVI_CHECK(11, i >= 0 && i < n);
            const uint32_t v = key[i];
            take = v < 32u && ((accept >> v) & 1u);
        }
        const uint32_t ballot = __ballot_sync(0xffffffffu, take);
        if (lane == 0) s_warp[warp] = __popc(ballot);
        __syncthreads();
        if (warp == 0) {   // inclusive scan of the 32 warp counts
            int v = s_warp[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, v, o);
                if (lane >= o) v += t;
            }
            s_warp[lane] = v;
        }
        __syncthreads();
        if (take) {
            const int slot = s_base + (warp ? s_warp[warp - 1] : 0) + __popc(ballot & ((1u << lane) - 1u));
            SVI_CHECK(11, slot >= 0 && slot < n);
            idx[slot] = i;
        }
        __syncthreads();
        if (tid == 0) s_base += s_warp[kCompactThreads / 32 - 1];
        __syncthreads();
    }
    if (tid == 0) *count = s_base;
}

__device__ __forceinline__ void copy32(uint8_t* dst, const uint8_t* src) {
    reinterpret_cast<uint4*>(dst)[0] = reinterpret_cast<const uint4*>(src)[0];
    reinterpret_cast<uint4*>(dst)[1] = reinterpret_cast<const uint4*>(src)[1];
}

// dst[j] = src[idx[j]] for j < *count (every field; n = entries of src and capacity of dst)
__global__ void sv_gather_kernel(SvLandmarksDev src, const int* __restrict__ idx, const int* __restrict__ count, int n, SvLandmarksDev dst) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= *count) return;
    SVI_CHECK(11, j >= 0 && j < n);
    const size_t i = (size_t)idx[j];
    SVI_CHECK(11, i < (size_t)n);
#pragma unroll
    for (int k = 0; k < 3; ++k) dst.xyz_w[3 * (size_t)j + k] = src.xyz_w[3 * i + k];
    copy32(dst.desc_l + 32 * (size_t)j, src.desc_l + 32 * i);
    copy32(dst.desc_r + 32 * (size_t)j, src.desc_r + 32 * i);
    copy32(dst.desc_ref + 32 * (size_t)j, src.desc_ref + 32 * i);
    dst.disparity[j] = src.disparity[i];
    dst.size[j] = src.size[i];
    dst.uv_ref[2 * (size_t)j] = src.uv_ref[2 * i];
    dst.uv_ref[2 * (size_t)j + 1] = src.uv_ref[2 * i + 1];
#pragma unroll
    for (int k = 0; k < 16; ++k) dst.T_det[16 * (size_t)j + k] = src.T_det[16 * i + k];
}

// The pose problem of one attempt (getPoseStereoPosit :525-534): the stage-1/2 hits of the gathered candidates, in candidate
// order (idx = the compaction of their stage bytes), become the solver's xyz_world / uv_left / uv_right.
__global__ void sv_posit_assemble_kernel(const int* __restrict__ idx, const int* __restrict__ count, int n, const double* __restrict__ xyz_w,
                                         TrackOutDev o, double* __restrict__ xyz, float* __restrict__ uv_l, float* __restrict__ uv_r) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= *count) return;
    SVI_CHECK(11, j >= 0 && j < n);
    const size_t i = (size_t)idx[j];
    SVI_CHECK(11, i < (size_t)n);
#pragma unroll
    for (int k = 0; k < 3; ++k) xyz[3 * (size_t)j + k] = xyz_w[3 * i + k];
    uv_l[2 * (size_t)j] = o.uv_l[2 * i]; uv_l[2 * (size_t)j + 1] = o.uv_l[2 * i + 1];
    uv_r[2 * (size_t)j] = o.uv_r[2 * i]; uv_r[2 * (size_t)j + 1] = o.uv_r[2 * i + 1];
}

// full[idx[j]] = sub[j] for j < *count, every result field.  route (may be null): a stage-3 item that found no translation since
// its landmark's detection (SVI_EPI_NO_TRANSLATION, :1804) moves to the regional stage 2, as trackEpipolar re-routes it.  With the
// split of sv_route_kernel in front of it this does not happen: epipolar_plan_dev sums the same products in the same order (only
// the host's leading 0.0 + is missing, which changes no non-zero sum), so an item routed to stage 3 has a non-zero translation
// there too.  The re-route stays so that the semantics are those of the composed calls whatever the two computations become.
__global__ void sv_scatter_kernel(const int* __restrict__ idx, const int* __restrict__ count, int n, TrackOutDev sub, TrackOutDev full,
                                  uint8_t* __restrict__ route) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= *count) return;
    SVI_CHECK(11, j >= 0 && j < n);
    const size_t i = (size_t)idx[j];
    SVI_CHECK(11, i < (size_t)n);
    full.status[i] = sub.status[j];
    full.stage[i] = sub.stage[j];
    full.uv_l[2 * i] = sub.uv_l[2 * (size_t)j]; full.uv_l[2 * i + 1] = sub.uv_l[2 * (size_t)j + 1];
    full.uv_r[2 * i] = sub.uv_r[2 * (size_t)j]; full.uv_r[2 * i + 1] = sub.uv_r[2 * (size_t)j + 1];
#pragma unroll
    for (int k = 0; k < 3; ++k) full.xyz[3 * i + k] = sub.xyz[3 * (size_t)j + k];
    copy32(full.desc_l + 32 * i, sub.desc_l + 32 * (size_t)j);
    copy32(full.desc_r + 32 * i, sub.desc_r + 32 * (size_t)j);
    if (route && sub.status[j] == SVI_EPI_NO_TRANSLATION) route[i] = kRouteRegionalNoTranslation;
}

struct SvPose { double T[16]; };   // WORLD->LEFT of the frame, row-major

// The split of trackEpipolar (:560-570) for the frame's pose T: a pose hit of the accepted solve was seen already; a landmark that
// leaves (flags bit 1: failed optimisation, or optimised and not optimal, :808-825) is dropped; the others go to the epipolar
// search when the camera moved since their detection, to the regional search otherwise.  "Moved" is the squared norm of the
// translation of T * T_left_to_world_at_detection, in the host's arithmetic: Isometry3d::operator* (host/Types.h:125, the sum
// starting at 0.0) and the sum order of CFundamentalMatcher.h:561-563, every operation rounded on its own.
__global__ void sv_route_kernel(int n, const uint8_t* __restrict__ flags, const uint8_t* __restrict__ pose_stage, int accepted, SvPose P,
                                const double* __restrict__ T_det, uint8_t* __restrict__ route) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    SVI_CHECK(11, i >= 0 && i < n);
    uint8_t r;
    if (accepted && pose_stage[i] > 0) r = kRoutePose;
    else if (flags[i] & 2) r = kRouteDropped;
    else {
        const double* B = T_det + 16 * (size_t)i;
        double t[3];
#pragma unroll
        for (int row = 0; row < 3; ++row) {
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < 3; ++k) s = __dadd_rn(s, __dmul_rn(P.T[4 * row + k], B[4 * k + 3]));
            t[row] = __dadd_rn(s, P.T[4 * row + 3]);
        }
        const double d2 = __dadd_rn(__dadd_rn(__dmul_rn(t[0], t[0]), __dmul_rn(t[1], t[1])), __dmul_rn(t[2], t[2]));
        r = (0.0 < d2) ? kRouteEpipolar : kRouteRegional;
    }
    route[i] = r;
}

}  // namespace svi
