// lr_check.cuh -- left-right consistency check of the dense new-landmark path's matches (optional mode:
// svi_params.lr_max_diff >= 0).
//
// Not a reference code path, but built from one: the reverse search is the reference's 7-argument
// CTriangulator::getPointTriangulatedInLEFT, the same triangulate_left_dev (plan, TMA window stage, unrolled pair tests,
// arg-min) that svi_triangulate_left and stage 1 RIGHT of the tracker run.  include/svi_gpu.h (svi_params.lr_max_diff)
// states the rule; tests/lr_check_np.py restates it on the CPU.  One launch per chunk after the matcher and before the
// sub-pixel refinement; it writes status only.
//
// Work decomposition: one warp per slot over the chunk's LEFT box-sum planes (map_l / map_ls: the shifted plane is written
// by the detector only while this mode is on), MATCH_WARPS slots per CTA with the scan-line kernels' shared-memory layout.
// A slot that is not SVI_OK returns before it touches shared memory.
#pragma once
#include "brief_match.cuh"

namespace svi {

struct LrCheckArgs {
    FrameGeom g;
    TriConst tc;
    float size, search_range;   // svi_params.keypoint_size, search_range_px
    float max_diff;             // svi_params.lr_max_diff >= 0
    const int* n_kp;            // [chunk frame] LEFT key-points (slots) of the frame
    int max_corners;
    StereoOutDev out;
    int out_frame0;
};

__global__ void __launch_bounds__(MATCH_WARPS * 32, 3)
lr_check_kernel(const __grid_constant__ CUtensorMap map_l, const __grid_constant__ CUtensorMap map_ls, const LrCheckArgs a) {
    extern __shared__ __align__(128) unsigned char match_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int f = blockIdx.y, slot = blockIdx.x * MATCH_WARPS + warp;
    if (slot >= min(a.n_kp[f], a.max_corners)) return;
    SVI_CHECK(14, slot < a.out.cap);
    const size_t o = (size_t)(a.out_frame0 + f) * a.out.cap + slot;
    if (a.out.status[o] != SVI_OK) return;   // warp-uniform
    PatchStage ps;
    patch_stage_init(ps, match_smem, &map_l, &map_ls, f * a.g.H, warp, lane);
    uint32_t ref[kDescWords];
    load_desc(a.out.desc_r + o * 32, ref);
    const float xl = a.out.uv_l[o * 2], y = a.out.uv_l[o * 2 + 1], xr = a.out.uv_r[o * 2];
    const float half = 4.f * a.size;
    SearchResult r;
    double xyz[3];
    triangulate_left_dev(a.g, a.tc, ps, a.search_range, __fsub_rn(xr, half), __fsub_rn(y, half), a.size, xr, ref, lane, r, xyz);
    const bool keep = r.status == SVI_OK && fabsf(__fsub_rn(r.u, xl)) <= a.max_diff;
    if (lane == 0 && !keep) a.out.status[o] = (uint8_t)SVI_LR_INCONSISTENT;
}

}  // namespace svi
