// svi_gpu.cu -- libsvi_gpu.so: context, scratch management, kernel pipeline and the C-ABI of
// include/svi_gpu.h.  sm_100a only; there is no CPU fallback anywhere in this file.
//
// Execution model.  A batch of independent stereo pairs is cut into chunks of `chunk_frames`
// frames; chunk c runs on lane c % n_lanes.  A lane is one CUDA stream plus the scratch of one
// chunk (box-sum planes of both images, candidate lists, corner lists, bin lists); different lanes overlap
// each other's copies, wide kernels (Harris, match) and the one-CTA-per-frame selection kernel.
// Per-query entry points (triangulate, describe, track, landmark refinement) run on lane 0's stream.
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <string>
#include <thread>
#include <vector>

#include "../../include/svi_gpu.h"
#include "band_match.cuh"
#include "brief_match.cuh"
#include "binned.cuh"
#include "harris.cuh"
#include "landmark_opt.cuh"
#include "posit.cuh"
#include "rectify.cuh"
#include "select.cuh"
#include "sv_frame.cuh"
#include "track_plan.cuh"

using namespace svi;

namespace {

constexpr int kMaxLanes = 8;
constexpr int kSmallFrames = 2;          // calls of up to this many frames go through the pinned bounce buffer
constexpr size_t kOutBytesPerSlot = 8 + 8 + 24 + 32 + 32 + 4 + 4 + 1;   // uv_l uv_r xyz desc_l desc_r dist idx status
constexpr int kStages = 5;
const char* const kStageNames[kStages] = {"harris_box", "boxsum_right", "select_corners", "describe_left", "stereo_match"};
constexpr int kStageDescribe = 3;   // present only on the batch path (LEFT descriptors ahead of the matcher)
constexpr int kRawFactor = 4;   // the Harris kernel's list (local maxima above the TILE threshold) vs max_candidates

std::string g_create_error;

struct Lane {
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    uint16_t* box_l = nullptr;   // S(y,x) of LEFT
    uint16_t* box_r = nullptr;   // S(y,x) of RIGHT
    uint16_t* box_ls = nullptr;  // planes stored shifted by one element, S(y,x+1): the odd-aligned TMA copies
    uint16_t* box_rs = nullptr;
    uint32_t* frame_max = nullptr;
    int* cand_count = nullptr;
    unsigned long long* cand = nullptr;
    ushort2* det_xy = nullptr;
    ushort2* kp_xy = nullptr;
    int* n_det = nullptr;
    int* n_kp = nullptr;
    uint32_t* g_head = nullptr;
    uint32_t* g_next = nullptr;
    uint8_t* g_state = nullptr;
    // staging for the host-buffer entry points
    uint8_t* img_l = nullptr;
    uint8_t* img_r = nullptr;
    uint8_t* mask = nullptr;
    // raw images while rectification is set (svi_set_rectification): rectify_kernel reads these and writes img_l / img_r
    uint8_t* raw_l = nullptr;
    uint8_t* raw_r = nullptr;
    CUtensorMap map_l{}, map_r{}, map_ls{}, map_rs{};  // TMA views of the four planes: (W, chunk*H) u16, row pitch box_pitch
    CUtensorMap map_l_patch{};                          // LEFT plane again, box = the 56 x 49 patch of one descriptor
    // binned matcher (binned.cuh): key-points sorted by image bin, one tile of the planes per bin
    int* bin_start = nullptr;          // [chunk][n_bins + 1]
    uint32_t* bin_slot = nullptr;      // [chunk][max_corners]
    ushort2* bin_kp = nullptr;         // [chunk][max_corners]
    CUtensorMap map_l_bin{}, map_r_bin{}, map_rs_bin{};
    StereoOutDev out{};
    // sparse frames (svi_stereo_frames_sparse): allocated at the first such call, [chunk][max_corners] lists padded by
    // BM_ALIGN elements (band_match_kernel's copies round the streamed range out to 16-byte addresses)
    ushort2* sp_kp_r = nullptr;        // RIGHT key-points after BRIEF's border filter, detector order
    int* sp_n_kp_r = nullptr;          // [chunk]: their count (host path; the device path writes the caller's array)
    int* sp_n_det_r = nullptr;         // [chunk]
    int* sp_row_l = nullptr;           // [chunk][H + 1]: row CSR of the LEFT key-points
    uint32_t* sp_slot_l = nullptr;     // LEFT key-points sorted by row: their slot ...
    ushort2* sp_kp_l = nullptr;        // ... and coordinates
    int* sp_row_r = nullptr;           // the same for RIGHT
    uint32_t* sp_slot_r = nullptr;
    ushort2* sp_kp_rs = nullptr;
    uint8_t* sp_desc_r = nullptr;      // RIGHT descriptors in row order
    int* sp_second = nullptr;          // second-smallest distance per LEFT slot (host path)
    // the left-right check (svi_sparse_band.mutual): allocated at the first call that asks for it
    uint8_t* sp_desc_lr = nullptr;     // LEFT descriptors in row order (the reverse pass's trains)
    unsigned long long* sp_rev = nullptr;   // [chunk][max_corners]: per RIGHT key-point, (distance << 32 | best LEFT slot) or ~0
    CUtensorMap map_r_patch{};         // RIGHT plane, box = the 56 x 49 patch of one descriptor
    std::vector<cudaEvent_t> ev;  // stage boundary events (profiling)
    size_t ev_used = 0;
    std::vector<uint8_t> ev_pre;  // per profiled chunk: did describe_left_kernel run between its two events?
};

}  // namespace

struct svi_ctx {
    int device = 0;
    svi_camera cam_l{}, cam_r{};
    svi_params p{};
    int W = 0, H = 0;
    int dev_pitch = 0;   // bytes per row of the staged images
    int resp_pitch = 0, box_pitch = 0;
    int chunk = 0, n_lanes = 0;
    int cand_cap = 0, raw_cap = 0;
    float* resp_one = nullptr;   // svi_harris_response only: one W x H plane
    int n_sms = 0;               // read at the first sparse call with the left-right check
    bool select_smem = true;
    int match_split = 0;     // warps per key-point in the scan-line matcher: 0 = chosen per launch; SVI_MATCH_SPLIT = 1 | 2 forces one
    bool trace = false;      // SVI_TRACE: host-side phase times of the tracking call on stderr (diagnostics)
    bool match_pre = true;   // LEFT descriptors by describe_left_kernel ahead of the matcher (SVI_MATCH_PRE = 0 | 1)
    bool match_binned = true;  // batch path: key-points binned by position, one TMA tile per bin (SVI_MATCH_BINNED = 0 | 1 | 2: off, by density, forced)
    int nbx = 0, n_bins = 0;
    SelectParams sel{};
    TriConst tc{};
    float f1 = 0, f0 = 0;
    Lane lanes[kMaxLanes];
    // candidate-list overflow flag: one int of mapped page-locked host memory.  Kernels write it in place (only when a
    // list overflows), the host reads it after the synchronisation it does anyway -- no copy, no extra round trip per call
    int* d_overflow = nullptr;            // device view
    volatile int* h_overflow = nullptr;   // host view
    cudaEvent_t fork = nullptr;
    // latency path (one pair per call): the RIGHT image travels and gets its box sums on a second stream while the
    // detector runs on LEFT; `side_done` joins it back before the first kernel that needs both
    cudaStream_t side = nullptr;
    cudaEvent_t side_done = nullptr;
    // tracking: both images of the current pair as two planes of one buffer, and the scratch of the
    // window-mode detector of stage 2 (grown on demand)
    uint8_t* trk_img = nullptr;
    struct RoiScratch {
        int items = 0;
        uint32_t* max = nullptr;
        int* cand_count = nullptr;
        unsigned long long* cand = nullptr;
        ushort2* det = nullptr;
        ushort2* kp = nullptr;
        int* n_det = nullptr;
        int* n_kp = nullptr;
        RoiItem* rois = nullptr;
        Stage2Item* s2 = nullptr;
        int* defer = nullptr;   // windows that do not fit the small selection configuration
        int* counters = nullptr;  // device-side item counts: stage 2 LEFT, stage 2 RIGHT, stage 3
    } roi;
    Stage3Item* s3_items = nullptr;
    // pinned bounce buffer of the small-call path (one or a few frames per call: the tracker's per-frame use)
    unsigned char* pin = nullptr;
    size_t pin_bytes = 0;
    // ... and its device-side result block: every output array of up to kSmallFrames frames in ONE allocation, so that the
    // results of a single-pair call come back with one copy
    unsigned char* small_block = nullptr;
    size_t small_bytes = 0;
    StereoOutDev small_out{};
    int* small_n_kp = nullptr;
    int* small_n_det = nullptr;
    int n_sm = 148;
    // the call buffer (DESIGN.md section 3): the per-call arrays of the per-query, tracking and solver entry points, one
    // device block + its pinned mirror of the same size, grown by reserve_call
    unsigned char* call_dev = nullptr;
    unsigned char* call_pin = nullptr;
    size_t call_bytes = 0;
    bool profiling = false;
    bool serial = false;   // profiling mode 2: every chunk on lane 0, so that the stage events bracket ONE kernel each
    // rectification (svi_set_rectification): both cameras' maps in one device block, [camera][xy short2 | frac uint16]
    // with rect_npad (W * H rounded up to 4) entries each; off = all null, no launch, copy or allocation anywhere
    bool rect = false;
    unsigned char* rect_map = nullptr;
    int rect_npad = 0;
    double stage_ms[kStages] = {};
    long stage_launches[kStages] = {};
    std::string err;
};

namespace {

int fail(svi_ctx* c, int code, const std::string& msg) {
    if (c) c->err = msg; else g_create_error = msg;
    return code;
}

#define CK(call)                                                                                  \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess)                                                                    \
            return fail(ctx, SVI_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));   \
    } while (0)

inline int align_up(int v, int a) { return (v + a - 1) / a * a; }

// grid of the Harris kernel: response tiles HT_SX x HT_SY apart, the tile interiors cover columns 1..W-2, rows 1..H-2
inline dim3 harris_grid(int W, int H, int layers) {
    return dim3((unsigned)std::max(1, (W - 2 + HT_SX - 1) / HT_SX), (unsigned)std::max(1, (H - 2 + HT_SY - 1) / HT_SY), (unsigned)layers);
}

FrameGeom make_geom(const svi_ctx* c, int img_pitch, size_t img_stride) {
    FrameGeom g;
    g.W = c->W; g.H = c->H;
    g.img_pitch = img_pitch;
    g.img_stride = img_stride;
    g.resp_pitch = c->resp_pitch;
    g.box_pitch = c->box_pitch;
    return g;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point lookup (no libcuda link needed).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

bool make_box_map(CUtensorMap* m, uint16_t* base, int W, int rows, int box_pitch, std::string* err, int box_w = PATCH_W,
                  int box_h = PATCH_ROWS) {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || !p ||
            q != cudaDriverEntryPointSuccess) {
            *err = "cuTensorMapEncodeTiled is not available from this driver";
            return false;
        }
        fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    const cuuint64_t gdim[2] = {(cuuint64_t)W, (cuuint64_t)rows};
    const cuuint64_t gstride[1] = {(cuuint64_t)box_pitch * sizeof(uint16_t)};
    const cuuint32_t box[2] = {(cuuint32_t)box_w, (cuuint32_t)box_h};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_UINT16, 2, base, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        *err = "cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r);
        return false;
    }
    return true;
}

// Stage-boundary events come from a per-lane pool that svi_set_profiling fills ahead of time (kEventPool events per
// lane), so that no event is created inside a timed region; the pool still grows if a step needs more.
constexpr size_t kEventPool = 1024;
void reserve_events(Lane& l, size_t count) {
    while (l.ev.size() < count) {
        cudaEvent_t e;
        if (cudaEventCreate(&e) != cudaSuccess) break;
        l.ev.push_back(e);
    }
}
cudaEvent_t lane_event(Lane& l) {
    if (l.ev_used == l.ev.size()) reserve_events(l, l.ev.size() + 64);
    return l.ev[l.ev_used++];
}

void mark(svi_ctx* c, Lane& l) {
    if (c->profiling) cudaEventRecord(lane_event(l), l.stream);
}

// Fold the recorded stage events into per-stage totals (call after the lanes are idle).
void collect_timings(svi_ctx* c) {
    for (int li = 0; li < c->n_lanes; ++li) {
        Lane& l = c->lanes[li];
        for (size_t i = 0, rec = 0; i + kStages < l.ev_used; i += kStages + 1, ++rec) {
            for (int s = 0; s < kStages; ++s) {
                if (s == kStageDescribe && !(rec < l.ev_pre.size() && l.ev_pre[rec])) continue;   // no kernel in that bracket
                float ms = 0.f;
                if (cudaEventElapsedTime(&ms, l.ev[i + s], l.ev[i + s + 1]) == cudaSuccess) {
                    c->stage_ms[s] += ms;
                    c->stage_launches[s] += 1;
                }
            }
        }
        l.ev_used = 0;
        l.ev_pre.clear();
    }
}

// Descriptor + match stages of the batch path, binned form (binned.cuh): sort the key-points into bins, LEFT descriptors
// per bin, scan-line searches per bin.
template <class G>
int run_binned(svi_ctx* ctx, Lane& l, const FrameGeom& g, int nf, const StereoOutDev& out, int out_frame0, const int* n_kp) {
    cudaStream_t s = l.stream;
    const dim3 bgrid(ctx->n_bins, nf);
    bin_keypoints_kernel<<<nf, BINK_THREADS, sizeof(uint32_t) * ctx->n_bins, s>>>(l.kp_xy, n_kp, ctx->p.max_corners, G::BIN_W, G::BIN_H, ctx->nbx,
                                                                                 ctx->n_bins, l.bin_start, l.bin_slot, l.bin_kp);
    describe_left_binned_kernel<G><<<bgrid, G::D_WARPS * 32, G::D_SMEM, s>>>(l.map_l_bin, g, l.bin_start, l.bin_slot, l.bin_kp, ctx->nbx, ctx->n_bins,
                                                                            ctx->p.max_corners, out.desc_l, out.cap, out_frame0);
    if (ctx->profiling) l.ev_pre.push_back(1);
    mark(ctx, l);
    stereo_match_binned_kernel<G><<<bgrid, G::M_WARPS * 32, G::M_SMEM, s>>>(l.map_r_bin, l.map_rs_bin, g, ctx->tc, ctx->p.keypoint_size,
                                                                           ctx->p.search_range_px, l.bin_start, l.bin_slot, l.bin_kp, ctx->nbx,
                                                                           ctx->n_bins, ctx->p.max_corners, out, out_frame0, ctx->d_overflow);
    mark(ctx, l);
    return SVI_SUCCESS;
}

template <class G>
int setup_binned(svi_ctx* ctx, Lane& l, size_t rows, std::string* err) {
    if (!make_box_map(&l.map_l_bin, l.box_l, ctx->W, (int)rows, ctx->box_pitch, err, G::D_COLS, G::ROWS) ||
        !make_box_map(&l.map_r_bin, l.box_r, ctx->W, (int)rows, ctx->box_pitch, err, G::COLS, G::ROWS) ||
        !make_box_map(&l.map_rs_bin, l.box_rs, ctx->W, (int)rows, ctx->box_pitch, err, G::COLS, G::ROWS))
        return SVI_ERR_CUDA;
    return SVI_SUCCESS;
}

// The detector on nf frames of one image: candidate lists in the lane's scratch (zeroed by the caller), and the image's box-sum
// plane `box` (harris_box writes it from its own tile; in FAST mode boxsum9, without the shifted copy).  With the selection
// below, the detection of the dense path (LEFT) and of both sides of the sparse path.
void launch_detector(svi_ctx* ctx, Lane& l, const uint8_t* d_img, const uint8_t* d_mask, const FrameGeom& g, int nf, uint16_t* box) {
    cudaStream_t s = l.stream;
    const dim3 tiles((g.W + HT_W - 1) / HT_W, (g.H + HT_H - 1) / HT_H, nf);
    if (ctx->p.detector == SVI_DETECTOR_FAST_9_16) {
        fast_candidates_kernel<<<tiles, HT_THREADS, 0, s>>>(d_img, d_mask, g, ctx->p.fast_threshold, ctx->p.fast_nonmax, l.cand,
                                                            l.cand_count, ctx->raw_cap);
        boxsum9_kernel<<<tiles, HT_THREADS, 0, s>>>(d_img, g, box, nullptr);
    } else {
        harris_box_kernel<<<harris_grid(g.W, g.H, nf), HT_THREADS, sizeof(HarrisSmem), s>>>(
            d_img, d_mask, g, ctx->f1, ctx->f0, ctx->p.harris_k, ctx->p.quality_level, nullptr, box, nullptr, l.frame_max, l.cand,
            l.cand_count, ctx->raw_cap, nullptr, nullptr, g.H);
    }
}

// Corner selection from the lane's candidate lists: the selected corners (det_xy / n_det) and the ones that survive BRIEF's
// border filter (kp_xy / n_kp), [nf][max_corners].
void launch_select(svi_ctx* ctx, Lane& l, int nf, ushort2* det_xy, int* n_det, ushort2* kp_xy, int* n_kp) {
    cudaStream_t s = l.stream;
    const uint32_t* fmax = ctx->p.detector == SVI_DETECTOR_FAST_9_16 ? nullptr : l.frame_max;
    if (ctx->select_smem) {
        select_corners_kernel<true><<<nf, SEL_THREADS, 13 * SEL_SMEM_KEYS, s>>>(
            l.cand, l.cand_count, fmax, ctx->sel, nullptr, nullptr, nullptr, det_xy, n_det, kp_xy, n_kp, ctx->d_overflow, nullptr);
    } else {
        select_corners_kernel<false><<<nf, SEL_THREADS, 4 * SEL_SMEM_CELLS, s>>>(
            l.cand, l.cand_count, fmax, ctx->sel, l.g_head, l.g_next, l.g_state, det_xy, n_det, kp_xy, n_kp, ctx->d_overflow, nullptr);
    }
}

// The kernels of the new-landmark path for `nf` frames on one lane: detector, RIGHT box sums, corner selection, then the
// descriptor / match stages in the form that fits the call (svi_kernels_per_chunk: 4 to 6 launches).
int run_pipeline(svi_ctx* ctx, Lane& l, const uint8_t* d_left, const uint8_t* d_right, const uint8_t* d_mask,
                 const FrameGeom& g, int nf, const StereoOutDev& out, int out_frame0, int* n_kp, int* n_det,
                 cudaStream_t side = nullptr, const std::function<int(cudaStream_t)>* upload_right = nullptr) {
    cudaStream_t s = l.stream;
    CK(cudaMemsetAsync(l.frame_max, 0, sizeof(uint32_t) * nf, s));
    CK(cudaMemsetAsync(l.cand_count, 0, sizeof(int) * nf, s));
    const dim3 tiles((g.W + HT_W - 1) / HT_W, (g.H + HT_H - 1) / HT_H, nf);
    mark(ctx, l);
    launch_detector(ctx, l, d_left, d_mask, g, nf, l.box_l);
    mark(ctx, l);
    // `side` (latency path): the RIGHT plane goes up on that stream -- staged by the caller's hook only now, so that the
    // host-side copy into the pinned mirror overlaps the detector -- and its box sums run there too
    if (upload_right) {
        const int rc = (*upload_right)(side ? side : s);
        if (rc != SVI_SUCCESS) return rc;
    }
    boxsum9_kernel<<<tiles, HT_THREADS, 0, side ? side : s>>>(d_right, g, l.box_r, l.box_rs);
    if (side) {
        CK(cudaEventRecord(ctx->side_done, side));
        CK(cudaStreamWaitEvent(s, ctx->side_done, 0));   // the selection kernel below does not need it, the matcher does;
                                                          // one wait here keeps the stage events of the profiler in order
    }
    mark(ctx, l);
    launch_select(ctx, l, nf, l.det_xy, n_det, l.kp_xy, n_kp);
    mark(ctx, l);
    // full batches amortise a warp's set-up over MATCH_KP_PER_WARP key-points; a small call (one pair per frame in a
    // tracker) would leave most SMs idle that way, so it spreads the key-points until two waves of warps exist
    const long long slots = (long long)nf * ctx->p.max_corners;
    const int kp_per_warp = (int)std::max<long long>(1, std::min<long long>(MATCH_KP_PER_WARP, slots / (2LL * ctx->n_sm * 9)));
    const int kp_per_cta = MATCH_WARPS * kp_per_warp;
    const dim3 mgrid((ctx->p.max_corners + kp_per_cta - 1) / kp_per_cta, nf);
    // full batches: the LEFT descriptors first (one TMA patch per key-point), then the matcher with match_split warps per
    // key-point; small calls keep the single fused kernel (one launch less on the latency path)
    const bool pre = ctx->match_pre && kp_per_warp == MATCH_KP_PER_WARP;
    // warps per key-point: measured (DESIGN.md section 6) -- two warps win whenever the LEFT gathers stay in the matcher
    // (small calls) and on multi-pass searches (scan lines longer than one window), one warp wins on the batch path
    const int split = ctx->match_split ? ctx->match_split : ((pre && ctx->p.search_range_px <= (float)PATCH_CHUNK) ? 1 : 2);
    // batch path with the reference's geometry (scan line of one pass, whole-pixel ROI border): key-points binned by
    // position, one shared tile per bin (binned.cuh)
    if (pre && ctx->match_binned && l.bin_start) {
        const int rc = run_binned<BinWide>(ctx, l, g, nf, out, out_frame0, n_kp);
        CK(cudaGetLastError());
        return rc;
    }
    if (pre) {
        const dim3 dgrid((ctx->p.max_corners + DL_WARPS * DL_KP_PER_WARP - 1) / (DL_WARPS * DL_KP_PER_WARP), nf);
        describe_left_kernel<<<dgrid, DL_WARPS * 32, DL_SMEM, s>>>(l.map_l_patch, g, l.kp_xy, n_kp, ctx->p.max_corners, out.desc_l, out.cap,
                                                                   out_frame0);
    }
    if (ctx->profiling) l.ev_pre.push_back(pre ? 1 : 0);
    mark(ctx, l);
#define SVI_MATCH_ARGS l.box_l, l.map_r, l.map_rs, g, ctx->tc, ctx->p.keypoint_size, ctx->p.search_range_px, l.kp_xy, n_kp, \
                       ctx->p.max_corners, out, out_frame0, kp_per_warp
    if (pre && split == 1)
        stereo_match_split_kernel<1, true><<<mgrid, MatchSplit<1>::THREADS, MatchSplit<1>::SMEM, s>>>(SVI_MATCH_ARGS);
    else if (pre && split == 2)
        stereo_match_split_kernel<2, true><<<mgrid, MatchSplit<2>::THREADS, MatchSplit<2>::SMEM, s>>>(SVI_MATCH_ARGS);
    else if (split == 2)
        stereo_match_split_kernel<2, false><<<mgrid, MatchSplit<2>::THREADS, MatchSplit<2>::SMEM, s>>>(SVI_MATCH_ARGS);
    else
        stereo_match_kernel<<<mgrid, MATCH_WARPS * 32, MATCH_SMEM, s>>>(SVI_MATCH_ARGS);
#undef SVI_MATCH_ARGS
    mark(ctx, l);
    CK(cudaGetLastError());
    return SVI_SUCCESS;
}

int check_overflow(svi_ctx* ctx) {
#ifdef SVI_BOUNDS_CHECK
    {
        int line = 0;
        CK(cudaMemcpyFromSymbol(&line, g_svi_check, sizeof(int)));
        if (line) return fail(ctx, SVI_ERR_CUDA, "bounds check failed in a kernel: tag/line " + std::to_string(line));
    }
#endif
    const int h = *ctx->h_overflow;   // every caller has synchronised the streams that could have written it
    if (h) *ctx->h_overflow = 0;
    if (h == 4) return fail(ctx, SVI_ERR_CUDA, "internal error: a search window left its tile in the binned matcher (SVI_MATCH_BINNED=0 selects the per-key-point kernels)");
    if (h == 3) {
        return fail(ctx, SVI_ERR_CAPACITY, "FAST found more corners than svi_params.max_corners in a frame (cv::FAST returns all of them): raise max_corners");
    }
    if (h) {
        return fail(ctx, SVI_ERR_CAPACITY,
                    "NMS candidate list overflow: raise svi_params.max_candidates (a frame produced more than " +
                        std::to_string(ctx->cand_cap) + " candidates)");
    }
    return SVI_SUCCESS;
}

int sync_lanes(svi_ctx* ctx) {
    for (int i = 0; i < ctx->n_lanes; ++i) CK(cudaStreamSynchronize(ctx->lanes[i].stream));
    if (ctx->profiling) collect_timings(ctx);
    return SVI_SUCCESS;
}

template <typename T>
cudaError_t dmalloc(T** p, size_t count) { return cudaMalloc(reinterpret_cast<void**>(p), count * sizeof(T)); }

// ---- sparse frames (svi_stereo_frames_sparse): per-lane scratch, allocated at the first sparse call; a ctx that never makes
// one allocates nothing for it.
int ensure_sparse_scratch(svi_ctx* ctx) {
    // bin_keypoints_kernel sorts by row with one counter per row in shared memory
    const int row_smem = (int)sizeof(uint32_t) * ctx->H;
    if (row_smem > 200 * 1024) return fail(ctx, SVI_ERR_UNSUPPORTED, "svi_stereo_frames_sparse: image height above 51200 rows");
    if (ctx->lanes[ctx->n_lanes - 1].sp_kp_r) return SVI_SUCCESS;
    CK(cudaFuncSetAttribute(bin_keypoints_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, std::max(row_smem, 48 * 1024)));
    const size_t C = (size_t)ctx->chunk, MC = (size_t)ctx->p.max_corners, L = C * MC + BM_ALIGN, rows = C * ((size_t)ctx->H + 1);
    for (int i = 0; i < ctx->n_lanes; ++i) {
        Lane& l = ctx->lanes[i];
        if (l.sp_kp_r) continue;
        CK(dmalloc(&l.sp_n_kp_r, C));
        CK(dmalloc(&l.sp_n_det_r, C));
        CK(dmalloc(&l.sp_row_l, rows));
        CK(dmalloc(&l.sp_slot_l, L));
        CK(dmalloc(&l.sp_kp_l, L));
        CK(dmalloc(&l.sp_row_r, rows));
        CK(dmalloc(&l.sp_slot_r, L));
        CK(dmalloc(&l.sp_kp_rs, L));
        CK(dmalloc(&l.sp_desc_r, 32 * L));
        CK(dmalloc(&l.sp_second, L));
        std::string merr;
        if (!make_box_map(&l.map_r_patch, l.box_r, ctx->W, (int)(C * ctx->H), ctx->box_pitch, &merr, DL_COLS)) return fail(ctx, SVI_ERR_CUDA, merr);
        CK(dmalloc(&l.sp_kp_r, L));   // last: marks the lane's scratch complete
    }
    return SVI_SUCCESS;
}

// The left-right check's scratch (40 B per key-point and chunk frame): allocated at the first call with mutual = 1.
int ensure_mutual_scratch(svi_ctx* ctx) {
    if (!ctx->n_sms) CK(cudaDeviceGetAttribute(&ctx->n_sms, cudaDevAttrMultiProcessorCount, ctx->device));
    const size_t C = (size_t)ctx->chunk, MC = (size_t)ctx->p.max_corners, L = C * MC + BM_ALIGN;
    for (int i = 0; i < ctx->n_lanes; ++i) {
        Lane& l = ctx->lanes[i];
        if (l.sp_rev) continue;
        CK(dmalloc(&l.sp_desc_lr, 32 * L));
        CK(dmalloc(&l.sp_rev, C * MC));   // last: marks the lane's scratch complete
    }
    return SVI_SUCCESS;
}

// The sparse frame of nf frames on one lane: detection and selection on LEFT (with the masks) and on RIGHT (without) -- the
// same launches as the dense path's, RIGHT after LEFT's selection so that the candidate lists are reused --, both key-point
// lists sorted by row (bin_keypoints_kernel with full-width bins one row high: a row CSR plus each key-point's slot), LEFT
// descriptors into out.desc_l as on the dense path, RIGHT descriptors over the row-sorted list, then band_match_kernel.  With
// the left-right check, the LEFT descriptors are first gathered into row order and the reverse pass (RIGHT queries, LEFT
// trains, mirrored bounds) writes each RIGHT key-point's best LEFT slot, which the forward pass's finish compares.
// second / n_kp_r: the call's second-distance slots (indexed like out) and RIGHT key-point counts (indexed by chunk frame).
int run_sparse(svi_ctx* ctx, Lane& l, const uint8_t* d_left, const uint8_t* d_right, const uint8_t* d_mask, const FrameGeom& g, int nf,
               const StereoOutDev& out, int out_frame0, int* n_kp, int* n_det, int* second, int* n_kp_r, const svi_sparse_band& band) {
    cudaStream_t s = l.stream;
    const int MC = ctx->p.max_corners, H = ctx->H;
    const struct { const uint8_t* img; const uint8_t* mask; uint16_t* box; int* n_det; ushort2* kp; int* n_kp; } sides[2] = {
        {d_left, d_mask, l.box_l, n_det, l.kp_xy, n_kp}, {d_right, nullptr, l.box_r, l.sp_n_det_r, l.sp_kp_r, n_kp_r}};
    for (const auto& sd : sides) {
        CK(cudaMemsetAsync(l.frame_max, 0, sizeof(uint32_t) * nf, s));
        CK(cudaMemsetAsync(l.cand_count, 0, sizeof(int) * nf, s));
        launch_detector(ctx, l, sd.img, sd.mask, g, nf, sd.box);
        launch_select(ctx, l, nf, l.det_xy, sd.n_det, sd.kp, sd.n_kp);   // LEFT's det_xy is not needed once it is selected
    }
    const size_t row_smem = sizeof(uint32_t) * H;
    bin_keypoints_kernel<<<nf, BINK_THREADS, row_smem, s>>>(l.kp_xy, n_kp, MC, ctx->W, 1, 1, H, l.sp_row_l, l.sp_slot_l, l.sp_kp_l);
    bin_keypoints_kernel<<<nf, BINK_THREADS, row_smem, s>>>(l.sp_kp_r, n_kp_r, MC, ctx->W, 1, 1, H, l.sp_row_r, l.sp_slot_r, l.sp_kp_rs);
    const dim3 dgrid((MC + DL_WARPS * DL_KP_PER_WARP - 1) / (DL_WARPS * DL_KP_PER_WARP), nf);
    describe_left_kernel<<<dgrid, DL_WARPS * 32, DL_SMEM, s>>>(l.map_l_patch, g, l.kp_xy, n_kp, MC, out.desc_l, out.cap, out_frame0);
    describe_left_kernel<<<dgrid, DL_WARPS * 32, DL_SMEM, s>>>(l.map_r_patch, g, l.sp_kp_rs, n_kp_r, MC, l.sp_desc_r, MC, 0);
    BandArgs a{};
    a.band_v = band.band_v; a.min_disp = band.min_disparity; a.max_disp = band.max_disparity;
    a.q_kp = l.sp_kp_l; a.q_slot = l.sp_slot_l; a.n_q = n_kp;
    a.t_kp = l.sp_kp_rs; a.t_slot = l.sp_slot_r; a.t_desc = l.sp_desc_r; a.t_row = l.sp_row_r;
    a.H = H; a.max_corners = MC;
    a.out = out; a.out_frame0 = out_frame0; a.tc = ctx->tc; a.second = second;
    const dim3 bgrid((MC + BM_THREADS - 1) / BM_THREADS, nf);
    if (band.mutual) {
        gather_rows_kernel<<<dim3((2 * MC + GR_THREADS - 1) / GR_THREADS, nf), GR_THREADS, 0, s>>>(out.desc_l, out.cap, out_frame0,
                                                                                                  l.sp_slot_l, n_kp, MC, l.sp_desc_lr);
        // splits of each RIGHT query block's LEFT range: about four CTAs per SM if every query block were full
        const int blocks = (int)bgrid.x * nf, splits = std::min(8, std::max(1, (4 * ctx->n_sms + blocks - 1) / blocks));
        CK(cudaMemsetAsync(l.sp_rev, 0xFF, sizeof(unsigned long long) * nf * MC, s));
        BandArgs r{};
        r.band_v = band.band_v; r.min_disp = -band.max_disparity; r.max_disp = -band.min_disparity;
        r.q_kp = l.sp_kp_rs; r.q_slot = l.sp_slot_r; r.n_q = n_kp_r; r.q_desc = l.sp_desc_r;
        r.t_kp = l.sp_kp_l; r.t_slot = l.sp_slot_l; r.t_desc = l.sp_desc_lr; r.t_row = l.sp_row_l;
        r.H = H; r.max_corners = MC; r.rev = l.sp_rev;
        band_match_kernel<BM_REVERSE><<<dim3(bgrid.x, nf, splits), BM_THREADS, BandTile<true>::SMEM, s>>>(r);
        a.mutual = 1; a.rev = l.sp_rev; a.n_t = n_kp_r;
    }
    band_match_kernel<BM_FRAME><<<bgrid, BM_THREADS, BandTile<true>::SMEM, s>>>(a);
    CK(cudaGetLastError());
    return SVI_SUCCESS;
}

// ---- rectification
// cvRound of OpenCV's x86 build (cvtsd2si / cvtss2si): half to even, and INT_MIN for NaN or anything outside int
int cv_round_host(double v) {
    if (!(v >= -2147483648.0 && v < 2147483648.0)) return INT32_MIN;
    return (int)std::nearbyint(v);
}
int16_t saturate_short(int v) { return (int16_t)std::min(32767, std::max(-32768, v)); }

// The numbers of Matx33d::determinant / Matx33d::inv (the cofactor form OpenCV uses for 3 x 3).
double det33(const double* a) {
    return a[0] * (a[4] * a[8] - a[7] * a[5]) - a[1] * (a[3] * a[8] - a[6] * a[5]) + a[2] * (a[3] * a[7] - a[6] * a[4]);
}

// cv::initUndistortRectifyMap(K, D, R, P, (W, H), CV_16SC2) -- or, with float_maps, CV_32FC1 followed by the conversion
// cv::remap applies to float maps (cv::convertMaps to CV_16SC2) -- in OpenCV's scalar operation order, fp64 without
// contraction (the library is built with -ffp-contract=off).  Empty string on success.
std::string rectify_map_host(const svi_camera* cam, const svi_rectification* r, int16_t* xy, uint16_t* frac) {
    if (!cam || !r || !xy || !frac) return "svi_rectify_map: null argument";
    if (cam->width == 0 || cam->height == 0 || cam->width > 65535 || cam->height > 65535) return "svi_rectify_map: bad image size";
    if (r->float_maps != 0 && r->float_maps != 1) return "svi_rectify_map: float_maps must be 0 or 1";
    const double dk = det33(r->K);
    if (!(dk != 0.0) || !std::isfinite(dk)) return "svi_rectify_map: matIntrinsic K is singular";
    double a[9];   // P[:3,:3] * R, Matx product order
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            double acc = 0.0;
            for (int k = 0; k < 3; ++k) acc += cam->P[i * 4 + k] * r->R[k * 3 + j];
            a[i * 3 + j] = acc;
        }
    double d = det33(a);
    if (!(d != 0.0) || !std::isfinite(d)) return "svi_rectify_map: P[:3,:3] * matRectification is singular";
    d = 1.0 / d;
    const double ir[9] = {(a[4] * a[8] - a[5] * a[7]) * d, (a[2] * a[7] - a[1] * a[8]) * d, (a[1] * a[5] - a[2] * a[4]) * d,
                          (a[5] * a[6] - a[3] * a[8]) * d, (a[0] * a[8] - a[2] * a[6]) * d, (a[2] * a[3] - a[0] * a[5]) * d,
                          (a[3] * a[7] - a[4] * a[6]) * d, (a[1] * a[6] - a[0] * a[7]) * d, (a[0] * a[4] - a[1] * a[3]) * d};
    const double u0 = r->K[2], v0 = r->K[5], fx = r->K[0], fy = r->K[4];
    const double k1 = r->D[0], k2 = r->D[1], p1 = r->D[2], p2 = r->D[3], k3 = 0.0, k4 = 0.0, k5 = 0.0, k6 = 0.0;
    const double s1 = 0.0, s2 = 0.0, s3 = 0.0, s4 = 0.0;
    const int W = (int)cam->width, H = (int)cam->height;
    for (int i = 0; i < H; ++i) {
        double _x = i * ir[1] + ir[2], _y = i * ir[4] + ir[5], _w = i * ir[7] + ir[8];
        for (int j = 0; j < W; ++j, _x += ir[0], _y += ir[3], _w += ir[6]) {
            const double w = 1. / _w, x = _x * w, y = _y * w;
            const double x2 = x * x, y2 = y * y;
            const double r2 = x2 + y2, _2xy = 2 * x * y;
            const double kr = (1 + ((k3 * r2 + k2) * r2 + k1) * r2) / (1 + ((k6 * r2 + k5) * r2 + k4) * r2);
            const double xd = (x * kr + p1 * _2xy + p2 * (r2 + 2 * x2) + s1 * r2 + s2 * r2 * r2);
            const double yd = (y * kr + p1 * (r2 + 2 * y2) + p2 * _2xy + s3 * r2 + s4 * r2 * r2);
            // the identity tilt matrix of the 4-coefficient model, applied as OpenCV applies it
            double t0 = 0.0, t1 = 0.0, t2 = 0.0;
            t0 += 1.0 * xd; t0 += 0.0 * yd; t0 += 0.0 * 1.0;
            t1 += 0.0 * xd; t1 += 1.0 * yd; t1 += 0.0 * 1.0;
            t2 += 0.0 * xd; t2 += 0.0 * yd; t2 += 1.0 * 1.0;
            const double inv_proj = t2 ? 1. / t2 : 1;
            const double u = fx * inv_proj * t0 + u0, v = fy * inv_proj * t1 + v0;
            int iu, iv;
            if (r->float_maps) {
                iu = cv_round_host((double)((float)u * 32.f));
                iv = cv_round_host((double)((float)v * 32.f));
            } else {
                iu = cv_round_host(u * 32.0);
                iv = cv_round_host(v * 32.0);
            }
            const size_t o = (size_t)i * W + j;
            xy[2 * o] = saturate_short(iu >> 5);
            xy[2 * o + 1] = saturate_short(iv >> 5);
            frac[o] = (uint16_t)((iv & 31) * 32 + (iu & 31));
        }
    }
    return std::string();
}

const short2* rect_xy(const svi_ctx* c, int cam) { return reinterpret_cast<const short2*>(c->rect_map + (size_t)cam * c->rect_npad * 6); }
const uint16_t* rect_frac(const svi_ctx* c, int cam) {
    return reinterpret_cast<const uint16_t*>(c->rect_map + (size_t)cam * c->rect_npad * 6 + (size_t)c->rect_npad * 4);
}

// One rectify_kernel launch for n_cams images of nf frames each: raw src[i] (src_pitch bytes per row, src_stride per
// frame) through the map of camera cams[i] into the dense plane stack dst[i] (W bytes per row, H * W per frame).
int launch_rectify(svi_ctx* ctx, int n_cams, const int* cams, const uint8_t* const* src, uint8_t* const* dst, size_t src_pitch,
                   size_t src_stride, int nf, cudaStream_t s) {
    RectifyArgs a{};
    for (int i = 0; i < n_cams; ++i) a.cam[i] = RectifySide{rect_xy(ctx, cams[i]), rect_frac(ctx, cams[i]), src[i], dst[i]};
    a.W = ctx->W; a.H = ctx->H; a.n_pix = ctx->W * ctx->H; a.n_pad = ctx->rect_npad; a.nf = nf;
    a.src_pitch = src_pitch; a.src_stride = src_stride; a.dst_stride = (size_t)ctx->H * ctx->dev_pitch;
    const int quads = (a.n_pix + RECT_PX - 1) / RECT_PX;
    rectify_kernel<<<dim3((quads + RECT_THREADS - 1) / RECT_THREADS, n_cams, (nf + RECT_FRAMES - 1) / RECT_FRAMES), RECT_THREADS, 0, s>>>(a);
    CK(cudaGetLastError());
    return SVI_SUCCESS;
}
int rectify_pair(svi_ctx* ctx, const uint8_t* left, const uint8_t* right, size_t pitch, size_t stride, uint8_t* d_left, uint8_t* d_right,
                 int nf, cudaStream_t s) {
    const int cams[2] = {0, 1};
    const uint8_t* src[2] = {left, right};
    uint8_t* dst[2] = {d_left, d_right};
    return launch_rectify(ctx, 2, cams, src, dst, pitch, stride, nf, s);
}
int rectify_one(svi_ctx* ctx, int cam, const uint8_t* raw, size_t pitch, size_t stride, uint8_t* d_out, int nf, cudaStream_t s) {
    return launch_rectify(ctx, 1, &cam, &raw, &d_out, pitch, stride, nf, s);
}

}  // namespace

// ---- per-query entry points: one image (or pair) staged in lane 0, queries in the call buffer ----
namespace {
// Page-locked caller memory (cudaMallocHost, cudaHostRegister, a pinned torch tensor: a camera driver's DMA buffers) is
// read by the copy engine directly; anything else goes through the library's pinned mirror, because a cudaMemcpyAsync
// from pageable memory is a blocking staged copy.  (One driver query per image, ~1 us; the mirror memcpy of a
// 1241 x 376 pair costs ~75 us of a 0.2 ms single-pair call.)
bool host_is_pinned(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

// One image of camera `cam` (0 = LEFT, 1 = RIGHT) into d_img plus its box sums.  While rectification is set the image is
// raw: it goes up into lane 0's raw plane of that camera and rectify_kernel writes d_img.
int stage_box(svi_ctx* ctx, const uint8_t* img, size_t pitch, uint8_t* d_img, uint16_t* d_box, uint16_t* d_box_shift,
              cudaStream_t s, int cam, int pin_plane = 0) {
    const FrameGeom g = make_geom(ctx, ctx->dev_pitch, (size_t)ctx->H * ctx->dev_pitch);
    const size_t plane = (size_t)ctx->H * ctx->dev_pitch;
    uint8_t* const d_rect = d_img;
    if (ctx->rect) d_img = cam ? ctx->lanes[0].raw_r : ctx->lanes[0].raw_l;
    if (host_is_pinned(img)) {
        if ((int)pitch == ctx->dev_pitch) CK(cudaMemcpyAsync(d_img, img, plane, cudaMemcpyHostToDevice, s));
        else CK(cudaMemcpy2DAsync(d_img, ctx->dev_pitch, img, pitch, ctx->W, ctx->H, cudaMemcpyHostToDevice, s));
    } else if (ctx->pin && pin_plane >= 0 && (size_t)(pin_plane + 1) * plane <= ctx->pin_bytes) {
        unsigned char* stage = ctx->pin + (size_t)pin_plane * plane;
        if ((int)pitch == ctx->dev_pitch) std::memcpy(stage, img, plane);
        else for (int y = 0; y < ctx->H; ++y) std::memcpy(stage + (size_t)y * ctx->dev_pitch, img + (size_t)y * pitch, ctx->W);
        CK(cudaMemcpyAsync(d_img, stage, plane, cudaMemcpyHostToDevice, s));
    } else {
        CK(cudaMemcpy2DAsync(d_img, ctx->dev_pitch, img, pitch, ctx->W, ctx->H, cudaMemcpyHostToDevice, s));
    }
    if (ctx->rect) {
        const int rc = rectify_one(ctx, cam, d_img, ctx->dev_pitch, plane, d_rect, 1, s);
        if (rc != SVI_SUCCESS) return rc;
    }
    const dim3 tiles((g.W + HT_W - 1) / HT_W, (g.H + HT_H - 1) / HT_H, 1);
    boxsum9_kernel<<<tiles, HT_THREADS, 0, s>>>(d_rect, g, d_box, d_box_shift);
    CK(cudaGetLastError());
    return SVI_SUCCESS;
}

// ---- the call buffer (DESIGN.md section 3).  Every user lays out [inputs | outputs | scratch] with CallLayout, makes
// room with reserve_call before it enqueues anything that touches the buffer, memcpys its inputs into the pinned mirror,
// sends them up with one copy (call_send), zeroes its outputs with one memset where it needs them zeroed, and brings them
// back with one copy and one synchronisation (call_fetch) before it memcpys them into the caller's arrays.  Pageable
// caller arrays therefore never turn a transfer into a blocking staged copy.
struct CallLayout {
    size_t end = 0;
    size_t take(size_t bytes) {   // 256-byte-aligned offset of the next `bytes`
        const size_t o = end;
        end = (end + bytes + 255) & ~size_t(255);
        return o;
    }
};

// The size svi_create gives the buffer before the cap; the match entry points still bound their inputs by it.
size_t query_bytes(const svi_ctx* c) {
    return (size_t)c->p.max_queries * 512 + (size_t)c->p.max_corners * 64 + 3 * (size_t)c->H * c->dev_pitch + (1 << 20);
}

// Grows the buffer to twice the need (a tracker's measurement lists get longer frame by frame).  Nothing is in flight on
// it: every user leaves lane 0 idle when it returns.
int reserve_call(svi_ctx* ctx, size_t bytes) {
    if (bytes <= ctx->call_bytes) return SVI_SUCCESS;
    if (ctx->call_dev) cudaFree(ctx->call_dev);
    if (ctx->call_pin) cudaFreeHost(ctx->call_pin);
    ctx->call_dev = nullptr; ctx->call_pin = nullptr; ctx->call_bytes = 0;
    const size_t want = std::max<size_t>(2 * bytes, 1u << 20);
    CK(cudaMalloc(reinterpret_cast<void**>(&ctx->call_dev), want));
    CK(cudaMallocHost(reinterpret_cast<void**>(&ctx->call_pin), want));
    ctx->call_bytes = want;
    return SVI_SUCCESS;
}

template <typename T = unsigned char>
T* dev_at(const svi_ctx* c, size_t o) { return reinterpret_cast<T*>(c->call_dev + o); }

void put(svi_ctx* c, size_t o, const void* h, size_t bytes) {   // a null host array stages nothing
    if (h) std::memcpy(c->call_pin + o, h, bytes);
}

int call_send(svi_ctx* ctx, size_t in_end, cudaStream_t s) {
    CK(cudaMemcpyAsync(ctx->call_dev, ctx->call_pin, in_end, cudaMemcpyHostToDevice, s));
    return SVI_SUCCESS;
}

int call_fetch(svi_ctx* ctx, size_t begin, size_t end, cudaStream_t s) {
    CK(cudaMemcpyAsync(ctx->call_pin + begin, ctx->call_dev + begin, end - begin, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return SVI_SUCCESS;
}

// Declared first in every user of the buffer: a call that fails part-way still leaves lane 0 idle, so that the next
// call may overwrite the mirror.  The successful path ends in a synchronisation of its own and sets `done`.
struct SyncOnFailure {
    cudaStream_t s;
    bool done = false;
    ~SyncOnFailure() { if (!done) cudaStreamSynchronize(s); }
};

// svi_landmarks of n landmarks, with or without the three stage-3 arrays
struct LandmarkLayout {
    bool stage3;
    size_t xyz, dl, dr, disp, size, uvref = 0, dref = 0, tdet = 0;
    LandmarkLayout(CallLayout& L, size_t n, bool with_stage3) : stage3(with_stage3) {
        xyz = L.take(24 * n); dl = L.take(32 * n); dr = L.take(32 * n); disp = L.take(4 * n); size = L.take(4 * n);
        if (stage3) { uvref = L.take(16 * n); dref = L.take(32 * n); tdet = L.take(128 * n); }
    }
    void put_all(svi_ctx* c, const svi_landmarks& lm, size_t n) const {
        put(c, xyz, lm.xyz_world, 24 * n); put(c, dl, lm.last_desc_left, 32 * n); put(c, dr, lm.last_desc_right, 32 * n);
        put(c, disp, lm.last_disparity, 4 * n); put(c, size, lm.keypoint_size, 4 * n);
        if (stage3) { put(c, uvref, lm.uv_reference_left, 16 * n); put(c, dref, lm.desc_reference_left, 32 * n); put(c, tdet, lm.T_left_to_world_at_detection, 128 * n); }
    }
    SvLandmarksDev sv(const svi_ctx* c) const {   // the stage-3 arrays are null without them
        return SvLandmarksDev{dev_at<double>(c, xyz), dev_at(c, dl), dev_at(c, dr), dev_at<float>(c, disp), dev_at<float>(c, size),
                              stage3 ? dev_at<double>(c, uvref) : nullptr, stage3 ? dev_at(c, dref) : nullptr, stage3 ? dev_at<double>(c, tdet) : nullptr};
    }
    LandmarksDev ld(const svi_ctx* c) const {
        const SvLandmarksDev s = sv(c);
        return LandmarksDev{s.xyz_w, s.desc_l, s.desc_r, s.disparity, s.size};
    }
    Stage3Extra ex(const svi_ctx* c) const {
        const SvLandmarksDev s = sv(c);
        return Stage3Extra{s.uv_ref, s.T_det};
    }
};

// The seven svi_track_result arrays of n landmarks, one contiguous range [status, end)
struct TrackLayout {
    size_t status, stage, uv_l, uv_r, xyz, desc_l, desc_r, end;
    TrackLayout(CallLayout& L, size_t n) {
        status = L.take(n); stage = L.take(n); uv_l = L.take(8 * n); uv_r = L.take(8 * n); xyz = L.take(24 * n);
        desc_l = L.take(32 * n); desc_r = L.take(32 * n); end = L.end;
    }
    TrackOutDev dev(const svi_ctx* c) const {
        return TrackOutDev{dev_at(c, status), dev_at(c, stage), dev_at<float>(c, uv_l), dev_at<float>(c, uv_r), dev_at<double>(c, xyz),
                           dev_at(c, desc_l), dev_at(c, desc_r)};
    }
    void copy_out(const svi_ctx* c, size_t n, const svi_track_result& r) const {   // from the mirror, after call_fetch
        const unsigned char* h = c->call_pin;
        std::memcpy(r.status, h + status, n);
        std::memcpy(r.stage, h + stage, n);
        std::memcpy(r.uv_left, h + uv_l, 8 * n);
        std::memcpy(r.uv_right, h + uv_r, 8 * n);
        std::memcpy(r.xyz_left, h + xyz, 24 * n);
        std::memcpy(r.desc_left, h + desc_l, 32 * n);
        std::memcpy(r.desc_right, h + desc_r, 32 * n);
    }
};

PositIn posit_in(const svi_ctx* ctx, const double* xyz, const float* uv_l, const float* uv_r, const double* T_estimate, const double* T_last,
                 const double* t_imu) {
    PositIn pi{};
    pi.xyz_world = xyz;
    pi.uv_left = uv_l;
    pi.uv_right = uv_r;
    std::memcpy(pi.P_left, ctx->cam_l.P, sizeof(pi.P_left));
    std::memcpy(pi.P_right, ctx->cam_r.P, sizeof(pi.P_right));
    std::memcpy(pi.T_estimate, T_estimate, sizeof(pi.T_estimate));
    std::memcpy(pi.T_last, T_last, sizeof(pi.T_last));
    std::memcpy(pi.t_imu, t_imu, sizeof(pi.t_imu));
    return pi;
}
void posit_result_from(const PositOut& po, svi_posit_result* r) {
    std::memcpy(r->T_world_to_left, po.T, sizeof(r->T_world_to_left));
    r->outcome = (uint8_t)po.outcome;
    r->iterations = po.iterations;
    r->inliers = po.inliers;
    r->average_squared_error = po.average_squared_error;
    r->risk = po.risk;
}
void posit_too_few(const double* T_estimate, svi_posit_result* r) {   // svi_solve_stereo_posit's answer for n <= 25
    std::memcpy(r->T_world_to_left, T_estimate, sizeof(r->T_world_to_left));
    r->outcome = SVI_POSIT_TOO_FEW_POINTS;
    r->iterations = 0;
    r->inliers = 0;
    r->average_squared_error = 0.0;
    r->risk = 0.0;
}
}  // namespace


namespace {
// getMaskActiveLandmarks on the device: lane.mask (plane 0) = 255 with a radius-7 disc of zeros per centre.  On success the
// centres may still be in flight: the caller synchronises lane 0 before it returns.
int build_mask(svi_ctx* ctx, Lane& l, const float* centres, int n_centres) {
    cudaStream_t s = l.stream;
    SyncOnFailure idle{s};
    const size_t bytes = (size_t)ctx->H * ctx->dev_pitch;
    mask_fill_kernel<<<(unsigned)((bytes / 16 + 256) / 256), 256, 0, s>>>(l.mask, bytes);
    if (n_centres > 0) {
        CallLayout L;
        const size_t i_c = L.take(sizeof(float) * 2 * n_centres);
        if (const int rc = reserve_call(ctx, L.end)) return rc;
        put(ctx, i_c, centres, sizeof(float) * 2 * n_centres);
        if (const int rc = call_send(ctx, L.end, s)) return rc;
        mask_discs_kernel<<<(n_centres * 15 + 255) / 256, 256, 0, s>>>(l.mask, ctx->W, ctx->H, ctx->dev_pitch, dev_at<float>(ctx, i_c), n_centres);
    }
    CK(cudaGetLastError());
    idle.done = true;
    return SVI_SUCCESS;
}

// ---- small call (the tracker's one pair per frame).  Pageable host buffers make every cudaMemcpyAsync a blocking
// staged copy; here the images are packed into the pinned buffer, every transfer is a real async DMA on the lane's
// stream, and the outputs come back as one batch that is scattered with memcpy.  The detection mask is either the
// caller's plane(s) or -- with `centres` -- built on the device from the landmark centres
// (getMaskActiveLandmarks, CFundamentalMatcher.cpp:2043-2073): 8 bytes per landmark go up instead of a W x H plane.
int small_call(svi_ctx* ctx, const uint8_t* left, const uint8_t* right, size_t pitch, size_t frame_stride, int n_frames,
               const uint8_t* masks, const float* centres, int n_centres, svi_stereo_result* out) {
    const int W = ctx->W, H = ctx->H, MC = ctx->p.max_corners, cap = out->capacity_per_frame;
    const size_t dstride = (size_t)H * ctx->dev_pitch;
    const FrameGeom g = make_geom(ctx, ctx->dev_pitch, dstride);
    {
        Lane& l = ctx->lanes[0];
        cudaStream_t s = l.stream;
        const int nf = n_frames;
        const size_t plane = dstride * nf;
        unsigned char* pin_in = ctx->pin;
        unsigned char* pin_out = ctx->pin + ((3 * (size_t)kSmallFrames * dstride + 15) & ~size_t(15));
        // upload order LEFT, mask, RIGHT: the detector starts as soon as LEFT (and the mask) is there; RIGHT goes up on the
        // side stream and its box sums run beside the detector (not while profiling: stage events live on one stream)
        cudaStream_t side = ctx->profiling ? nullptr : ctx->side;
        if (side) {   // whatever is still queued on the lane (an un-synchronised device-resident batch) uses the same scratch
            CK(cudaEventRecord(ctx->fork, s));
            CK(cudaStreamWaitEvent(side, ctx->fork, 0));
        }
        const uint8_t* srcs[3] = {left, masks, right};
        uint8_t* dsts[3] = {ctx->rect ? l.raw_l : l.img_l, l.mask, ctx->rect ? l.raw_r : l.img_r};
        auto upload_plane = [&](int k, cudaStream_t sk) -> int {
            if (!srcs[k]) return SVI_SUCCESS;
            if (host_is_pinned(srcs[k])) {   // the caller's buffer is page-locked: DMA straight from it
                if ((int)pitch == ctx->dev_pitch && (nf == 1 || frame_stride == dstride)) {
                    CK(cudaMemcpyAsync(dsts[k], srcs[k], plane, cudaMemcpyHostToDevice, sk));
                } else {
                    for (int f = 0; f < nf; ++f)
                        CK(cudaMemcpy2DAsync(dsts[k] + f * dstride, ctx->dev_pitch, srcs[k] + (size_t)f * frame_stride, pitch, W, H,
                                             cudaMemcpyHostToDevice, sk));
                }
                return SVI_SUCCESS;
            }
            unsigned char* stage = pin_in + k * (size_t)kSmallFrames * dstride;
            for (int f = 0; f < nf; ++f) {
                const uint8_t* src = srcs[k] + (size_t)f * frame_stride;
                if ((int)pitch == ctx->dev_pitch) std::memcpy(stage + f * dstride, src, dstride);
                else for (int y = 0; y < H; ++y) std::memcpy(stage + f * dstride + (size_t)y * ctx->dev_pitch, src + (size_t)y * pitch, W);
            }
            CK(cudaMemcpyAsync(dsts[k], stage, plane, cudaMemcpyHostToDevice, sk));
            return SVI_SUCCESS;
        };
        for (int k = 0; k < 2; ++k) {
            const int rc = upload_plane(k, s);
            if (rc != SVI_SUCCESS) return rc;
        }
        const std::function<int(cudaStream_t)> upload_right = [&](cudaStream_t sk) { return upload_plane(2, sk); };
        if (ctx->rect) {
            // raw images: RIGHT goes up on the side stream beside LEFT, one launch rectifies both into img_l / img_r, and the
            // RIGHT box sums still run on the side stream beside the detector
            const int rc = upload_plane(2, side ? side : s);
            if (rc != SVI_SUCCESS) { cudaStreamSynchronize(s); if (side) cudaStreamSynchronize(side); return rc; }
            if (side) {
                CK(cudaEventRecord(ctx->side_done, side));
                CK(cudaStreamWaitEvent(s, ctx->side_done, 0));
            }
            const int rr = rectify_pair(ctx, l.raw_l, l.raw_r, ctx->dev_pitch, dstride, l.img_l, l.img_r, nf, s);
            if (rr != SVI_SUCCESS) return rr;
            if (side) {
                CK(cudaEventRecord(ctx->fork, s));
                CK(cudaStreamWaitEvent(side, ctx->fork, 0));
            }
        }
        bool have_mask = masks != nullptr;
        if (centres) {
            int rc = build_mask(ctx, l, centres, n_centres);
            if (rc != SVI_SUCCESS) return rc;
            have_mask = true;
        }
        int rc = run_pipeline(ctx, l, l.img_l, l.img_r, have_mask ? l.mask : nullptr, g, nf, ctx->small_out, 0, ctx->small_n_kp, ctx->small_n_det, side,
                              ctx->rect ? nullptr : &upload_right);
        if (rc != SVI_SUCCESS) { cudaStreamSynchronize(s); if (side) cudaStreamSynchronize(side); return rc; }
        // one copy brings the whole result block back; only the live slots are scattered to the caller's arrays
        CK(cudaMemcpyAsync(pin_out, ctx->small_block, ctx->small_bytes, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        const StereoOutDev& so = ctx->small_out;
        auto host = [&](const void* d) { return pin_out + (static_cast<const unsigned char*>(d) - ctx->small_block); };
        const int* pin_kp = reinterpret_cast<const int*>(host(ctx->small_n_kp));
        const int* pin_det = reinterpret_cast<const int*>(host(ctx->small_n_det));
        struct Part { const void* dev; void* host; size_t elem; };   // elem = bytes per key-point slot
        const Part parts[8] = {{so.uv_l, out->uv_left, 8}, {so.uv_r, out->uv_right, 8}, {so.xyz, out->xyz_left, 24},
                               {so.desc_l, out->desc_left, 32}, {so.desc_r, out->desc_right, 32}, {so.dist, out->distance, 4},
                               {so.idx, out->match_index, 4}, {so.status, out->status, 1}};
        for (const Part& q : parts)
            for (int f = 0; f < nf; ++f)
                std::memcpy(static_cast<unsigned char*>(q.host) + (size_t)f * cap * q.elem, host(q.dev) + (size_t)f * MC * q.elem,
                            (size_t)std::min(std::max(pin_kp[f], 0), MC) * q.elem);
        std::memcpy(out->n_keypoints, pin_kp, sizeof(int) * nf);
        if (out->n_detected) std::memcpy(out->n_detected, pin_det, sizeof(int) * nf);
        return check_overflow(ctx);
    }
}

int triangulate_common(svi_ctx* ctx, bool left_search, const uint8_t* img, size_t pitch, int n, const float* search_range,
                       const float* top_left, const float* uv_ref, const uint8_t* desc_ref, float size, svi_tri_result* out) {
    if (!img || !top_left || !uv_ref || !desc_ref || !out || n < 0 || (int)pitch < ctx->W || (left_search && !search_range))
        return fail(ctx, SVI_ERR_INVALID, "svi_triangulate: bad argument");
    if (!out->uv || !out->xyz_left || !out->desc || !out->distance || !out->match_index || !out->status)
        return fail(ctx, SVI_ERR_INVALID, "svi_triangulate: null output array");
    if (n > ctx->p.max_queries) return fail(ctx, SVI_ERR_CAPACITY, "svi_triangulate: n > max_queries");
    if (n == 0) return SVI_SUCCESS;
    CK(cudaSetDevice(ctx->device));
    Lane& l = ctx->lanes[0];
    cudaStream_t s = l.stream;
    SyncOnFailure idle{s};
    const size_t N = (size_t)n;
    CallLayout L;   // [range (left search) | top_left | uv_ref | desc_ref] -> [uv | xyz | desc | dist | idx | status]
    const size_t i_range = left_search ? L.take(4 * N) : 0, i_tl = L.take(8 * N), i_uv = L.take(8 * N), i_desc = L.take(32 * N);
    const size_t in_end = L.end;
    const size_t o_uv = L.take(8 * N), o_xyz = L.take(24 * N), o_desc = L.take(32 * N), o_dist = L.take(4 * N), o_idx = L.take(4 * N),
                 o_status = L.take(N);
    if (const int rc = reserve_call(ctx, L.end)) return rc;
    int rc = stage_box(ctx, img, pitch, l.img_l, l.box_l, l.box_ls, s, left_search ? 0 : 1);
    if (rc != SVI_SUCCESS) return rc;
    if (left_search) put(ctx, i_range, search_range, 4 * N);
    put(ctx, i_tl, top_left, 8 * N);
    put(ctx, i_uv, uv_ref, 8 * N);
    put(ctx, i_desc, desc_ref, 32 * N);
    if ((rc = call_send(ctx, in_end, s)) != SVI_SUCCESS) return rc;
    CK(cudaMemsetAsync(ctx->call_dev + in_end, 0, L.end - in_end, s));
    const TriOutDev o{dev_at<float>(ctx, o_uv), dev_at<double>(ctx, o_xyz), dev_at(ctx, o_desc), dev_at<int>(ctx, o_dist), dev_at<int>(ctx, o_idx),
                      dev_at(ctx, o_status)};
    const float* d_tl = dev_at<float>(ctx, i_tl);
    const float* d_uv = dev_at<float>(ctx, i_uv);
    const uint8_t* d_desc = dev_at(ctx, i_desc);
    const FrameGeom g = make_geom(ctx, ctx->dev_pitch, (size_t)ctx->H * ctx->dev_pitch);
    const int blocks = (n + MATCH_WARPS - 1) / MATCH_WARPS;
    if (left_search)
        triangulate_kernel<true><<<blocks, MATCH_WARPS * 32, MATCH_SMEM, s>>>(l.map_l, l.map_ls, g, ctx->tc, n, dev_at<float>(ctx, i_range), d_tl, d_uv,
                                                                            d_desc, size, o);
    else
        triangulate_kernel<false><<<blocks, MATCH_WARPS * 32, MATCH_SMEM, s>>>(l.map_l, l.map_ls, g, ctx->tc, n, nullptr, d_tl, d_uv, d_desc, size, o);
    CK(cudaGetLastError());
    if ((rc = call_fetch(ctx, in_end, L.end, s)) != SVI_SUCCESS) return rc;
    idle.done = true;
    const unsigned char* h = ctx->call_pin;
    std::memcpy(out->uv, h + o_uv, 8 * N);
    std::memcpy(out->xyz_left, h + o_xyz, 24 * N);
    std::memcpy(out->desc, h + o_desc, 32 * N);
    std::memcpy(out->distance, h + o_dist, 4 * N);
    std::memcpy(out->match_index, h + o_idx, 4 * N);
    std::memcpy(out->status, h + o_status, N);
    return SVI_SUCCESS;
}
}  // namespace



namespace {

constexpr int kRoiRawCap = 8192;   // local maxima per stage-2 window (windows are at most ~600 x 600 px at the largest scaling)
constexpr int kRoiBatch = 4096;    // landmarks per wave of the window-mode detector

// Scratch of the tracking cascade: allocated once, at the first tracking call, sized from max_queries; never
// reallocated or freed inside a call.
int ensure_track_scratch(svi_ctx* ctx) {
    svi_ctx::RoiScratch& r = ctx->roi;
    if (r.items) return SVI_SUCCESS;
    const int items = std::min(std::max(ctx->p.max_queries, 64), kRoiBatch);
    const size_t MC = (size_t)ctx->p.max_corners;
    // [max | cand_count | defer | counters]: one block, so that a stage-2 side zeroes its bookkeeping with one memset
    CK(dmalloc(&r.max, (size_t)items * 3 + 4));
    r.cand_count = reinterpret_cast<int*>(r.max) + items;
    r.defer = r.cand_count + items;
    r.counters = r.defer + items;
    CK(dmalloc(&r.cand, (size_t)items * kRoiRawCap));
    CK(dmalloc(&r.det, (size_t)items * MC));
    CK(dmalloc(&r.kp, (size_t)items * MC));
    CK(dmalloc(&r.n_det, (size_t)items));
    CK(dmalloc(&r.n_kp, (size_t)items));
    CK(dmalloc(&r.rois, (size_t)items));
    CK(dmalloc(&r.s2, (size_t)items));
    CK(dmalloc(&ctx->s3_items, (size_t)std::max(ctx->p.max_queries, 64)));
    r.items = items;
    return SVI_SUCCESS;
}

TrackPlanConst make_plan(const svi_ctx* ctx, const double* T, const svi_camera& cam, double motion_scaling) {
    TrackPlanConst k;
    for (int i = 0; i < 12; ++i) { k.T[i] = T[i]; k.P[i] = cam.P[i]; }
    k.motion_scaling = motion_scaling;
    k.W = ctx->W; k.H = ctx->H;
    k.block = 15;        // m_uSearchBlockSizePoseOptimization (CFundamentalMatcher.h:95)
    k.epi_base = 15.0;   // m_dEpipolarLineBaseLength (CFundamentalMatcher.h:92)
    return k;
}

// One side of trackManual stage 2 for every landmark that is still untracked, entirely enqueued on the lane's stream:
// window arithmetic (:1548-1575) in stage2_plan_kernel, GFTT inside the windows (window-mode Harris + selection),
// description, matching and triangulation in track_stage2_kernel.  Landmarks go through in waves of kRoiBatch.
int track_stage2_side(svi_ctx* ctx, Lane& l, const FrameGeom& g, int n, const double* T, double motion_scaling, bool left,
                      const LandmarksDev& ld, const TrackOutDev& o) {
    cudaStream_t s = l.stream;
    const svi_camera& cam = left ? ctx->cam_l : ctx->cam_r;
    svi_ctx::RoiScratch& r = ctx->roi;
    if (!ctx->select_smem) return fail(ctx, SVI_ERR_UNSUPPORTED, "svi_track_landmarks: stage 2 needs max_candidates <= 16384");
    const TrackPlanConst k = make_plan(ctx, T, cam, motion_scaling);
    // upper bound of the window size (the grid of the window-mode detector): the principal weight is largest at the
    // image edge that is farthest from the principal point
    const double cx = cam.P[2], cy = cam.P[6];
    const double su = std::round(std::sqrt(std::max(std::fabs(cx), std::fabs((double)ctx->W - cx))) / 10.0 + motion_scaling);
    const double sv = std::round(std::sqrt(std::max(std::fabs(cy), std::fabs((double)ctx->H - cy))) / 10.0 + motion_scaling);
    const int max_w = std::min(ctx->W, 2 * (int)std::round(su * 15.0) + 2), max_h = std::min(ctx->H, 2 * (int)std::round(sv * 15.0) + 2);
    if (max_w <= 0 || max_h <= 0) return SVI_SUCCESS;   // no window can exist: the plan kernel reports "no features" per landmark
    SelectParams sp = ctx->sel;
    sp.raw_cap = kRoiRawCap;
    sp.cand_cap = std::min(ctx->cand_cap, kRoiRawCap);
    sp.cell = std::max(1, (int)std::ceil(ctx->p.min_distance));
    sp.cell_magic = sp.cell < 256 ? (uint32_t)(((1u << 24) + sp.cell - 1) / sp.cell) : 0u;
    int* n_items = r.counters + (left ? 0 : 1);
    for (int q0 = 0; q0 < n; q0 += r.items) {
        const int nb = std::min(r.items, n - q0);
        CK(cudaMemsetAsync(r.max, 0, sizeof(int) * ((size_t)r.items * 3 + 4), s));   // max, cand_count, defer, counters
        stage2_plan_kernel<<<(nb + 127) / 128, 128, 0, s>>>(k, left ? 0 : 1, (float)(1.0 + motion_scaling), ld, q0, q0 + nb, o, r.rois, r.s2, n_items);
        harris_box_kernel<<<harris_grid(max_w, max_h, nb), HT_THREADS, sizeof(HarrisSmem), s>>>(
            ctx->trk_img, nullptr, g, ctx->f1, ctx->f0, ctx->p.harris_k, ctx->p.quality_level, nullptr, nullptr, nullptr, r.max, r.cand,
            r.cand_count, kRoiRawCap, r.rois, n_items, 0);
        // thousands of small windows: seven small-configuration CTAs per SM; the rare window that does not fit is
        // deferred to the frame-size configuration (its CTAs return at once for every other window)
        select_corners_kernel<true, SEL_SMALL_THREADS, SEL_SMALL_KEYS, SEL_SMALL_CELLS>
            <<<nb, SEL_SMALL_THREADS, select_smem_bytes(SEL_SMALL_KEYS, SEL_SMALL_CELLS), s>>>(
                r.cand, r.cand_count, r.max, sp, nullptr, nullptr, nullptr, r.det, r.n_det, r.kp, r.n_kp, ctx->d_overflow, r.rois, r.defer, nullptr, n_items);
        select_corners_kernel<true><<<nb, SEL_THREADS, 13 * SEL_SMEM_KEYS, s>>>(r.cand, r.cand_count, r.max, sp, nullptr, nullptr, nullptr, r.det,
                                                                              r.n_det, r.kp, r.n_kp, ctx->d_overflow, r.rois, nullptr, r.defer, n_items);
        const int blocks = (nb + MATCH_WARPS - 1) / MATCH_WARPS;
        if (left)
            track_stage2_kernel<true><<<blocks, MATCH_WARPS * 32, MATCH_SMEM, s>>>(l.box_l, l.map_r, l.map_rs, g, ctx->tc, ctx->p.cutoff_stage2,
                                                                                  r.s2, n_items, r.det, r.n_det, ctx->p.max_corners, ld, o);
        else
            track_stage2_kernel<false><<<blocks, MATCH_WARPS * 32, MATCH_SMEM, s>>>(l.box_r, l.map_l, l.map_ls, g, ctx->tc, ctx->p.cutoff_stage2,
                                                                                   r.s2, n_items, r.det, r.n_det, ctx->p.max_corners, ld, o);
        CK(cudaGetLastError());
    }
    return SVI_SUCCESS;
}

// Stage 3 (epipolar line in LEFT): line geometry per landmark in stage3_plan_kernel (:1795-1947), sampling / matching /
// triangulation in track_stage3_kernel, both enqueued on the lane's stream.
int track_stage3_all(svi_ctx* ctx, Lane& l, const FrameGeom& g, int n, const double* T, double motion_scaling, const LandmarksDev& ld,
                     const Stage3Extra& ex, const uint8_t* d_orig, const TrackOutDev& o, const int* n_dev) {
    cudaStream_t s = l.stream;
    int* n_items = ctx->roi.counters + 2;
    const TrackPlanConst k = make_plan(ctx, T, ctx->cam_l, motion_scaling);
    CK(cudaMemsetAsync(n_items, 0, sizeof(int), s));
    stage3_plan_kernel<<<(n + 127) / 128, 128, 0, s>>>(k, ld, ex, n, n_dev, o, ctx->s3_items, n_items);
    track_stage3_kernel<<<(n + MATCH_WARPS - 1) / MATCH_WARPS, MATCH_WARPS * 32, MATCH_SMEM, s>>>(
        l.box_l, l.map_r, l.map_rs, g, ctx->tc, ctx->p.cutoff_stage3, ctx->p.cutoff_original, ctx->s3_items, n_items, d_orig, ld, o);
    CK(cudaGetLastError());
    return SVI_SUCCESS;
}

// Both images of the pair into the tracking planes of lane 0 (rectified first while svi_set_rectification is set) with their box
// sums: RIGHT goes up and gets its box sums on the side stream, beside LEFT's; lane 0's stream waits for both.
int stage_track_pair(svi_ctx* ctx, const uint8_t* img_left, const uint8_t* img_right, size_t pitch) {
    Lane& l = ctx->lanes[0];
    cudaStream_t s = l.stream;
    const size_t plane = (size_t)ctx->H * ctx->dev_pitch;
    // both images as planes 0 / 1 of one buffer (the window-mode detector indexes them by plane)
    CK(cudaEventRecord(ctx->fork, s));
    CK(cudaStreamWaitEvent(ctx->side, ctx->fork, 0));
    int rc = stage_box(ctx, img_right, pitch, ctx->trk_img + plane, l.box_r, l.box_rs, ctx->side, 1, 1);
    if (rc == SVI_SUCCESS) rc = stage_box(ctx, img_left, pitch, ctx->trk_img, l.box_l, l.box_ls, s, 0);
    if (cudaEventRecord(ctx->side_done, ctx->side) != cudaSuccess || cudaStreamWaitEvent(s, ctx->side_done, 0) != cudaSuccess)
        rc = rc == SVI_SUCCESS ? fail(ctx, SVI_ERR_CUDA, "svi_track_landmarks: joining the side stream failed") : rc;
    if (rc != SVI_SUCCESS) { cudaStreamSynchronize(ctx->side); cudaStreamSynchronize(s); }
    return rc;
}

// The tracking cascade restricted to stage_mask on n device-resident landmarks whose outputs `o` are zeroed, entirely enqueued on
// lane 0's stream after the images staged by stage_track_pair: every stage reads the stage / status bytes the previous one left on
// the device and plans its own work items there.  n_dev (stage 3 alone, may be null): the landmark count when only the device
// knows it, n is then its upper bound.
int enqueue_cascade(svi_ctx* ctx, int n, const double* T_world_to_left, double motion_scaling, uint32_t stage_mask, const LandmarksDev& ld,
                    const Stage3Extra& ex, const uint8_t* d_orig, const TrackOutDev& o, const int* n_dev) {
    Lane& l = ctx->lanes[0];
    cudaStream_t s = l.stream;
    TrackConst k;
    for (int i = 0; i < 12; ++i) { k.T[i] = T_world_to_left[i]; k.PL[i] = ctx->cam_l.P[i]; k.PR[i] = ctx->cam_r.P[i]; }
    k.tri_scale = (float)(1.0 + motion_scaling);
    k.cutoff1 = ctx->p.cutoff_stage1;
    k.stage1_match = (stage_mask & SVI_STAGE_1) ? 1 : 0;
    const FrameGeom g = make_geom(ctx, ctx->dev_pitch, (size_t)ctx->H * ctx->dev_pitch);
    if (stage_mask & (SVI_STAGE_1 | SVI_STAGE_2)) {
        // ---- stage 1 LEFT / RIGHT for every landmark (or only its field-of-view gate when stage 2 runs alone)
        track_stage1_kernel<<<(n + MATCH_WARPS - 1) / MATCH_WARPS, MATCH_WARPS * 32, MATCH_SMEM, s>>>(l.box_l, l.box_r, l.map_l, l.map_ls, l.map_r, l.map_rs, g,
                                                                                                      ctx->tc, k, ld, n, o);
        CK(cudaGetLastError());
    } else {
        // stage 3 alone (trackEpipolar :828-1020): no gate, every landmark is an untracked candidate
        CK(cudaMemsetAsync(o.status, SVI_TRK_STAGE1_DIST, (size_t)n, s));
        CK(cudaMemsetAsync(o.stage, 0, (size_t)n, s));
    }
    // ---- stage 2 LEFT, then stage 2 RIGHT, for what is still untracked
    for (int side = 0; side < 2 && (stage_mask & SVI_STAGE_2); ++side) {
        const int rc = track_stage2_side(ctx, l, g, n, T_world_to_left, motion_scaling, side == 0, ld, o);
        if (rc != SVI_SUCCESS) { cudaStreamSynchronize(s); return rc; }
    }
    // ---- stage 3 (epipolar line in LEFT)
    if (stage_mask & SVI_STAGE_3) {
        const int rc = track_stage3_all(ctx, l, g, n, T_world_to_left, motion_scaling, ld, ex, d_orig, o, n_dev);
        if (rc != SVI_SUCCESS) { cudaStreamSynchronize(s); return rc; }
    }
    return SVI_SUCCESS;
}

}  // namespace

// ---- the batch frame entry points (svi_stereo_frames[_sparse][_device]): argument checks and the chunk loops they share
namespace {
int check_frames_args(svi_ctx* ctx, const char* name, const uint8_t* left, const uint8_t* right, size_t pitch, size_t frame_stride,
                      int n_frames, const svi_stereo_result* out, bool device) {
    const std::string n(name);
    if (!left || !right || !out || n_frames < 0 || (int)pitch < ctx->W ||
        (device ? frame_stride < pitch * (size_t)ctx->H : (n_frames > 1 && frame_stride < pitch * (size_t)ctx->H)))
        return fail(ctx, SVI_ERR_INVALID, n + ": bad argument");
    if (out->capacity_per_frame < ctx->p.max_corners) return fail(ctx, SVI_ERR_CAPACITY, n + ": capacity_per_frame < max_corners");
    if (!out->n_keypoints || !out->uv_left || !out->uv_right || !out->xyz_left || !out->desc_left || !out->desc_right ||
        !out->distance || !out->match_index || !out->status)
        return fail(ctx, SVI_ERR_INVALID, n + ": null output array");
    return SVI_SUCCESS;
}

// nf frames of one per-slot array of a lane (max_corners slots per frame, elem bytes each) into the caller's host array of
// cap slots per frame, from frame f0 on
cudaError_t d2h_slots(void* dst, const void* src, size_t elem, int MC, int cap, int f0, int nf, cudaStream_t s) {
    unsigned char* d = static_cast<unsigned char*>(dst) + (size_t)f0 * cap * elem;
    if (cap == MC) return cudaMemcpyAsync(d, src, (size_t)nf * MC * elem, cudaMemcpyDeviceToHost, s);
    return cudaMemcpy2DAsync(d, (size_t)cap * elem, src, (size_t)MC * elem, (size_t)MC * elem, nf, cudaMemcpyDeviceToHost, s);
}

// Host buffers: chunk c on lane c % n_lanes; its images (and masks) go straight from the caller's buffers into the lane's
// staging (raw planes first while rectification is set), `run` enqueues the kernels on the lane's planes, the slot arrays and
// counts come back into the caller's arrays, `fetch` (may be null) adds the entry point's own; one synchronisation at the end.
using HostChunkFn = std::function<int(Lane&, const FrameGeom&, int f0, int nf)>;
int host_frames(svi_ctx* ctx, const uint8_t* left, const uint8_t* right, size_t pitch, size_t frame_stride, int n_frames,
                const uint8_t* masks, svi_stereo_result* out, const HostChunkFn& run, const HostChunkFn& fetch) {
    const int W = ctx->W, H = ctx->H, MC = ctx->p.max_corners, cap = out->capacity_per_frame;
    const size_t dstride = (size_t)H * ctx->dev_pitch;
    const FrameGeom g = make_geom(ctx, ctx->dev_pitch, dstride);
    const bool dense = (frame_stride == pitch * (size_t)H);
    int chunk_id = 0;
    for (int f0 = 0; f0 < n_frames; f0 += ctx->chunk, ++chunk_id) {
        Lane& l = ctx->lanes[chunk_id % ctx->n_lanes];
        cudaStream_t s = l.stream;
        const int nf = std::min(ctx->chunk, n_frames - f0);
        const uint8_t* srcs[3] = {left, right, masks};
        uint8_t* dsts[3] = {ctx->rect ? l.raw_l : l.img_l, ctx->rect ? l.raw_r : l.img_r, l.mask};
        for (int k = 0; k < 3; ++k) {
            if (!srcs[k]) continue;
            if (dense && (int)pitch == ctx->dev_pitch) {
                CK(cudaMemcpyAsync(dsts[k], srcs[k] + (size_t)f0 * frame_stride, (size_t)nf * frame_stride, cudaMemcpyHostToDevice, s));
            } else if (dense) {
                CK(cudaMemcpy2DAsync(dsts[k], ctx->dev_pitch, srcs[k] + (size_t)f0 * frame_stride, pitch, W, (size_t)H * nf,
                                     cudaMemcpyHostToDevice, s));
            } else {
                for (int f = 0; f < nf; ++f)
                    CK(cudaMemcpy2DAsync(dsts[k] + f * dstride, ctx->dev_pitch, srcs[k] + (size_t)(f0 + f) * frame_stride,
                                         pitch, W, H, cudaMemcpyHostToDevice, s));
            }
        }
        if (ctx->rect) {
            const int rr = rectify_pair(ctx, l.raw_l, l.raw_r, ctx->dev_pitch, dstride, l.img_l, l.img_r, nf, s);
            if (rr != SVI_SUCCESS) return rr;
        }
        int rc = run(l, g, f0, nf);
        if (rc != SVI_SUCCESS) return rc;
        CK(d2h_slots(out->uv_left, l.out.uv_l, 2 * sizeof(float), MC, cap, f0, nf, s));
        CK(d2h_slots(out->uv_right, l.out.uv_r, 2 * sizeof(float), MC, cap, f0, nf, s));
        CK(d2h_slots(out->xyz_left, l.out.xyz, 3 * sizeof(double), MC, cap, f0, nf, s));
        CK(d2h_slots(out->desc_left, l.out.desc_l, 32, MC, cap, f0, nf, s));
        CK(d2h_slots(out->desc_right, l.out.desc_r, 32, MC, cap, f0, nf, s));
        CK(d2h_slots(out->distance, l.out.dist, sizeof(int32_t), MC, cap, f0, nf, s));
        CK(d2h_slots(out->match_index, l.out.idx, sizeof(int32_t), MC, cap, f0, nf, s));
        CK(d2h_slots(out->status, l.out.status, 1, MC, cap, f0, nf, s));
        CK(cudaMemcpyAsync(out->n_keypoints + f0, l.n_kp, sizeof(int) * nf, cudaMemcpyDeviceToHost, s));
        if (out->n_detected) CK(cudaMemcpyAsync(out->n_detected + f0, l.n_det, sizeof(int) * nf, cudaMemcpyDeviceToHost, s));
        if (fetch && (rc = fetch(l, g, f0, nf)) != SVI_SUCCESS) return rc;
    }
    int rc = sync_lanes(ctx);
    if (rc != SVI_SUCCESS) return rc;
    return check_overflow(ctx);
}

// Device buffers: enqueued after everything on the caller's stream, chunk c on lane c % n_lanes (lane 0 while profiling in
// mode 2); `run` enqueues the kernels on device images and writes the caller's arrays at frame f0 (o, n_kp, n_det); the
// lanes join the caller's stream again, no synchronisation.
using DeviceChunkFn = std::function<int(Lane&, const uint8_t*, const uint8_t*, const uint8_t*, const FrameGeom&, int f0, int nf,
                                        const StereoOutDev& o, int* n_kp, int* n_det)>;
int device_frames(svi_ctx* ctx, const uint8_t* left, const uint8_t* right, size_t pitch, size_t frame_stride, int n_frames,
                  const uint8_t* masks, const svi_stereo_result* out, void* cuda_stream, const DeviceChunkFn& run) {
    cudaStream_t user = reinterpret_cast<cudaStream_t>(cuda_stream);
    CK(cudaEventRecord(ctx->fork, user));
    for (int i = 0; i < ctx->n_lanes; ++i) CK(cudaStreamWaitEvent(ctx->lanes[i].stream, ctx->fork, 0));
    const FrameGeom g = make_geom(ctx, (int)pitch, frame_stride);
    const size_t dstride = (size_t)ctx->H * ctx->dev_pitch;
    const FrameGeom g_rect = make_geom(ctx, ctx->dev_pitch, dstride);   // rectified planes in the lane's staging
    StereoOutDev o;
    o.cap = out->capacity_per_frame;
    o.uv_l = out->uv_left; o.uv_r = out->uv_right; o.xyz = out->xyz_left;
    o.desc_l = out->desc_left; o.desc_r = out->desc_right;
    o.dist = out->distance; o.idx = out->match_index; o.status = out->status;
    int chunk_id = 0, rc = SVI_SUCCESS;
    for (int f0 = 0; f0 < n_frames; f0 += ctx->chunk, ++chunk_id) {
        Lane& l = ctx->lanes[ctx->serial ? 0 : chunk_id % ctx->n_lanes];
        const int nf = std::min(ctx->chunk, n_frames - f0);
        int* n_det = out->n_detected ? out->n_detected + f0 : l.n_det;
        const uint8_t* m = masks ? masks + (size_t)f0 * frame_stride : nullptr;
        if (ctx->rect) {   // the caller's raw frames are read in place; the pipeline reads the rectified planes
            rc = rectify_pair(ctx, left + (size_t)f0 * frame_stride, right + (size_t)f0 * frame_stride, pitch, frame_stride, l.img_l, l.img_r, nf,
                              l.stream);
            if (rc != SVI_SUCCESS) break;
            if (m && ((int)pitch != ctx->dev_pitch || frame_stride != dstride)) {   // the masks follow the planes' layout
                for (int f = 0; f < nf && rc == SVI_SUCCESS; ++f)
                    if (cudaMemcpy2DAsync(l.mask + f * dstride, ctx->dev_pitch, m + (size_t)f * frame_stride, pitch, ctx->W, ctx->H,
                                          cudaMemcpyDeviceToDevice, l.stream) != cudaSuccess)
                        rc = fail(ctx, SVI_ERR_CUDA, "svi_stereo_frames_device: mask copy failed");
                if (rc != SVI_SUCCESS) break;
                m = l.mask;
            }
            rc = run(l, l.img_l, l.img_r, m, g_rect, f0, nf, o, out->n_keypoints + f0, n_det);
        } else {
            rc = run(l, left + (size_t)f0 * frame_stride, right + (size_t)f0 * frame_stride, m, g, f0, nf, o, out->n_keypoints + f0, n_det);
        }
        if (rc != SVI_SUCCESS) break;
    }
    // join the lanes back into the caller's stream -- also after a failure, so that nothing queued so far can outlive
    // the caller's next use of its buffers
    for (int i = 0; i < ctx->n_lanes; ++i) {
        if (cudaEventRecord(ctx->lanes[i].done, ctx->lanes[i].stream) == cudaSuccess)
            cudaStreamWaitEvent(user, ctx->lanes[i].done, 0);
    }
    return rc;
}

}  // namespace

extern "C" {

int svi_params_default(svi_params* p) {
    if (!p) return SVI_ERR_INVALID;
    std::memset(p, 0, sizeof(*p));
    p->quality_level = 0.01;
    p->min_distance = 7.0;
    p->harris_k = 0.04;
    p->min_disparity_px = 0.01;
    p->max_corners = 1000;
    p->keypoint_size = 7.0f;
    p->search_range_px = 60.0f;
    p->match_cutoff = 100.0f;
    p->cutoff_stage1 = 25.0f;
    p->cutoff_stage2 = 50.0f;
    p->cutoff_stage3 = 50.0f;
    p->cutoff_original = 100.0f;
    p->max_candidates = 16384;
    p->chunk_frames = 0;
    p->max_queries = 16384;
    p->detector = SVI_DETECTOR_GFTT_HARRIS;
    p->fast_threshold = 10;
    p->fast_nonmax = 1;
    return SVI_SUCCESS;
}

const char* svi_status_text(int status) {
    switch (status) {
        case SVI_OK: return "ok";
        case SVI_TRI_RANGE: return "<CTriangulator>(getPointTriangulatedInRIGHT) insufficient search range";
        case SVI_TRI_NO_DESC: return "<CTriangulator>(getPointTriangulatedInRIGHT) could not compute descriptors";
        case SVI_TRI_NO_MATCH: return "<CTriangulator>(getPointTriangulatedInRIGHT) no match found";
        case SVI_TRI_DISTANCE: return "<CTriangulator>(getPointTriangulatedInRIGHT) matching distance";
        case SVI_TRI_ZERO_DISP: return "<CTriangulator>(getPointInLEFT) zero disparity";
        case SVI_TRI_BAD_ROI: return "search region outside image";
        case SVI_TRK_DEPTH: return "invalid depth";
        case SVI_TRK_STAGE1_DIST: return "insufficient matching distance";
        case SVI_TRK_TRI_DESC: return "triangulation descriptor mismatch";
        case SVI_TRK_OUT_OF_FOV: return "projection outside the field of view";
        case SVI_TRK_NO_FEATURES: return "no features detected";
        case SVI_TRK_NO_MATCHES: return "no matches found";
        case SVI_TRK_DESC: return "descriptor mismatch";
        case SVI_TRK_RANGE: return "out of tracking range";
        case SVI_EPI_OUT_OF_SIGHT: return "<CFundamentalMatcher>(getVisibleLandmarksFundamental) projection out of sight";
        case SVI_EPI_VERTICAL: return "<CFundamentalMatcher>(getVisibleLandmarksFundamental) vertical out of sight";
        case SVI_EPI_NEG_SLOPE: return "<CFundamentalMatcher>(getVisibleLandmarksFundamental) caught bad projection negative slope";
        case SVI_EPI_POS_SLOPE: return "<CFundamentalMatcher>(getVisibleLandmarksFundamental) caught bad projection positive slope";
        case SVI_EPI_ZERO_LEN: return "<CFundamentalMatcher>(getVisibleLandmarksFundamental) zero line length";
        case SVI_EPI_POOL_EMPTY: return "could not find a matching descriptor (empty key point pool)";
        case SVI_EPI_NO_MATCHES: return "could not find any matches (empty matches pool)";
        case SVI_EPI_DIST: return "could not find a matching descriptor";
        case SVI_EPI_ORIG_DIST: return "could not find a matching descriptor (ORIGINAL matching distance too big)";
        case SVI_EPI_NO_TRANSLATION: return "no translation since detection: epipolar search skipped";
        case SVI_SPARSE_NOT_MUTUAL: return "left-right check: the matched RIGHT key-point's best LEFT match is another key-point";
        default: return "unknown status";
    }
}

const char* svi_brief_table_info(void) { return SVI_BRIEF_PATTERN_SOURCE; }

int svi_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

const char* svi_last_error(const svi_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

void svi_destroy(svi_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    for (int i = 0; i < kMaxLanes; ++i) {
        Lane& l = ctx->lanes[i];
        if (l.stream) cudaStreamSynchronize(l.stream);
        void* ptrs[] = {l.box_l, l.box_r, l.box_ls, l.box_rs, l.frame_max, l.cand_count, l.cand, l.det_xy, l.kp_xy, l.n_det, l.n_kp,
                        l.g_head, l.g_next, l.g_state, l.img_l, l.img_r, l.mask, l.out.uv_l, l.out.uv_r, l.out.xyz,
                        l.out.desc_l, l.out.desc_r, l.out.dist, l.out.idx, l.out.status, l.bin_start, l.bin_slot, l.bin_kp,
                        l.raw_l, l.raw_r, l.sp_kp_r, l.sp_n_kp_r, l.sp_n_det_r, l.sp_row_l, l.sp_slot_l, l.sp_kp_l, l.sp_row_r,
                        l.sp_slot_r, l.sp_kp_rs, l.sp_desc_r, l.sp_second, l.sp_desc_lr, l.sp_rev};
        for (void* p : ptrs) if (p) cudaFree(p);
        for (cudaEvent_t e : l.ev) cudaEventDestroy(e);
        if (l.done) cudaEventDestroy(l.done);
        if (l.stream) cudaStreamDestroy(l.stream);
    }
    if (ctx->h_overflow) cudaFreeHost(const_cast<int*>(ctx->h_overflow));
    if (ctx->side_done) cudaEventDestroy(ctx->side_done);
    if (ctx->side) cudaStreamDestroy(ctx->side);
    if (ctx->call_dev) cudaFree(ctx->call_dev);
    if (ctx->call_pin) cudaFreeHost(ctx->call_pin);
    if (ctx->pin) cudaFreeHost(ctx->pin);
    if (ctx->small_block) cudaFree(ctx->small_block);
    if (ctx->trk_img) cudaFree(ctx->trk_img);
    if (ctx->s3_items) cudaFree(ctx->s3_items);
    if (ctx->resp_one) cudaFree(ctx->resp_one);
    if (ctx->rect_map) cudaFree(ctx->rect_map);
    {
        void* rp[] = {ctx->roi.max, ctx->roi.cand, ctx->roi.det, ctx->roi.kp, ctx->roi.n_det, ctx->roi.n_kp, ctx->roi.rois, ctx->roi.s2};
        for (void* q : rp) if (q) cudaFree(q);
    }
    if (ctx->fork) cudaEventDestroy(ctx->fork);
    delete ctx;
}

int svi_create(const svi_camera* left, const svi_camera* right, const svi_params* params, int device, svi_ctx** out) {
    svi_ctx* ctx = nullptr;
    if (!left || !right || !out) return fail(nullptr, SVI_ERR_INVALID, "svi_create: null argument");
    *out = nullptr;
    int ndev = svi_device_count();
    if (ndev <= 0) return fail(nullptr, SVI_ERR_NO_DEVICE, "svi_create: no CUDA device (libsvi_gpu has no CPU fallback)");
    if (device < 0 || device >= ndev) return fail(nullptr, SVI_ERR_INVALID, "svi_create: bad device index");
    if (left->width != right->width || left->height != right->height)
        return fail(nullptr, SVI_ERR_INVALID, "svi_create: left/right image sizes differ");
    if (left->width < 64 || left->height < 64 || left->width > 65535 || left->height > 65535)
        return fail(nullptr, SVI_ERR_INVALID, "svi_create: image size must be within [64, 65535]");
    svi_params p;
    if (params) p = *params; else svi_params_default(&p);
    if (p.max_corners <= 0 || p.max_corners > 65535) return fail(nullptr, SVI_ERR_INVALID, "svi_create: max_corners must be in [1, 65535]");
    // CTriangulator rejects a match whose disparity is below the minimum; at 0 a zero-disparity match would pass and put
    // the point at infinite depth (and the depth bound du / min_disparity_px would be infinite too)
    if (!(p.min_disparity_px > 0.0)) return fail(nullptr, SVI_ERR_INVALID, "svi_create: min_disparity_px must be positive");
    if (p.max_candidates < 1024) p.max_candidates = 1024;
    if (p.max_queries < 1) p.max_queries = 1;
    {
        cudaError_t e = cudaSetDevice(device);
        if (e != cudaSuccess) return fail(nullptr, SVI_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
    }
    ctx = new svi_ctx();
#undef CK
#define CK(call)                                                                                 \
    do {                                                                                         \
        cudaError_t e_ = (call);                                                                 \
        if (e_ != cudaSuccess) {                                                                 \
            std::string m_ = std::string(#call) + ": " + cudaGetErrorString(e_);                 \
            svi_destroy(ctx);                                                                    \
            return fail(nullptr, SVI_ERR_CUDA, m_);                                              \
        }                                                                                        \
    } while (0)
    ctx->device = device;
    ctx->cam_l = *left;
    ctx->cam_r = *right;
    ctx->p = p;
    {
        int n_sm = 0;
        if (cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && n_sm > 0) ctx->n_sm = n_sm;
    }
    ctx->W = (int)left->width;
    ctx->H = (int)left->height;
    ctx->dev_pitch = ctx->W;  // dense rows: staging copies are 1-D DMA transfers at full PCIe rate
    ctx->resp_pitch = align_up(ctx->W, 32);
    ctx->box_pitch = align_up(ctx->W, 64);
    const char* env_chunk = std::getenv("SVI_CHUNK_FRAMES");
    const char* env_lanes = std::getenv("SVI_LANES");
    // default: 64 KITTI-size frames per launch (measured sweep, profiles/r1_lane_sweep.txt), fewer for larger images so
    // that the scratch of a lane stays near half a gigabyte
    const int auto_chunk = (int)std::max<long long>(4, std::min<long long>(64, 30000000LL / ((long long)ctx->W * ctx->H)));
    ctx->chunk = p.chunk_frames > 0 ? p.chunk_frames : (env_chunk ? std::atoi(env_chunk) : auto_chunk);
    ctx->chunk = std::max(1, std::min(ctx->chunk, 4096));
    ctx->n_lanes = env_lanes ? std::max(1, std::min(std::atoi(env_lanes), kMaxLanes)) : 6;
    ctx->profiling = std::getenv("SVI_PROFILE") != nullptr;
    if (const char* e = std::getenv("SVI_MATCH_SPLIT")) {
        const int v = std::atoi(e);
        if (v == 1 || v == 2) ctx->match_split = v;
    }
    if (const char* e = std::getenv("SVI_MATCH_PRE")) ctx->match_pre = std::atoi(e) != 0;
    {   // The binned matcher's tile is laid out for scan lines of one pass (pool size ceil(range) + 1 <= 62 candidates) whose
        // ROI border 4 * size is a whole number of pixels: the reference's 60 px / size 7.  It pays on dense frames only
        // (measured, frames/s device-resident: C2, ~13 key-points per bin, 109.0 k vs 103.9 k for the per-key-point
        // kernels; C4, ~7 per bin, 132.2 k vs 136.0 k): expected key-points per bin = ~0.8 of max_corners (BRIEF's border
        // filter) spread over the image minus that border.  Anything else keeps the per-key-point kernels.
        int mode = 1;
        if (const char* e = std::getenv("SVI_MATCH_BINNED")) mode = std::atoi(e);
        const float b4 = 4.f * p.keypoint_size;
        const bool geom_ok = p.search_range_px > 0.f && std::ceil(p.search_range_px) + 1.f <= (float)BT_REACH && b4 == std::floor(b4) && b4 >= 1.f;
        const double per_bin = 0.8 * p.max_corners * (double)(BinWide::BIN_W * BinWide::BIN_H) /
                               std::max(1.0, (double)(ctx->W - 2 * kBriefBorder) * (double)(ctx->H - 2 * kBriefBorder));
        ctx->match_binned = geom_ok && (mode == 2 || (mode == 1 && per_bin >= 10.0));
        ctx->nbx = (ctx->W + BinWide::BIN_W - 1) / BinWide::BIN_W;
        ctx->n_bins = ctx->nbx * ((ctx->H + BinWide::BIN_H - 1) / BinWide::BIN_H);
        if (ctx->n_bins * (int)sizeof(uint32_t) > 40000) ctx->match_binned = false;   // the bin histogram must fit the default dynamic shared memory
    }
    ctx->trace = std::getenv("SVI_TRACE") != nullptr;
    int cap = 1024;
    while (cap < p.max_candidates) cap <<= 1;
    ctx->cand_cap = cap;
    ctx->raw_cap = cap * kRawFactor;

    // cornerHarris scale: 1 / ((1 << (ksize-1)) * blockSize) / 255 for 8-bit input (ksize 3, block 7)
    const double scale = 1.0 / (4.0 * 7.0 * 255.0);
    ctx->f1 = (float)scale;
    ctx->f0 = (float)(2.0 * scale);

    // goodFeaturesToTrack's bucket grid; cell >= minDistance keeps the 3x3 neighbourhood sufficient
    SelectParams& sp = ctx->sel;
    sp.W = ctx->W; sp.H = ctx->H;
    sp.cand_cap = cap;
    sp.raw_cap = cap * kRawFactor;
    sp.quality = p.quality_level;
    sp.max_corners = p.max_corners;
    sp.filter = p.min_distance >= 1.0 ? 1 : 0;
    sp.cap_is_error = 0;
    if (p.detector == SVI_DETECTOR_FAST_9_16) {   // cv::FAST: no distance filter, no maxCorners cut
        sp.filter = 0;
        sp.cap_is_error = 1;
    } else if (p.detector != SVI_DETECTOR_GFTT_HARRIS) {
        delete ctx;
        return fail(nullptr, SVI_ERR_INVALID, "svi_create: unknown detector");
    }
    sp.min_dist_sq = p.min_distance * p.min_distance;
    int cell = std::max(1, (int)std::ceil(p.min_distance));
    while (((ctx->W + cell - 1) / cell) * ((ctx->H + cell - 1) / cell) > SEL_SMEM_CELLS && cap <= SEL_SMEM_KEYS && cell < 64) ++cell;
    sp.cell = cell;
    sp.cell_magic = cell < 256 ? (uint32_t)(((1u << 24) + cell - 1) / cell) : 0u;
    sp.min_dist_sq_ceil = (int)std::min(std::ceil(sp.min_dist_sq), 2.0e9);
    sp.gw = (ctx->W + cell - 1) / cell;
    sp.gh = (ctx->H + cell - 1) / cell;
    ctx->select_smem = (cap <= SEL_SMEM_KEYS) && (sp.gw * sp.gh <= SEL_SMEM_CELLS);

    // CTriangulator constants (src/core/CTriangulator.cpp:13-21)
    TriConst& tc = ctx->tc;
    const double f = left->P[0];
    tc.f_inv = 1.0 / f;
    tc.pu = left->P[2];
    tc.pv = left->P[6];
    tc.du_r_flipped = -right->P[3];
    tc.min_disp = p.min_disparity_px;
    tc.depth_min = tc.du_r_flipped / (double)left->width;
    tc.depth_max = tc.du_r_flipped / p.min_disparity_px;
    tc.width_left = (float)left->width;
    tc.width_right = (float)right->width;
    tc.match_cutoff = p.match_cutoff;

    CK(cudaFuncSetAttribute(harris_box_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(HarrisSmem)));
    CK(cudaFuncSetAttribute(select_corners_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 13 * SEL_SMEM_KEYS));
    CK(cudaFuncSetAttribute(stereo_match_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, MATCH_SMEM));
    CK(cudaFuncSetAttribute(stereo_match_split_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, MatchSplit<1>::SMEM));
    CK(cudaFuncSetAttribute(stereo_match_split_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, MatchSplit<2>::SMEM));
    CK(cudaFuncSetAttribute(stereo_match_split_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, MatchSplit<2>::SMEM));
    CK(cudaFuncSetAttribute(describe_left_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DL_SMEM));
    CK(cudaFuncSetAttribute(stereo_match_binned_kernel<BinWide>, cudaFuncAttributeMaxDynamicSharedMemorySize, BinWide::M_SMEM));
    CK(cudaFuncSetAttribute(describe_left_binned_kernel<BinWide>, cudaFuncAttributeMaxDynamicSharedMemorySize, BinWide::D_SMEM));
    CK(cudaFuncSetAttribute(triangulate_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, MATCH_SMEM));
    CK(cudaFuncSetAttribute(triangulate_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, MATCH_SMEM));
    CK(cudaFuncSetAttribute(track_stage1_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, MATCH_SMEM));
    CK(cudaFuncSetAttribute(track_stage2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, MATCH_SMEM));
    CK(cudaFuncSetAttribute(track_stage2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, MATCH_SMEM));
    CK(cudaFuncSetAttribute(track_stage3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, MATCH_SMEM));
    CK(cudaFuncSetAttribute(stereo_posit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPositSmemBytes));
    CK(cudaFuncSetAttribute(stereo_posit_count_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPositSmemBytes));
    // one shared-memory carve-out for every kernel of the pipeline: back-to-back kernels with different
    // carve-outs make the SMs drain and reconfigure between launches
    {
        const void* kernels[] = {(const void*)harris_box_kernel, (const void*)boxsum9_kernel,
                                 (const void*)select_corners_kernel<true>, (const void*)select_corners_kernel<false>,
                                 (const void*)stereo_match_kernel, (const void*)stereo_match_split_kernel<1, true>,
                                 (const void*)stereo_match_split_kernel<2, true>, (const void*)stereo_match_split_kernel<2, false>,
                                 (const void*)describe_left_kernel, (const void*)stereo_match_binned_kernel<BinWide>,
                                 (const void*)describe_left_binned_kernel<BinWide>, (const void*)bin_keypoints_kernel,
                                 (const void*)triangulate_kernel<true>,
                                 (const void*)triangulate_kernel<false>, (const void*)track_stage1_kernel,
                                 (const void*)track_stage2_kernel<true>, (const void*)track_stage2_kernel<false>,
                                 (const void*)track_stage3_kernel, (const void*)fast_candidates_kernel,
                                 (const void*)describe_kernel, (const void*)hamming_match_kernel, (const void*)rectify_kernel,
                                 (const void*)band_match_kernel<BM_FRAME>, (const void*)band_match_kernel<BM_EPIPOLAR>,
                                 (const void*)band_match_kernel<BM_REVERSE>, (const void*)gather_rows_kernel};
        for (const void* k : kernels)
            CK(cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    }

    const size_t C = (size_t)ctx->chunk, HH = (size_t)ctx->H, MC = (size_t)p.max_corners;
    for (int i = 0; i < ctx->n_lanes; ++i) {
        Lane& l = ctx->lanes[i];
        CK(cudaStreamCreateWithFlags(&l.stream, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&l.done, cudaEventDisableTiming));
        CK(dmalloc(&l.box_l, C * HH * ctx->box_pitch));
        CK(dmalloc(&l.box_r, C * HH * ctx->box_pitch));
        CK(dmalloc(&l.box_ls, C * HH * ctx->box_pitch));
        CK(dmalloc(&l.box_rs, C * HH * ctx->box_pitch));
        CK(cudaMemset(l.box_ls, 0, sizeof(uint16_t) * C * HH * ctx->box_pitch));
        CK(cudaMemset(l.box_rs, 0, sizeof(uint16_t) * C * HH * ctx->box_pitch));
        {
            std::string merr;
            if (!make_box_map(&l.map_l, l.box_l, ctx->W, (int)(C * HH), ctx->box_pitch, &merr) ||
                !make_box_map(&l.map_ls, l.box_ls, ctx->W, (int)(C * HH), ctx->box_pitch, &merr) ||
                !make_box_map(&l.map_rs, l.box_rs, ctx->W, (int)(C * HH), ctx->box_pitch, &merr) ||
                !make_box_map(&l.map_r, l.box_r, ctx->W, (int)(C * HH), ctx->box_pitch, &merr) ||
                !make_box_map(&l.map_l_patch, l.box_l, ctx->W, (int)(C * HH), ctx->box_pitch, &merr, DL_COLS)) {
                svi_destroy(ctx);
                return fail(nullptr, SVI_ERR_CUDA, merr);
            }
        }
        if (ctx->match_binned) {
            std::string merr;
            CK(dmalloc(&l.bin_start, C * (size_t)(ctx->n_bins + 1)));
            CK(dmalloc(&l.bin_slot, C * MC));
            CK(dmalloc(&l.bin_kp, C * MC));
            if (setup_binned<BinWide>(ctx, l, C * HH, &merr) != SVI_SUCCESS) {
                svi_destroy(ctx);
                return fail(nullptr, SVI_ERR_CUDA, merr);
            }
        }
        CK(dmalloc(&l.frame_max, C));
        CK(dmalloc(&l.cand_count, C));
        CK(dmalloc(&l.cand, C * (size_t)ctx->raw_cap));
        CK(dmalloc(&l.det_xy, C * MC));
        CK(dmalloc(&l.kp_xy, C * MC));
        CK(dmalloc(&l.n_det, C));
        CK(dmalloc(&l.n_kp, C));
        if (!ctx->select_smem) {
            CK(dmalloc(&l.g_head, C * sp.gw * sp.gh));
            CK(dmalloc(&l.g_next, C * cap));
            CK(dmalloc(&l.g_state, C * cap));
        }
        CK(dmalloc(&l.img_l, C * HH * ctx->dev_pitch));
        CK(dmalloc(&l.img_r, C * HH * ctx->dev_pitch));
        CK(dmalloc(&l.mask, C * HH * ctx->dev_pitch));
        l.out.cap = p.max_corners;
        CK(dmalloc(&l.out.uv_l, C * MC * 2));
        CK(dmalloc(&l.out.uv_r, C * MC * 2));
        CK(dmalloc(&l.out.xyz, C * MC * 3));
        CK(dmalloc(&l.out.desc_l, C * MC * 32));
        CK(dmalloc(&l.out.desc_r, C * MC * 32));
        CK(dmalloc(&l.out.dist, C * MC));
        CK(dmalloc(&l.out.idx, C * MC));
        CK(dmalloc(&l.out.status, C * MC));
    }
    {
        int* h = nullptr;
        CK(cudaHostAlloc(reinterpret_cast<void**>(&h), sizeof(int), cudaHostAllocMapped));
        *h = 0;
        ctx->h_overflow = h;
        CK(cudaHostGetDevicePointer(reinterpret_cast<void**>(&ctx->d_overflow), h, 0));
    }
    CK(cudaEventCreateWithFlags(&ctx->fork, cudaEventDisableTiming));
    CK(cudaStreamCreateWithFlags(&ctx->side, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&ctx->side_done, cudaEventDisableTiming));
    CK(dmalloc(&ctx->trk_img, 2 * HH * ctx->dev_pitch));
    // sized so that the per-query and tracking calls of up to max_queries items never grow it (reserve_call)
    ctx->call_bytes = std::min<size_t>(query_bytes(ctx), 64u << 20);
    CK(cudaMalloc(reinterpret_cast<void**>(&ctx->call_dev), ctx->call_bytes));
    CK(cudaMallocHost(reinterpret_cast<void**>(&ctx->call_pin), ctx->call_bytes));
    // room for kSmallFrames frames: three image planes in, every output array out
    ctx->pin_bytes = (size_t)kSmallFrames * (3 * HH * ctx->dev_pitch + (size_t)p.max_corners * kOutBytesPerSlot + 64) + 16;
    if (ctx->pin_bytes <= (64u << 20)) CK(cudaMallocHost(reinterpret_cast<void**>(&ctx->pin), ctx->pin_bytes));
    else ctx->pin_bytes = 0;
    {   // layout (descending alignment): xyz | uv_l | uv_r | dist | idx | n_kp | n_det | desc_l | desc_r | status
        const size_t S = (size_t)kSmallFrames * MC;
        ctx->small_bytes = S * kOutBytesPerSlot + 2 * sizeof(int) * kSmallFrames;
        CK(cudaMalloc(reinterpret_cast<void**>(&ctx->small_block), ctx->small_bytes));
        unsigned char* q = ctx->small_block;
        StereoOutDev& o = ctx->small_out;
        o.cap = p.max_corners;
        o.xyz = reinterpret_cast<double*>(q); q += S * 24;
        o.uv_l = reinterpret_cast<float*>(q); q += S * 8;
        o.uv_r = reinterpret_cast<float*>(q); q += S * 8;
        o.dist = reinterpret_cast<int*>(q); q += S * 4;
        o.idx = reinterpret_cast<int*>(q); q += S * 4;
        ctx->small_n_kp = reinterpret_cast<int*>(q); q += sizeof(int) * kSmallFrames;
        ctx->small_n_det = reinterpret_cast<int*>(q); q += sizeof(int) * kSmallFrames;
        o.desc_l = q; q += S * 32;
        o.desc_r = q; q += S * 32;
        o.status = q;
    }
    *out = ctx;
    return SVI_SUCCESS;
#undef CK
#define CK(call)                                                                                  \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess)                                                                    \
            return fail(ctx, SVI_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));   \
    } while (0)
}

int svi_stereo_frames_device(svi_ctx* ctx, const uint8_t* left, const uint8_t* right, size_t pitch, size_t frame_stride,
                             int n_frames, const uint8_t* masks, const svi_stereo_result* out, void* cuda_stream) {
    if (!ctx) return SVI_ERR_INVALID;
    const int rc = check_frames_args(ctx, "svi_stereo_frames_device", left, right, pitch, frame_stride, n_frames, out, true);
    if (rc != SVI_SUCCESS) return rc;
    CK(cudaSetDevice(ctx->device));
    return device_frames(ctx, left, right, pitch, frame_stride, n_frames, masks, out, cuda_stream,
                         [&](Lane& l, const uint8_t* dl, const uint8_t* dr, const uint8_t* dm, const FrameGeom& g, int f0, int nf,
                             const StereoOutDev& o, int* n_kp, int* n_det) {
                             return run_pipeline(ctx, l, dl, dr, dm, g, nf, o, f0, n_kp, n_det);
                         });
}

int svi_stereo_frames(svi_ctx* ctx, const uint8_t* left, const uint8_t* right, size_t pitch, size_t frame_stride,
                      int n_frames, const uint8_t* masks, svi_stereo_result* out) {
    if (!ctx) return SVI_ERR_INVALID;
    const int rc = check_frames_args(ctx, "svi_stereo_frames", left, right, pitch, frame_stride, n_frames, out, false);
    if (rc != SVI_SUCCESS) return rc;
    CK(cudaSetDevice(ctx->device));
    if (n_frames > 0 && n_frames <= std::min(kSmallFrames, ctx->chunk) && ctx->pin)
        return small_call(ctx, left, right, pitch, frame_stride, n_frames, masks, nullptr, 0, out);
    return host_frames(ctx, left, right, pitch, frame_stride, n_frames, masks, out,
                       [&](Lane& l, const FrameGeom& g, int, int nf) {
                           return run_pipeline(ctx, l, l.img_l, l.img_r, masks ? l.mask : nullptr, g, nf, l.out, 0, l.n_kp, l.n_det);
                       },
                       nullptr);
}

namespace {
int check_sparse_args(svi_ctx* ctx, const char* name, const svi_sparse_band* band, const svi_sparse_result* sparse) {
    if (!band || !sparse) return fail(ctx, SVI_ERR_INVALID, std::string(name) + ": bad argument");
    if (std::isnan(band->band_v) || std::isnan(band->min_disparity) || std::isnan(band->max_disparity) ||
        band->min_disparity > band->max_disparity)
        return fail(ctx, SVI_ERR_INVALID, std::string(name) + ": band fields must not be NaN and min_disparity <= max_disparity");
    if (band->mutual != 0 && band->mutual != 1) return fail(ctx, SVI_ERR_INVALID, std::string(name) + ": band.mutual must be 0 or 1");
    if (!sparse->second_distance || !sparse->n_keypoints_right) return fail(ctx, SVI_ERR_INVALID, std::string(name) + ": null output array");
    const int rc = ensure_sparse_scratch(ctx);
    if (rc != SVI_SUCCESS || !band->mutual) return rc;
    return ensure_mutual_scratch(ctx);
}
}  // namespace

int svi_stereo_frames_sparse(svi_ctx* ctx, const uint8_t* left, const uint8_t* right, size_t pitch, size_t frame_stride, int n_frames,
                             const uint8_t* masks, const svi_sparse_band* band, svi_stereo_result* out, svi_sparse_result* sparse) {
    if (!ctx) return SVI_ERR_INVALID;
    int rc = check_frames_args(ctx, "svi_stereo_frames_sparse", left, right, pitch, frame_stride, n_frames, out, false);
    if (rc != SVI_SUCCESS) return rc;
    CK(cudaSetDevice(ctx->device));
    if ((rc = check_sparse_args(ctx, "svi_stereo_frames_sparse", band, sparse)) != SVI_SUCCESS) return rc;
    const int MC = ctx->p.max_corners, cap = out->capacity_per_frame;
    return host_frames(ctx, left, right, pitch, frame_stride, n_frames, masks, out,
                       [&](Lane& l, const FrameGeom& g, int, int nf) {
                           return run_sparse(ctx, l, l.img_l, l.img_r, masks ? l.mask : nullptr, g, nf, l.out, 0, l.n_kp, l.n_det, l.sp_second,
                                             l.sp_n_kp_r, *band);
                       },
                       [&](Lane& l, const FrameGeom&, int f0, int nf) -> int {
                           CK(d2h_slots(sparse->second_distance, l.sp_second, sizeof(int32_t), MC, cap, f0, nf, l.stream));
                           CK(cudaMemcpyAsync(sparse->n_keypoints_right + f0, l.sp_n_kp_r, sizeof(int) * nf, cudaMemcpyDeviceToHost, l.stream));
                           return SVI_SUCCESS;
                       });
}

int svi_stereo_frames_sparse_device(svi_ctx* ctx, const uint8_t* left, const uint8_t* right, size_t pitch, size_t frame_stride,
                                    int n_frames, const uint8_t* masks, const svi_sparse_band* band, const svi_stereo_result* out,
                                    const svi_sparse_result* sparse, void* cuda_stream) {
    if (!ctx) return SVI_ERR_INVALID;
    int rc = check_frames_args(ctx, "svi_stereo_frames_sparse_device", left, right, pitch, frame_stride, n_frames, out, true);
    if (rc != SVI_SUCCESS) return rc;
    CK(cudaSetDevice(ctx->device));
    if ((rc = check_sparse_args(ctx, "svi_stereo_frames_sparse_device", band, sparse)) != SVI_SUCCESS) return rc;
    return device_frames(ctx, left, right, pitch, frame_stride, n_frames, masks, out, cuda_stream,
                         [&](Lane& l, const uint8_t* dl, const uint8_t* dr, const uint8_t* dm, const FrameGeom& g, int f0, int nf,
                             const StereoOutDev& o, int* n_kp, int* n_det) {
                             return run_sparse(ctx, l, dl, dr, dm, g, nf, o, f0, n_kp, n_det, sparse->second_distance,
                                               sparse->n_keypoints_right + f0, *band);
                         });
}

int svi_mask_active_landmarks(svi_ctx* ctx, const float* centres_xy, int n_centres, uint8_t* mask, size_t pitch) {
    if (!ctx) return SVI_ERR_INVALID;
    if (!mask || n_centres < 0 || (n_centres > 0 && !centres_xy) || (int)pitch < ctx->W)
        return fail(ctx, SVI_ERR_INVALID, "svi_mask_active_landmarks: bad argument");
    if (n_centres > ctx->p.max_queries) return fail(ctx, SVI_ERR_CAPACITY, "svi_mask_active_landmarks: n_centres > max_queries");
    CK(cudaSetDevice(ctx->device));
    Lane& l = ctx->lanes[0];
    SyncOnFailure idle{l.stream};
    int rc = build_mask(ctx, l, centres_xy, n_centres);
    if (rc != SVI_SUCCESS) return rc;
    CK(cudaMemcpy2DAsync(mask, pitch, l.mask, ctx->dev_pitch, ctx->W, ctx->H, cudaMemcpyDeviceToHost, l.stream));
    CK(cudaStreamSynchronize(l.stream));
    idle.done = true;
    return SVI_SUCCESS;
}

int svi_stereo_frame_masked(svi_ctx* ctx, const uint8_t* left, const uint8_t* right, size_t pitch, const float* centres_xy,
                            int n_centres, svi_stereo_result* out) {
    if (!ctx) return SVI_ERR_INVALID;
    if (!left || !right || !out || n_centres < 0 || (n_centres > 0 && !centres_xy) || (int)pitch < ctx->W)
        return fail(ctx, SVI_ERR_INVALID, "svi_stereo_frame_masked: bad argument");
    if (out->capacity_per_frame < ctx->p.max_corners) return fail(ctx, SVI_ERR_CAPACITY, "svi_stereo_frame_masked: capacity_per_frame < max_corners");
    if (!out->n_keypoints || !out->uv_left || !out->uv_right || !out->xyz_left || !out->desc_left || !out->desc_right ||
        !out->distance || !out->match_index || !out->status)
        return fail(ctx, SVI_ERR_INVALID, "svi_stereo_frame_masked: null output array");
    if (n_centres > ctx->p.max_queries) return fail(ctx, SVI_ERR_CAPACITY, "svi_stereo_frame_masked: n_centres > max_queries");
    if (!ctx->pin) return fail(ctx, SVI_ERR_UNSUPPORTED, "svi_stereo_frame_masked: frame too large for the pinned bounce buffer");
    CK(cudaSetDevice(ctx->device));
    static const float kNone[2] = {-1.0e9f, -1.0e9f};   // no landmark yet: an all-255 mask
    return small_call(ctx, left, right, pitch, pitch * (size_t)ctx->H, 1, nullptr, n_centres > 0 ? centres_xy : kNone,
                      n_centres > 0 ? n_centres : 1, out);
}

int svi_harris_response(svi_ctx* ctx, const uint8_t* img, size_t pitch, float* response) {
    if (!ctx) return SVI_ERR_INVALID;
    if (!img || !response || (int)pitch < ctx->W) return fail(ctx, SVI_ERR_INVALID, "svi_harris_response: bad argument");
    CK(cudaSetDevice(ctx->device));
    Lane& l = ctx->lanes[0];
    cudaStream_t s = l.stream;
    const FrameGeom g = make_geom(ctx, ctx->dev_pitch, (size_t)ctx->H * ctx->dev_pitch);
    CK(cudaMemcpy2DAsync(ctx->rect ? l.raw_l : l.img_l, ctx->dev_pitch, img, pitch, ctx->W, ctx->H, cudaMemcpyHostToDevice, s));
    if (ctx->rect) {
        const int rc = rectify_one(ctx, 0, l.raw_l, ctx->dev_pitch, (size_t)ctx->H * ctx->dev_pitch, l.img_l, 1, s);
        if (rc != SVI_SUCCESS) return rc;
    }
    CK(cudaMemsetAsync(l.frame_max, 0, sizeof(uint32_t), s));
    if (!ctx->resp_one) CK(dmalloc(&ctx->resp_one, (size_t)ctx->H * ctx->resp_pitch));
    harris_box_kernel<<<harris_grid(g.W, g.H, 1), HT_THREADS, sizeof(HarrisSmem), s>>>(
        l.img_l, nullptr, g, ctx->f1, ctx->f0, ctx->p.harris_k, ctx->p.quality_level, ctx->resp_one, nullptr, nullptr, l.frame_max, nullptr,
        nullptr, 0, nullptr, nullptr, g.H);
    CK(cudaGetLastError());
    CK(cudaMemcpy2DAsync(response, sizeof(float) * ctx->W, ctx->resp_one, sizeof(float) * ctx->resp_pitch, sizeof(float) * ctx->W,
                         ctx->H, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return SVI_SUCCESS;
}

int svi_detect(svi_ctx* ctx, const uint8_t* img, size_t pitch, size_t frame_stride, int n_frames, const uint8_t* masks,
               float* xy, int32_t* counts) {
    if (!ctx) return SVI_ERR_INVALID;
    if (!img || !xy || !counts || n_frames < 0 || (int)pitch < ctx->W) return fail(ctx, SVI_ERR_INVALID, "svi_detect: bad argument");
    CK(cudaSetDevice(ctx->device));
    Lane& l = ctx->lanes[0];
    cudaStream_t s = l.stream;
    const int W = ctx->W, H = ctx->H, MC = ctx->p.max_corners;
    const size_t dstride = (size_t)H * ctx->dev_pitch;
    const FrameGeom g = make_geom(ctx, ctx->dev_pitch, dstride);
    std::vector<ushort2> h_xy((size_t)ctx->chunk * MC);
    for (int f0 = 0; f0 < n_frames; f0 += ctx->chunk) {
        const int nf = std::min(ctx->chunk, n_frames - f0);
        for (int f = 0; f < nf; ++f) {
            CK(cudaMemcpy2DAsync((ctx->rect ? l.raw_l : l.img_l) + f * dstride, ctx->dev_pitch, img + (size_t)(f0 + f) * frame_stride, pitch, W, H,
                                 cudaMemcpyHostToDevice, s));
            if (masks)
                CK(cudaMemcpy2DAsync(l.mask + f * dstride, ctx->dev_pitch, masks + (size_t)(f0 + f) * frame_stride, pitch, W, H,
                                     cudaMemcpyHostToDevice, s));
        }
        if (ctx->rect) {
            const int rc = rectify_one(ctx, 0, l.raw_l, ctx->dev_pitch, dstride, l.img_l, nf, s);
            if (rc != SVI_SUCCESS) return rc;
        }
        const uint8_t* d_mask = masks ? l.mask : nullptr;
        CK(cudaMemsetAsync(l.frame_max, 0, sizeof(uint32_t) * nf, s));
        CK(cudaMemsetAsync(l.cand_count, 0, sizeof(int) * nf, s));
        const dim3 tiles((W + HT_W - 1) / HT_W, (H + HT_H - 1) / HT_H, nf);
        const bool fast = ctx->p.detector == SVI_DETECTOR_FAST_9_16;
        if (fast) {
            fast_candidates_kernel<<<tiles, HT_THREADS, 0, s>>>(l.img_l, d_mask, g, ctx->p.fast_threshold, ctx->p.fast_nonmax, l.cand,
                                                                l.cand_count, ctx->raw_cap);
        } else {
            harris_box_kernel<<<harris_grid(W, H, nf), HT_THREADS, sizeof(HarrisSmem), s>>>(
                l.img_l, d_mask, g, ctx->f1, ctx->f0, ctx->p.harris_k, ctx->p.quality_level, nullptr, nullptr, nullptr, l.frame_max, l.cand,
                l.cand_count, ctx->raw_cap, nullptr, nullptr, g.H);
        }
        const uint32_t* fmax = fast ? nullptr : l.frame_max;
        if (ctx->select_smem)
            select_corners_kernel<true><<<nf, SEL_THREADS, 13 * SEL_SMEM_KEYS, s>>>(l.cand, l.cand_count, fmax, ctx->sel, nullptr, nullptr,
                                                                                  nullptr, l.det_xy, l.n_det, l.kp_xy, l.n_kp,
                                                                                  ctx->d_overflow, nullptr);
        else
            select_corners_kernel<false><<<nf, SEL_THREADS, 4 * SEL_SMEM_CELLS, s>>>(l.cand, l.cand_count, fmax, ctx->sel, l.g_head, l.g_next, l.g_state,
                                                                   l.det_xy, l.n_det, l.kp_xy, l.n_kp, ctx->d_overflow, nullptr);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(h_xy.data(), l.det_xy, sizeof(ushort2) * (size_t)nf * MC, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(counts + f0, l.n_det, sizeof(int) * nf, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        for (int f = 0; f < nf; ++f)
            for (int i = 0; i < counts[f0 + f]; ++i) {
                xy[((size_t)(f0 + f) * MC + i) * 2] = (float)h_xy[(size_t)f * MC + i].x;
                xy[((size_t)(f0 + f) * MC + i) * 2 + 1] = (float)h_xy[(size_t)f * MC + i].y;
            }
    }
    return check_overflow(ctx);
}

int svi_describe(svi_ctx* ctx, const uint8_t* img, size_t pitch, const float* xy, int n, uint8_t* desc32, uint8_t* kept) {
    if (!ctx) return SVI_ERR_INVALID;
    if (!img || !xy || !desc32 || !kept || n < 0 || (int)pitch < ctx->W) return fail(ctx, SVI_ERR_INVALID, "svi_describe: bad argument");
    if (n > ctx->p.max_queries) return fail(ctx, SVI_ERR_CAPACITY, "svi_describe: n > max_queries");
    if (n == 0) return SVI_SUCCESS;
    CK(cudaSetDevice(ctx->device));
    Lane& l = ctx->lanes[0];
    cudaStream_t s = l.stream;
    SyncOnFailure idle{s};
    const size_t N = (size_t)n;
    CallLayout L;   // [xy] -> [desc | kept]
    const size_t i_xy = L.take(8 * N), o_desc = L.take(32 * N), o_kept = L.take(N);
    if (const int rc = reserve_call(ctx, L.end)) return rc;
    int rc = stage_box(ctx, img, pitch, l.img_l, l.box_l, l.box_ls, s, 0);
    if (rc != SVI_SUCCESS) return rc;
    put(ctx, i_xy, xy, 8 * N);
    if ((rc = call_send(ctx, o_desc, s)) != SVI_SUCCESS) return rc;
    const FrameGeom g = make_geom(ctx, ctx->dev_pitch, (size_t)ctx->H * ctx->dev_pitch);
    describe_kernel<<<(n + 3) / 4, 128, 0, s>>>(l.box_l, g, dev_at<float>(ctx, i_xy), n, dev_at(ctx, o_desc), dev_at(ctx, o_kept));
    CK(cudaGetLastError());
    if ((rc = call_fetch(ctx, o_desc, L.end, s)) != SVI_SUCCESS) return rc;
    idle.done = true;
    std::memcpy(desc32, ctx->call_pin + o_desc, 32 * N);
    std::memcpy(kept, ctx->call_pin + o_kept, N);
    return SVI_SUCCESS;
}

int svi_match_hamming(svi_ctx* ctx, const uint8_t* query32, int n_query, const uint8_t* train32, int n_train, int32_t* index,
                      int32_t* distance) {
    if (!ctx) return SVI_ERR_INVALID;
    if (!query32 || !index || !distance || n_query < 0 || n_train < 0 || (n_train > 0 && !train32))
        return fail(ctx, SVI_ERR_INVALID, "svi_match_hamming: bad argument");
    if ((size_t)(n_query + n_train) * 40 > query_bytes(ctx)) return fail(ctx, SVI_ERR_CAPACITY, "svi_match_hamming: raise max_queries");
    if (n_query == 0) return SVI_SUCCESS;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->lanes[0].stream;
    SyncOnFailure idle{s};
    const size_t Q = (size_t)n_query, T = (size_t)std::max(n_train, 1);
    CallLayout L;   // [query | train] -> [index | distance]
    const size_t i_q = L.take(32 * Q), i_t = L.take(32 * T), o_i = L.take(4 * Q), o_d = L.take(4 * Q);
    if (const int rc = reserve_call(ctx, L.end)) return rc;
    put(ctx, i_q, query32, 32 * Q);
    put(ctx, i_t, n_train > 0 ? train32 : nullptr, 32 * T);
    int rc = call_send(ctx, o_i, s);
    if (rc != SVI_SUCCESS) return rc;
    hamming_match_kernel<<<(n_query + 3) / 4, 128, 0, s>>>(dev_at(ctx, i_q), n_query, dev_at(ctx, i_t), n_train, dev_at<int>(ctx, o_i), dev_at<int>(ctx, o_d));
    CK(cudaGetLastError());
    if ((rc = call_fetch(ctx, o_i, L.end, s)) != SVI_SUCCESS) return rc;
    idle.done = true;
    std::memcpy(index, ctx->call_pin + o_i, 4 * Q);
    std::memcpy(distance, ctx->call_pin + o_d, 4 * Q);
    return SVI_SUCCESS;
}

int svi_match_epipolar(svi_ctx* ctx, const uint8_t* query32, const float* query_xy, int n_query, const uint8_t* train32,
                       const float* train_xy, int n_train, float band_v, float min_disparity, float max_disparity,
                       int32_t* index, int32_t* distance, int32_t* second_distance) {
    if (!ctx) return SVI_ERR_INVALID;
    if (!query32 || !query_xy || !index || !distance || !second_distance || n_query < 0 || n_train < 0 ||
        (n_train > 0 && (!train32 || !train_xy)))
        return fail(ctx, SVI_ERR_INVALID, "svi_match_epipolar: bad argument");
    if ((size_t)(n_query + n_train) * 48 + (size_t)n_query * 16 > query_bytes(ctx))
        return fail(ctx, SVI_ERR_CAPACITY, "svi_match_epipolar: raise max_queries");
    if (n_query == 0) return SVI_SUCCESS;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->lanes[0].stream;
    SyncOnFailure idle{s};
    const size_t Q = (size_t)n_query, T = (size_t)std::max(n_train, 1);
    CallLayout L;   // [query | query_xy | train | train_xy] -> [index | distance | second_distance]
    const size_t i_q = L.take(32 * Q), i_qxy = L.take(8 * Q), i_t = L.take(32 * T), i_txy = L.take(8 * T);
    const size_t o_i = L.take(4 * Q), o_d = L.take(4 * Q), o_s = L.take(4 * Q);
    if (const int rc = reserve_call(ctx, L.end)) return rc;
    put(ctx, i_q, query32, 32 * Q);
    put(ctx, i_qxy, query_xy, 8 * Q);
    put(ctx, i_t, n_train > 0 ? train32 : nullptr, 32 * T);
    put(ctx, i_txy, n_train > 0 ? train_xy : nullptr, 8 * T);
    int rc = call_send(ctx, o_i, s);
    if (rc != SVI_SUCCESS) return rc;
    // the trains in caller order as one range (band_match_kernel reads up to BM_ALIGN - 1 elements past each array: the
    // call buffer's 256-byte alignment of every region covers them)
    BandArgs a{};
    a.band_v = band_v; a.min_disp = min_disparity; a.max_disp = max_disparity;
    a.q_desc = dev_at(ctx, i_q); a.q_xy = dev_at<float2>(ctx, i_qxy); a.nq = n_query;
    a.t_desc = dev_at(ctx, i_t); a.t_xy = dev_at<float2>(ctx, i_txy); a.nt = n_train;
    a.index = dev_at<int>(ctx, o_i); a.distance = dev_at<int>(ctx, o_d); a.second = dev_at<int>(ctx, o_s);
    band_match_kernel<BM_EPIPOLAR><<<(n_query + BM_THREADS - 1) / BM_THREADS, BM_THREADS, BandTile<false>::SMEM, s>>>(a);
    CK(cudaGetLastError());
    if ((rc = call_fetch(ctx, o_i, L.end, s)) != SVI_SUCCESS) return rc;
    idle.done = true;
    std::memcpy(index, ctx->call_pin + o_i, 4 * Q);
    std::memcpy(distance, ctx->call_pin + o_d, 4 * Q);
    std::memcpy(second_distance, ctx->call_pin + o_s, 4 * Q);
    return SVI_SUCCESS;
}

int svi_triangulate_right(svi_ctx* ctx, const uint8_t* img_right, size_t pitch, int n, const float* top_left,
                          const float* uv_left, const uint8_t* desc_left, float keypoint_size, svi_tri_result* out) {
    if (!ctx) return SVI_ERR_INVALID;
    return triangulate_common(ctx, false, img_right, pitch, n, nullptr, top_left, uv_left, desc_left, keypoint_size, out);
}

int svi_triangulate_left(svi_ctx* ctx, const uint8_t* img_left, size_t pitch, int n, const float* search_range,
                         const float* top_left, const float* uv_right, const uint8_t* desc_right, float keypoint_size,
                         svi_tri_result* out) {
    if (!ctx) return SVI_ERR_INVALID;
    return triangulate_common(ctx, true, img_left, pitch, n, search_range, top_left, uv_right, desc_right, keypoint_size, out);
}

int svi_point_in_left(svi_ctx* ctx, int n, const float* uv_left, const float* uv_right, double* xyz_left, uint8_t* status) {
    if (!ctx) return SVI_ERR_INVALID;
    if (!uv_left || !uv_right || !xyz_left || !status || n < 0) return fail(ctx, SVI_ERR_INVALID, "svi_point_in_left: bad argument");
    if (n > ctx->p.max_queries) return fail(ctx, SVI_ERR_CAPACITY, "svi_point_in_left: n > max_queries");
    if (n == 0) return SVI_SUCCESS;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->lanes[0].stream;
    SyncOnFailure idle{s};
    const size_t N = (size_t)n;
    CallLayout L;   // [uv_left | uv_right] -> [xyz | status]
    const size_t i_l = L.take(8 * N), i_r = L.take(8 * N), o_xyz = L.take(24 * N), o_st = L.take(N);
    if (const int rc = reserve_call(ctx, L.end)) return rc;
    put(ctx, i_l, uv_left, 8 * N);
    put(ctx, i_r, uv_right, 8 * N);
    int rc = call_send(ctx, o_xyz, s);
    if (rc != SVI_SUCCESS) return rc;
    point_in_left_kernel<<<(n + 127) / 128, 128, 0, s>>>(ctx->tc, n, dev_at<float>(ctx, i_l), dev_at<float>(ctx, i_r), dev_at<double>(ctx, o_xyz), dev_at(ctx, o_st));
    CK(cudaGetLastError());
    if ((rc = call_fetch(ctx, o_xyz, L.end, s)) != SVI_SUCCESS) return rc;
    idle.done = true;
    std::memcpy(xyz_left, ctx->call_pin + o_xyz, 24 * N);
    std::memcpy(status, ctx->call_pin + o_st, N);
    return SVI_SUCCESS;
}

int svi_track_landmarks(svi_ctx* ctx, const uint8_t* img_left, const uint8_t* img_right, size_t pitch,
                        const double* T_world_to_left, const svi_landmarks* lm, int n, double motion_scaling,
                        svi_track_result* out) {
    if (!ctx) return SVI_ERR_INVALID;
    if (!lm) return fail(ctx, SVI_ERR_INVALID, "svi_track_landmarks: bad argument");
    const bool any3 = lm->uv_reference_left || lm->desc_reference_left || lm->T_left_to_world_at_detection;
    return svi_track_landmarks_stages(ctx, img_left, img_right, pitch, T_world_to_left, lm, n, motion_scaling,
                                      SVI_STAGE_1 | SVI_STAGE_2 | (any3 ? SVI_STAGE_3 : 0), out);
}

int svi_track_landmarks_stages(svi_ctx* ctx, const uint8_t* img_left, const uint8_t* img_right, size_t pitch,
                               const double* T_world_to_left, const svi_landmarks* lm, int n, double motion_scaling,
                               uint32_t stage_mask, svi_track_result* out) {
    if (!ctx) return SVI_ERR_INVALID;
    if (!img_left || !img_right || !T_world_to_left || !lm || !out || n < 0 || (int)pitch < ctx->W ||
        !(stage_mask & (SVI_STAGE_1 | SVI_STAGE_2 | SVI_STAGE_3)) || (stage_mask & ~(uint32_t)(SVI_STAGE_1 | SVI_STAGE_2 | SVI_STAGE_3)))
        return fail(ctx, SVI_ERR_INVALID, "svi_track_landmarks: bad argument");
    if (!lm->xyz_world || !lm->last_desc_left || !lm->last_desc_right || !lm->last_disparity || !lm->keypoint_size ||
        !out->status || !out->stage || !out->uv_left || !out->uv_right || !out->xyz_left || !out->desc_left || !out->desc_right)
        return fail(ctx, SVI_ERR_INVALID, "svi_track_landmarks: null array");
    if (n > ctx->p.max_queries) return fail(ctx, SVI_ERR_CAPACITY, "svi_track_landmarks: n > max_queries");
    // the reference computes the scaling as min(1 + ..., 5) (CTrackerGT.cpp:157) and asserts it positive; the search
    // windows grow with it, so an absurd value is rejected here instead of producing image-sized windows
    if (!(motion_scaling >= 0.0 && motion_scaling <= 16.0))
        return fail(ctx, SVI_ERR_INVALID, "svi_track_landmarks: motion_scaling must be within [0, 16]");
    const bool stage3 = (stage_mask & SVI_STAGE_3) != 0;
    if (stage3 && !(lm->uv_reference_left && lm->desc_reference_left && lm->T_left_to_world_at_detection))
        return fail(ctx, SVI_ERR_INVALID, "svi_track_landmarks: stage 3 needs all three reference arrays");
    if (n == 0) return SVI_SUCCESS;
    CK(cudaSetDevice(ctx->device));
    int rc = ensure_track_scratch(ctx);
    if (rc != SVI_SUCCESS) return rc;
    cudaStream_t s = ctx->lanes[0].stream;
    SyncOnFailure idle{s};
    // every input array goes up in ONE copy; the outputs form one contiguous range behind them: one memset, one copy back
    CallLayout L;
    const LandmarkLayout li(L, (size_t)n, stage3);
    const size_t in_end = L.end;
    const TrackLayout lo(L, (size_t)n);
    if ((rc = reserve_call(ctx, L.end)) != SVI_SUCCESS) return rc;
    using clk = std::chrono::steady_clock;
    clk::time_point tp[6];
    auto tick = [&](int i) { if (ctx->trace) tp[i] = clk::now(); };
    tick(0);
    rc = stage_track_pair(ctx, img_left, img_right, pitch);
    if (rc != SVI_SUCCESS) return rc;
    li.put_all(ctx, *lm, (size_t)n);
    tick(1);
    if ((rc = call_send(ctx, in_end, s)) != SVI_SUCCESS) return rc;
    CK(cudaMemsetAsync(ctx->call_dev + lo.status, 0, lo.end - lo.status, s));
    // The whole cascade is ONE stream of kernels; the host only waits once, for the results.
    rc = enqueue_cascade(ctx, n, T_world_to_left, motion_scaling, stage_mask, li.ld(ctx), li.ex(ctx), li.sv(ctx).desc_ref, lo.dev(ctx), nullptr);
    if (rc != SVI_SUCCESS) return rc;
    tick(2);
    if ((rc = call_fetch(ctx, lo.status, lo.end, s)) != SVI_SUCCESS) return rc;
    idle.done = true;
    tick(3);
    lo.copy_out(ctx, (size_t)n, *out);
    tick(4);
    const int rd = check_overflow(ctx);
    tick(5);
    if (ctx->trace) {
        auto us = [&](int a, int b) { return std::chrono::duration<double, std::micro>(tp[b] - tp[a]).count(); };
        std::fprintf(stderr, "svi_track_landmarks n=%d: stage images + mirror inputs %.0f us | enqueue cascade %.0f us | wait %.0f us | "
                             "scatter outputs %.0f us | overflow check %.0f us | total %.0f us\n",
                     n, us(0, 1), us(1, 2), us(2, 3), us(3, 4), us(4, 5), us(0, 5));
    }
    return rd;
}

int svi_optimize_landmarks(svi_ctx* ctx, const svi_landmark_measurements* in, int n, svi_optimize_result* out) {
    if (!ctx) return SVI_ERR_INVALID;
    if (!in || !out || n < 0 || !out->xyz_world || !out->outcome || !out->average_squared_error)
        return fail(ctx, SVI_ERR_INVALID, "svi_optimize_landmarks: bad argument");
    if (n == 0) return SVI_SUCCESS;
    if (!in->xyz_world_guess || !in->first || in->n_poses < 0) return fail(ctx, SVI_ERR_INVALID, "svi_optimize_landmarks: null array");
    const int m = in->first[n];
    if (in->first[0] != 0 || m < 0) return fail(ctx, SVI_ERR_INVALID, "svi_optimize_landmarks: first[] must start at 0 and end at the measurement count");
    for (int i = 0; i < n; ++i)
        if (in->first[i + 1] < in->first[i]) return fail(ctx, SVI_ERR_INVALID, "svi_optimize_landmarks: first[] must not decrease");
    if (m > 0 && (!in->pose_index || !in->uv_left || !in->uv_right || !in->proj_world_to_left || !in->proj_world_to_right || in->n_poses == 0))
        return fail(ctx, SVI_ERR_INVALID, "svi_optimize_landmarks: null measurement array");
    for (int k = 0; k < m; ++k)
        if (in->pose_index[k] < 0 || in->pose_index[k] >= in->n_poses) return fail(ctx, SVI_ERR_INVALID, "svi_optimize_landmarks: pose_index out of range");
    CK(cudaSetDevice(ctx->device));
    using clk = std::chrono::steady_clock;
    const clk::time_point t_begin = clk::now();
    cudaStream_t s = ctx->lanes[0].stream;
    SyncOnFailure idle{s};
    const size_t P = (size_t)in->n_poses;
    CallLayout L;   // [xyz_guess | proj_left | proj_right | first | pose_index | uv_left | uv_right] -> [xyz | avg | iterations | outcome]
    const size_t o_guess = L.take(sizeof(double) * 3 * n), o_pl = L.take(sizeof(double) * 12 * P), o_pr = L.take(sizeof(double) * 12 * P);
    const size_t o_first = L.take(sizeof(int) * ((size_t)n + 1)), o_pose = L.take(sizeof(int) * (size_t)m);
    const size_t o_uvl = L.take(sizeof(float) * 2 * (size_t)m), o_uvr = L.take(sizeof(float) * 2 * (size_t)m);
    const size_t o_xyz = L.take(sizeof(double) * 3 * n), o_avg = L.take(sizeof(double) * n), o_it = L.take(sizeof(int) * (size_t)n), o_out = L.take((size_t)n);
    if (const int rc = reserve_call(ctx, L.end)) return rc;
    put(ctx, o_guess, in->xyz_world_guess, sizeof(double) * 3 * n);
    put(ctx, o_first, in->first, sizeof(int) * ((size_t)n + 1));
    if (m > 0) {
        put(ctx, o_pl, in->proj_world_to_left, sizeof(double) * 12 * P);
        put(ctx, o_pr, in->proj_world_to_right, sizeof(double) * 12 * P);
        put(ctx, o_pose, in->pose_index, sizeof(int) * (size_t)m);
        put(ctx, o_uvl, in->uv_left, sizeof(float) * 2 * (size_t)m);
        put(ctx, o_uvr, in->uv_right, sizeof(float) * 2 * (size_t)m);
    }
    const clk::time_point t_staged = clk::now();
    int rc = call_send(ctx, o_xyz, s);
    if (rc != SVI_SUCCESS) return rc;
    LandmarkOptIn li{dev_at<const double>(ctx, o_guess), dev_at<const int>(ctx, o_first), dev_at<const int>(ctx, o_pose), dev_at<const float>(ctx, o_uvl),
                     dev_at<const float>(ctx, o_uvr), dev_at<const double>(ctx, o_pl), dev_at<const double>(ctx, o_pr), in->n_poses};
    LandmarkOptOut lo{dev_at<double>(ctx, o_xyz), dev_at(ctx, o_out), dev_at<double>(ctx, o_avg), dev_at<int>(ctx, o_it)};
    optimize_landmarks_kernel<<<(n + kOptWarps - 1) / kOptWarps, kOptWarps * 32, 0, s>>>(li, n, lo);
    CK(cudaGetLastError());
    if ((rc = call_fetch(ctx, o_xyz, L.end, s)) != SVI_SUCCESS) return rc;
    idle.done = true;
    const unsigned char* hp = ctx->call_pin;
    std::memcpy(out->xyz_world, hp + o_xyz, sizeof(double) * 3 * n);
    std::memcpy(out->average_squared_error, hp + o_avg, sizeof(double) * n);
    std::memcpy(out->outcome, hp + o_out, (size_t)n);
    if (out->iterations) std::memcpy(out->iterations, hp + o_it, sizeof(int) * (size_t)n);
    if (const char* dump = std::getenv("SVI_OPT_DUMP")) {   // diagnostics: the landmark with the most iterations, in facade_demo --landmark format
        const int* it = reinterpret_cast<const int*>(hp + o_it);
        int worst = 0;
        for (int i = 1; i < n; ++i) if (it[i] > it[worst]) worst = i;
        if (std::FILE* f = std::fopen(dump, "w")) {
            std::fprintf(f, "%.17g %.17g %.17g\n", in->xyz_world_guess[3 * worst], in->xyz_world_guess[3 * worst + 1], in->xyz_world_guess[3 * worst + 2]);
            for (int k = in->first[worst]; k < in->first[worst + 1]; ++k) {
                for (int q = 0; q < 12; ++q) std::fprintf(f, "%.17g ", in->proj_world_to_left[12 * (size_t)in->pose_index[k] + q]);
                for (int q = 0; q < 12; ++q) std::fprintf(f, "%.17g ", in->proj_world_to_right[12 * (size_t)in->pose_index[k] + q]);
                std::fprintf(f, "%.9g %.9g %.9g %.9g\n", in->uv_left[2 * k], in->uv_left[2 * k + 1], in->uv_right[2 * k], in->uv_right[2 * k + 1]);
            }
            std::fprintf(f, "# iterations %d outcome %d\n", it[worst], (int)hp[o_out + worst]);
            std::fclose(f);
        }
    }
    if (ctx->trace) {
        const clk::time_point t_end = clk::now();
        auto us = [](clk::time_point a, clk::time_point b) { return std::chrono::duration<double, std::micro>(b - a).count(); };
        std::fprintf(stderr, "svi_optimize_landmarks n=%d m=%d poses=%d: check + stage inputs %.0f us | copy up, kernel, copy back %.0f us | total %.0f us\n",
                     n, m, in->n_poses, us(t_begin, t_staged), us(t_staged, t_end), us(t_begin, t_end));
    }
    return check_overflow(ctx);
}

int svi_solve_stereo_posit(svi_ctx* ctx, const svi_posit_problem* in, svi_posit_result* out) {
    if (!ctx) return SVI_ERR_INVALID;
    if (!in || !out || in->n < 0) return fail(ctx, SVI_ERR_INVALID, "svi_solve_stereo_posit: bad argument");
    const int n = in->n;
    if (n > 0 && (!in->xyz_world || !in->uv_left || !in->uv_right)) return fail(ctx, SVI_ERR_INVALID, "svi_solve_stereo_posit: null array");
    if (n <= kPositMinimumPoints) {   // !(m_uMinimumPointsForPoseOptimization < uNumberOfMeasurements): fails before any iteration
        posit_too_few(in->T_estimate, out);
        return SVI_SUCCESS;
    }
    CK(cudaSetDevice(ctx->device));
    using clk = std::chrono::steady_clock;
    const clk::time_point t_begin = clk::now();
    cudaStream_t s = ctx->lanes[0].stream;
    SyncOnFailure idle{s};
    const size_t N = (size_t)n;
    CallLayout L;   // [xyz | uv_left | uv_right] -> [PositOut]
    const size_t o_xyz = L.take(24 * N), o_uvl = L.take(8 * N), o_uvr = L.take(8 * N), o_out = L.take(sizeof(PositOut));
    if (const int rc = reserve_call(ctx, L.end)) return rc;
    put(ctx, o_xyz, in->xyz_world, 24 * N);
    put(ctx, o_uvl, in->uv_left, 8 * N);
    put(ctx, o_uvr, in->uv_right, 8 * N);
    const PositIn pi = posit_in(ctx, dev_at<double>(ctx, o_xyz), dev_at<float>(ctx, o_uvl), dev_at<float>(ctx, o_uvr), in->T_estimate, in->T_last, in->t_imu);
    const clk::time_point t_staged = clk::now();
    int rc = call_send(ctx, o_out, s);
    if (rc != SVI_SUCCESS) return rc;
    stereo_posit_kernel<<<1, kPositThreads, kPositSmemBytes, s>>>(pi, n, dev_at<PositOut>(ctx, o_out));
    CK(cudaGetLastError());
    if ((rc = call_fetch(ctx, o_out, L.end, s)) != SVI_SUCCESS) return rc;
    idle.done = true;
    PositOut po;
    std::memcpy(&po, ctx->call_pin + o_out, sizeof(po));
    posit_result_from(po, out);
    if (ctx->trace) {
        const clk::time_point t_end = clk::now();
        auto us = [](clk::time_point a, clk::time_point b) { return std::chrono::duration<double, std::micro>(b - a).count(); };
        std::fprintf(stderr, "svi_solve_stereo_posit n=%d: outcome %d after %d iterations | check + stage inputs %.0f us | copy up, kernel, copy back %.0f us | total %.0f us\n",
                     n, po.outcome, po.iterations, us(t_begin, t_staged), us(t_staged, t_end), us(t_begin, t_end));
    }
    return check_overflow(ctx);
}

namespace {
bool track_result_ok(const svi_track_result& r) {
    return r.status && r.stage && r.uv_left && r.uv_right && r.xyz_left && r.desc_left && r.desc_right;
}
}  // namespace

int svi_track_frame_stereo_only(svi_ctx* ctx, const uint8_t* img_left, const uint8_t* img_right, size_t pitch, const svi_sv_frame* in, int n,
                                svi_sv_frame_result* out) {
    if (!ctx) return SVI_ERR_INVALID;
    if (!img_left || !img_right || !in || !out || n < 0 || (int)pitch < ctx->W) return fail(ctx, SVI_ERR_INVALID, "svi_track_frame_stereo_only: bad argument");
    const svi_landmarks& lm = in->landmarks;
    if (n > 0 && (!lm.xyz_world || !lm.last_desc_left || !lm.last_desc_right || !lm.last_disparity || !lm.keypoint_size || !lm.uv_reference_left ||
                  !lm.desc_reference_left || !lm.T_left_to_world_at_detection || !in->flags || !out->route || !track_result_ok(out->pose_stage) ||
                  !track_result_ok(out->epipolar_stage)))
        return fail(ctx, SVI_ERR_INVALID, "svi_track_frame_stereo_only: null array");
    if (n > ctx->p.max_queries) return fail(ctx, SVI_ERR_CAPACITY, "svi_track_frame_stereo_only: n > max_queries");
    if (!(in->motion_scaling >= 0.0 && in->motion_scaling <= 16.0))
        return fail(ctx, SVI_ERR_INVALID, "svi_track_frame_stereo_only: motion_scaling must be within [0, 16]");
    int n_cand = 0;
    for (int i = 0; i < n; ++i) {
        if (in->flags[i] & ~(SVI_SV_POSE_CANDIDATE | SVI_SV_LEAVES)) return fail(ctx, SVI_ERR_INVALID, "svi_track_frame_stereo_only: unknown flag bits");
        n_cand += in->flags[i] & SVI_SV_POSE_CANDIDATE;
    }
    if (n == 0) {   // no landmark: no hit, both solves fail before an iteration, the pose is the damped prior
        posit_too_few(in->T_estimate, &out->attempt[0]);
        posit_too_few(in->T_estimate_damped, &out->attempt[1]);
        out->measurements[0] = out->measurements[1] = 0;
        out->attempts = 2;
        out->source = SVI_SV_PRIOR;
        std::memcpy(out->T_world_to_left, in->T_estimate_damped, sizeof(out->T_world_to_left));
        return SVI_SUCCESS;
    }
    CK(cudaSetDevice(ctx->device));
    int rc = ensure_track_scratch(ctx);
    if (rc != SVI_SUCCESS) return rc;
    cudaStream_t s = ctx->lanes[0].stream;
    SyncOnFailure idle{s};
    // The call buffer:
    //   [inputs: the landmark arrays and flags]            one copy up
    //   [outputs: attempts, pose stage, route, epipolar]   one memset, one copy down
    //   [scratch: counts, index lists, gathered subset, subset results, pose problem]
    const size_t N = (size_t)n;
    CallLayout L;
    const LandmarkLayout i_lm(L, N, true);
    const size_t i_flags = L.take(N);
    const size_t in_end = L.end;
    const size_t o_posit = L.take(2 * sizeof(PositOut));
    const TrackLayout o_pose(L, N);
    const size_t o_route = L.take(N);
    const TrackLayout o_epi(L, N);
    const size_t out_end = L.end;
    // counts: [0] candidates, [1] pose hits, [2] epipolar set, [3] regional set
    const size_t x_cnt = L.take(4 * sizeof(int)), x_cand = L.take(4 * N), x_hits = L.take(4 * N), x_epi = L.take(4 * N), x_reg = L.take(4 * N);
    const LandmarkLayout x_lm(L, N, true);
    const TrackLayout x_sub(L, N);
    const size_t x_pxyz = L.take(24 * N), x_puvl = L.take(8 * N), x_puvr = L.take(8 * N);
    if ((rc = reserve_call(ctx, L.end)) != SVI_SUCCESS) return rc;
    rc = stage_track_pair(ctx, img_left, img_right, pitch);
    if (rc != SVI_SUCCESS) return rc;
    unsigned char* hp = ctx->call_pin;
    i_lm.put_all(ctx, lm, N);
    put(ctx, i_flags, in->flags, N);
    if ((rc = call_send(ctx, in_end, s)) != SVI_SUCCESS) return rc;
    CK(cudaMemsetAsync(ctx->call_dev + o_posit, 0, out_end - o_posit, s));
    auto dp = [ctx](size_t o) { return dev_at(ctx, o); };
    auto di = [ctx](size_t o) { return dev_at<int>(ctx, o); };
    const SvLandmarksDev all = i_lm.sv(ctx), sub = x_lm.sv(ctx);
    const TrackOutDev pose_out = o_pose.dev(ctx), epi_out = o_epi.dev(ctx), sub_out = x_sub.dev(ctx);
    int* cnt = di(x_cnt);
    PositOut* posit_dev = dev_at<PositOut>(ctx, o_posit);
    uint8_t* route = dp(o_route);
    const unsigned blocks = (unsigned)((n + 127) / 128);
    // the subset results start as a fresh tracking call's outputs: zero
    auto clear_sub = [&]() -> int {
        CK(cudaMemsetAsync(ctx->call_dev + x_sub.status, 0, x_sub.end - x_sub.status, s));
        return SVI_SUCCESS;
    };

    // ---- pose stage: the candidates (flags bit 0) in caller order, gathered once for both attempts
    sv_compact_kernel<<<1, kCompactThreads, 0, s>>>(dp(i_flags), n, (1u << 1) | (1u << 3), di(x_cand), cnt + 0);
    sv_gather_kernel<<<blocks, 128, 0, s>>>(all, di(x_cand), cnt + 0, n, sub);
    CK(cudaGetLastError());
    const double* priors[2] = {in->T_estimate, in->T_estimate_damped};
    int accepted = -1, attempts = 0, measurements[2] = {0, 0};
    for (int a = 0; a < 2 && accepted < 0; ++a) {
        attempts = a + 1;
        if (n_cand > 0) {
            if ((rc = clear_sub()) != SVI_SUCCESS) return rc;
            rc = enqueue_cascade(ctx, n_cand, priors[a], in->motion_scaling, SVI_STAGE_1 | SVI_STAGE_2, x_lm.ld(ctx), x_lm.ex(ctx), nullptr, sub_out, nullptr);
            if (rc != SVI_SUCCESS) return rc;
        }
        // the solver's measurements: the hits in candidate order
        sv_compact_kernel<<<1, kCompactThreads, 0, s>>>(sub_out.stage, n_cand, 0x1Eu /* stages 1..4 */, di(x_hits), cnt + 1);
        const PositIn pi = posit_in(ctx, dev_at<double>(ctx, x_pxyz), dev_at<float>(ctx, x_puvl), dev_at<float>(ctx, x_puvr), priors[a], in->T_last, in->t_imu);
        sv_posit_assemble_kernel<<<blocks, 128, 0, s>>>(di(x_hits), cnt + 1, n, sub.xyz_w, sub_out, dev_at<double>(ctx, x_pxyz), dev_at<float>(ctx, x_puvl),
                                                        dev_at<float>(ctx, x_puvr));
        stereo_posit_count_kernel<<<1, kPositThreads, kPositSmemBytes, s>>>(pi, cnt + 1, posit_dev + a);
        CK(cudaGetLastError());
        // wait: the outcome decides whether the damped attempt runs
        CK(cudaMemcpyAsync(hp + o_posit + a * sizeof(PositOut), posit_dev + a, sizeof(PositOut), cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(hp + x_cnt + sizeof(int), cnt + 1, sizeof(int), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        PositOut po;
        std::memcpy(&po, hp + o_posit + a * sizeof(PositOut), sizeof(po));
        std::memcpy(&measurements[a], hp + x_cnt + sizeof(int), sizeof(int));
        if (po.outcome == SVI_POSIT_OK) accepted = a;
    }
    // the stage-1/2 results of the last attempt that ran, at the candidates' places
    if (n_cand > 0) sv_scatter_kernel<<<blocks, 128, 0, s>>>(di(x_cand), cnt + 0, n, sub_out, pose_out, nullptr);
    double T[16];
    if (accepted >= 0) std::memcpy(T, reinterpret_cast<const PositOut*>(hp + o_posit + accepted * sizeof(PositOut))->T, sizeof(T));
    else std::memcpy(T, in->T_estimate_damped, sizeof(T));
    SvPose pose;
    std::memcpy(pose.T, T, sizeof(T));

    // ---- epipolar stage: route every landmark, stage 3 on the moved ones (the count stays on the device)
    sv_route_kernel<<<blocks, 128, 0, s>>>(n, dp(i_flags), pose_out.stage, accepted >= 0 ? 1 : 0, pose, all.T_det, route);
    sv_compact_kernel<<<1, kCompactThreads, 0, s>>>(route, n, 1u << kRouteEpipolar, di(x_epi), cnt + 2);
    sv_gather_kernel<<<blocks, 128, 0, s>>>(all, di(x_epi), cnt + 2, n, sub);
    CK(cudaGetLastError());
    if ((rc = clear_sub()) != SVI_SUCCESS) return rc;
    rc = enqueue_cascade(ctx, n, T, in->motion_scaling, SVI_STAGE_3, x_lm.ld(ctx), x_lm.ex(ctx), sub.desc_ref, sub_out, cnt + 2);
    if (rc != SVI_SUCCESS) return rc;
    sv_scatter_kernel<<<blocks, 128, 0, s>>>(di(x_epi), cnt + 2, n, sub_out, epi_out, route);   // + the SVI_EPI_NO_TRANSLATION re-route
    // ---- regional stage 2 on the unmoved ones and the re-routed ones; wait: its launch sizes need the count
    sv_compact_kernel<<<1, kCompactThreads, 0, s>>>(route, n, (1u << kRouteRegional) | (1u << kRouteRegionalNoTranslation), di(x_reg), cnt + 3);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(hp + x_cnt, cnt, 4 * sizeof(int), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    int n_reg = 0;
    std::memcpy(&n_reg, hp + x_cnt + 3 * sizeof(int), sizeof(int));
    if (n_reg < 0 || n_reg > n) return fail(ctx, SVI_ERR_CUDA, "svi_track_frame_stereo_only: regional count out of range");
    if (n_reg > 0) {
        sv_gather_kernel<<<blocks, 128, 0, s>>>(all, di(x_reg), cnt + 3, n, sub);
        CK(cudaGetLastError());
        if ((rc = clear_sub()) != SVI_SUCCESS) return rc;
        rc = enqueue_cascade(ctx, n_reg, T, in->motion_scaling, SVI_STAGE_2, x_lm.ld(ctx), x_lm.ex(ctx), nullptr, sub_out, nullptr);
        if (rc != SVI_SUCCESS) return rc;
        sv_scatter_kernel<<<blocks, 128, 0, s>>>(di(x_reg), cnt + 3, n, sub_out, epi_out, nullptr);
        CK(cudaGetLastError());
    }
    // ---- every result in one copy
    if ((rc = call_fetch(ctx, o_posit, out_end, s)) != SVI_SUCCESS) return rc;
    idle.done = true;
    for (int a = 0; a < 2; ++a) {
        if (a < attempts) posit_result_from(*reinterpret_cast<const PositOut*>(hp + o_posit + a * sizeof(PositOut)), &out->attempt[a]);
        else std::memset(&out->attempt[a], 0, sizeof(out->attempt[a]));
    }
    out->attempts = attempts;
    out->measurements[0] = measurements[0];
    out->measurements[1] = measurements[1];
    out->source = accepted == 0 ? SVI_SV_POSIT : accepted == 1 ? SVI_SV_POSIT_DAMPED : SVI_SV_PRIOR;
    std::memcpy(out->T_world_to_left, T, sizeof(T));
    o_pose.copy_out(ctx, N, out->pose_stage);
    std::memcpy(out->route, hp + o_route, N);
    o_epi.copy_out(ctx, N, out->epipolar_stage);
    return check_overflow(ctx);
}

int svi_set_profiling(svi_ctx* ctx, int enable) {
    if (!ctx) return SVI_ERR_INVALID;
    for (int i = 0; i < ctx->n_lanes; ++i) cudaStreamSynchronize(ctx->lanes[i].stream);
    collect_timings(ctx);
    for (int s = 0; s < kStages; ++s) { ctx->stage_ms[s] = 0.0; ctx->stage_launches[s] = 0; }
    ctx->profiling = enable != 0;
    ctx->serial = enable == 2;
    if (ctx->profiling)
        for (int i = 0; i < ctx->n_lanes; ++i) reserve_events(ctx->lanes[i], ctx->serial && i == 0 ? 8 * kEventPool : kEventPool);
    return SVI_SUCCESS;
}

int svi_check_overflow(svi_ctx* ctx) {
    if (!ctx) return SVI_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    for (int i = 0; i < ctx->n_lanes; ++i) CK(cudaStreamSynchronize(ctx->lanes[i].stream));
    return check_overflow(ctx);
}

int svi_stage_timings(svi_ctx* ctx, const char** names, double* total_ms, int64_t* launches, int capacity) {
    if (!ctx || !names || !total_ms || !launches) return SVI_ERR_INVALID;
    for (int i = 0; i < ctx->n_lanes; ++i) cudaStreamSynchronize(ctx->lanes[i].stream);
    collect_timings(ctx);
    int n = std::min(capacity, kStages);
    for (int i = 0; i < n; ++i) {
        names[i] = kStageNames[i];
        total_ms[i] = ctx->stage_ms[i];
        launches[i] = ctx->stage_launches[i];
    }
    return n;
}

// ---- undistortion + rectification of raw images (CStereoCamera.h:102-107: cv::initUndistortRectifyMap + cv::remap)
int svi_rectify_map(const svi_camera* cam, const svi_rectification* r, int16_t* xy, uint16_t* frac) {
    const std::string e = rectify_map_host(cam, r, xy, frac);
    return e.empty() ? SVI_SUCCESS : fail(nullptr, SVI_ERR_INVALID, e);
}

int svi_set_rectification(svi_ctx* ctx, const svi_rectification* left, const svi_rectification* right) {
    if (!ctx) return SVI_ERR_INVALID;
    if (!left != !right) return fail(ctx, SVI_ERR_INVALID, "svi_set_rectification: give both cameras or neither");
    CK(cudaSetDevice(ctx->device));
    const size_t npix = (size_t)ctx->W * ctx->H, npad = (npix + 7) & ~size_t(7);   // 8: camera 1's xy block stays 16-byte aligned
    std::vector<int16_t> xy;
    std::vector<uint16_t> frac;
    if (left) {   // both maps first: a rejected calibration leaves the ctx as it was
        xy.assign(2 * 2 * npad, 0);
        frac.assign(2 * npad, 0);
        for (int c = 0; c < 2; ++c) {
            const std::string e = rectify_map_host(c ? &ctx->cam_r : &ctx->cam_l, c ? right : left, xy.data() + c * 2 * npad, frac.data() + c * npad);
            if (!e.empty()) return fail(ctx, SVI_ERR_INVALID, e + (c ? " (right camera)" : " (left camera)"));
        }
    }
    // nothing queued may still read the maps or the raw planes that are replaced below
    for (int i = 0; i < ctx->n_lanes; ++i) CK(cudaStreamSynchronize(ctx->lanes[i].stream));
    CK(cudaStreamSynchronize(ctx->side));
    if (ctx->profiling) collect_timings(ctx);
    if (!left) {
        for (int i = 0; i < ctx->n_lanes; ++i) {
            Lane& l = ctx->lanes[i];
            if (l.raw_l) cudaFree(l.raw_l);
            if (l.raw_r) cudaFree(l.raw_r);
            l.raw_l = l.raw_r = nullptr;
        }
        if (ctx->rect_map) cudaFree(ctx->rect_map);
        ctx->rect_map = nullptr;
        ctx->rect_npad = 0;
        ctx->rect = false;
        return SVI_SUCCESS;
    }
    ctx->rect = false;   // until everything below is in place
    const size_t raw = (size_t)ctx->chunk * ctx->H * ctx->dev_pitch;   // allocated once, kept until rectification is switched off
    for (int i = 0; i < ctx->n_lanes; ++i) {
        if (!ctx->lanes[i].raw_l) CK(dmalloc(&ctx->lanes[i].raw_l, raw));
        if (!ctx->lanes[i].raw_r) CK(dmalloc(&ctx->lanes[i].raw_r, raw));
    }
    if (!ctx->rect_map) CK(cudaMalloc(reinterpret_cast<void**>(&ctx->rect_map), 2 * npad * 6));
    ctx->rect_npad = (int)npad;
    for (int c = 0; c < 2; ++c) {
        CK(cudaMemcpy(ctx->rect_map + c * npad * 6, xy.data() + c * 2 * npad, npad * 4, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(ctx->rect_map + c * npad * 6 + npad * 4, frac.data() + c * npad, npad * 2, cudaMemcpyHostToDevice));
    }
    ctx->rect = true;
    return SVI_SUCCESS;
}

int svi_rectify(svi_ctx* ctx, int side, const uint8_t* raw, size_t pitch, size_t frame_stride, int n_frames, uint8_t* out, size_t out_pitch) {
    if (!ctx) return SVI_ERR_INVALID;
    if (!raw || !out || (side != 0 && side != 1) || n_frames < 0 || (int)pitch < ctx->W || (int)out_pitch < ctx->W ||
        (n_frames > 1 && frame_stride < pitch * (size_t)ctx->H))
        return fail(ctx, SVI_ERR_INVALID, "svi_rectify: bad argument");
    if (!ctx->rect) return fail(ctx, SVI_ERR_INVALID, "svi_rectify: no rectification set (svi_set_rectification)");
    CK(cudaSetDevice(ctx->device));
    Lane& l = ctx->lanes[0];
    cudaStream_t s = l.stream;
    const size_t dstride = (size_t)ctx->H * ctx->dev_pitch;
    uint8_t* d_raw = side ? l.raw_r : l.raw_l;
    for (int f0 = 0; f0 < n_frames; f0 += ctx->chunk) {
        const int nf = std::min(ctx->chunk, n_frames - f0);
        for (int f = 0; f < nf; ++f)
            CK(cudaMemcpy2DAsync(d_raw + f * dstride, ctx->dev_pitch, raw + (size_t)(f0 + f) * frame_stride, pitch, ctx->W, ctx->H,
                                 cudaMemcpyHostToDevice, s));
        const int rc = rectify_one(ctx, side, d_raw, ctx->dev_pitch, dstride, l.img_l, nf, s);
        if (rc != SVI_SUCCESS) { cudaStreamSynchronize(s); return rc; }
        CK(cudaMemcpy2DAsync(out + (size_t)f0 * ctx->H * out_pitch, out_pitch, l.img_l, ctx->dev_pitch, ctx->W, (size_t)ctx->H * nf,
                             cudaMemcpyDeviceToHost, s));
    }
    CK(cudaStreamSynchronize(s));
    return check_overflow(ctx);
}

// ---- frame-partitioned batches over several GPUs (SURVEY.md 8e): stereo pairs are independent, so a batch of F
// frames is cut into contiguous ranges [g*F/G, (g+1)*F/G), one per device; each range runs through its own svi_ctx on
// its own host thread and writes a disjoint slice of the caller's arrays.  No collective, no peer access: the result is
// byte-for-byte the one a single device produces.
struct svi_multi {
    std::vector<svi_ctx*> ctx;
    std::vector<int> devices;
    std::string err;
};

int svi_multi_create(const svi_camera* left, const svi_camera* right, const svi_params* params, const int* devices, int n_devices,
                     svi_multi** out) {
    if (!left || !right || !out || n_devices < 1 || n_devices > 64) return fail(nullptr, SVI_ERR_INVALID, "svi_multi_create: bad argument");
    *out = nullptr;
    svi_multi* m = new svi_multi();
    for (int g = 0; g < n_devices; ++g) {
        svi_ctx* c = nullptr;
        const int dev = devices ? devices[g] : g;
        const int rc = svi_create(left, right, params, dev, &c);
        if (rc != SVI_SUCCESS) {   // g_create_error holds the reason
            for (svi_ctx* q : m->ctx) svi_destroy(q);
            delete m;
            return rc;
        }
        m->ctx.push_back(c);
        m->devices.push_back(dev);
    }
    *out = m;
    return SVI_SUCCESS;
}

void svi_multi_destroy(svi_multi* m) {
    if (!m) return;
    for (svi_ctx* c : m->ctx) svi_destroy(c);
    delete m;
}

const char* svi_multi_last_error(const svi_multi* m) { return m ? m->err.c_str() : g_create_error.c_str(); }
int svi_multi_device_count(const svi_multi* m) { return m ? (int)m->ctx.size() : 0; }

int svi_multi_frame_range(const svi_multi* m, int n_frames, int part, int* first, int* count) {
    if (!m || !first || !count || n_frames < 0 || part < 0 || part >= (int)m->ctx.size()) return SVI_ERR_INVALID;
    const long long G = (long long)m->ctx.size();
    const long long f0 = (long long)part * n_frames / G, f1 = (long long)(part + 1) * n_frames / G;
    *first = (int)f0;
    *count = (int)(f1 - f0);
    return SVI_SUCCESS;
}

int svi_multi_stereo_frames(svi_multi* m, const uint8_t* left, const uint8_t* right, size_t pitch, size_t frame_stride, int n_frames,
                            const uint8_t* masks, svi_stereo_result* out) {
    if (!m) return SVI_ERR_INVALID;
    if (!left || !right || !out || n_frames < 0) { m->err = "svi_multi_stereo_frames: bad argument"; return SVI_ERR_INVALID; }
    const int G = (int)m->ctx.size();
    std::vector<int> rc(G, SVI_SUCCESS);
    std::vector<std::thread> workers;
    const size_t cap = (size_t)out->capacity_per_frame;
    for (int g = 0; g < G; ++g) {
        int f0 = 0, nf = 0;
        svi_multi_frame_range(m, n_frames, g, &f0, &nf);
        if (nf == 0) continue;
        workers.emplace_back([=, &rc]() {
            svi_stereo_result sub = *out;   // the same arrays, advanced to this range's first frame
            const size_t o0 = (size_t)f0 * cap;
            sub.n_keypoints = out->n_keypoints ? out->n_keypoints + f0 : nullptr;
            sub.n_detected = out->n_detected ? out->n_detected + f0 : nullptr;
            sub.uv_left = out->uv_left ? out->uv_left + o0 * 2 : nullptr;
            sub.uv_right = out->uv_right ? out->uv_right + o0 * 2 : nullptr;
            sub.xyz_left = out->xyz_left ? out->xyz_left + o0 * 3 : nullptr;
            sub.desc_left = out->desc_left ? out->desc_left + o0 * 32 : nullptr;
            sub.desc_right = out->desc_right ? out->desc_right + o0 * 32 : nullptr;
            sub.distance = out->distance ? out->distance + o0 : nullptr;
            sub.match_index = out->match_index ? out->match_index + o0 : nullptr;
            sub.status = out->status ? out->status + o0 : nullptr;
            rc[g] = svi_stereo_frames(m->ctx[g], left + (size_t)f0 * frame_stride, right + (size_t)f0 * frame_stride, pitch, frame_stride, nf,
                                      masks ? masks + (size_t)f0 * frame_stride : nullptr, &sub);
        });
    }
    for (std::thread& t : workers) t.join();
    for (int g = 0; g < G; ++g)
        if (rc[g] != SVI_SUCCESS) {
            m->err = "device " + std::to_string(m->devices[g]) + ": " + svi_last_error(m->ctx[g]);
            return rc[g];
        }
    return SVI_SUCCESS;
}

int svi_multi_set_rectification(svi_multi* m, const svi_rectification* left, const svi_rectification* right) {
    if (!m) return SVI_ERR_INVALID;
    for (size_t g = 0; g < m->ctx.size(); ++g) {
        const int rc = svi_set_rectification(m->ctx[g], left, right);
        if (rc != SVI_SUCCESS) {
            m->err = "device " + std::to_string(m->devices[g]) + ": " + svi_last_error(m->ctx[g]);
            return rc;
        }
    }
    return SVI_SUCCESS;
}

int svi_kernels_per_chunk(const svi_ctx* ctx, int n_frames) {
    if (!ctx || n_frames <= 0) return SVI_ERR_INVALID;
    const long long slots = (long long)std::min(n_frames, ctx->chunk) * ctx->p.max_corners;
    const bool pre = ctx->match_pre && slots / (2LL * ctx->n_sm * 9) >= MATCH_KP_PER_WARP;
    // detector, RIGHT box sums, corner selection, matcher (+ LEFT descriptors as a kernel of their own, + the bin sort)
    return 4 + (pre ? 1 : 0) + (pre && ctx->match_binned ? 1 : 0) + (ctx->rect ? 1 : 0);
}

int svi_config(const svi_ctx* ctx, int32_t* chunk_frames, int32_t* n_lanes, int32_t* select_in_smem) {
    if (!ctx) return SVI_ERR_INVALID;
    if (chunk_frames) *chunk_frames = ctx->chunk;
    if (n_lanes) *n_lanes = ctx->n_lanes;
    if (select_in_smem) *select_in_smem = ctx->select_smem ? 1 : 0;
    return SVI_SUCCESS;
}

}  // extern "C"
