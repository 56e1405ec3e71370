/* svi_gpu.h -- C-ABI of libsvi_gpu.so: svi_mapper's stereo front-end hot path on one B200.
 *
 * This boundary does not exist in the reference (it is a single C++ process calling OpenCV);
 * it is what the reference's own seams would bind if the arithmetic moved to the GPU.  Each
 * entry point cites the reference interface it replaces (paths relative to the svi_mapper tree).
 *
 *   - plain C, no C++ types, no exceptions across the boundary
 *   - the caller owns every host buffer (inputs and pre-sized outputs); the library owns all
 *     device memory inside svi_ctx; nothing returned outlives svi_destroy
 *   - call-level failures are negative return codes + svi_last_error(); per-item outcomes
 *     (the reference's CExceptionNoMatchFound control flow) are DATA: one svi_status per item
 *   - one svi_ctx per (host thread, GPU); calls on one ctx are serialised by the caller;
 *     every export is synchronous on return unless its name ends in _device
 */
#ifndef SVI_GPU_H
#define SVI_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SVI_DESCRIPTOR_BYTES 32 /* src/types/Types.h:73-75 DESCRIPTOR_SIZE_BYTES */

typedef struct svi_ctx svi_ctx;

/* call-level return codes */
enum {
    SVI_SUCCESS = 0,
    SVI_ERR_INVALID = -1,    /* bad argument */
    SVI_ERR_CUDA = -2,       /* CUDA runtime error, text in svi_last_error */
    SVI_ERR_CAPACITY = -3,   /* a caller- or ctx-sized buffer was too small (never a silent drop) */
    SVI_ERR_NO_DEVICE = -4,
    SVI_ERR_UNSUPPORTED = -5
};

/* Per-item outcome: one value per distinct failure string the reference throws on this path
 * (SURVEY.md Appendix C).  svi_status_text() returns the reference's what() text. */
typedef enum svi_status {
    SVI_OK = 0,
    SVI_TRI_RANGE = 1,      /* src/core/CTriangulator.cpp:65,199,270  "insufficient search range"   */
    SVI_TRI_NO_DESC = 2,    /* src/core/CTriangulator.cpp:88,222,293  "could not compute descriptors" */
    SVI_TRI_NO_MATCH = 3,   /* src/core/CTriangulator.cpp:97,231,302  "no match found"               */
    SVI_TRI_DISTANCE = 4,   /* src/core/CTriangulator.cpp:117,251,322 "matching distance"            */
    SVI_TRI_ZERO_DISP = 5,  /* src/core/CTriangulator.cpp:332         "zero disparity"               */
    SVI_TRI_BAD_ROI = 6,    /* search ROI leaves the image: the reference aborts in cv::Mat::operator() */
    SVI_TRK_DEPTH = 7,      /* src/core/CFundamentalMatcher.cpp:1446,1508 "invalid depth"            */
    SVI_TRK_STAGE1_DIST = 8,/* src/core/CFundamentalMatcher.cpp:1471,1533 "insufficient matching distance" */
    SVI_TRK_TRI_DESC = 9,   /* src/core/CFundamentalMatcher.cpp:1452,1514 "triangulation descriptor mismatch" */
    SVI_TRK_OUT_OF_FOV = 10, /* src/core/CFundamentalMatcher.cpp:1416 projection outside m_cFieldOfView */
    SVI_TRK_NO_FEATURES = 11, /* src/core/CFundamentalMatcher.cpp:1660,1780 "no features detected"  */
    SVI_TRK_NO_MATCHES = 12,  /* src/core/CFundamentalMatcher.cpp:1654,1775 "no matches found"      */
    SVI_TRK_DESC = 13,        /* src/core/CFundamentalMatcher.cpp:1648,1770 "descriptor mismatch"   */
    SVI_TRK_RANGE = 14,       /* src/core/CFundamentalMatcher.cpp:1642,1765 "out of tracking range" */
    SVI_EPI_OUT_OF_SIGHT = 15, /* CExceptionEpipolarLine :1814 "projection out of sight"                      */
    SVI_EPI_VERTICAL = 16,     /* :1845 "vertical out of sight"                                               */
    SVI_EPI_NEG_SLOPE = 17,    /* :1871 "caught bad projection negative slope"                                */
    SVI_EPI_POS_SLOPE = 18,    /* :1900 "caught bad projection positive slope"                                */
    SVI_EPI_ZERO_LEN = 19,     /* :1939 "zero line length"                                                    */
    SVI_EPI_POOL_EMPTY = 20,   /* :2351 "could not find a matching descriptor (empty key point pool)"         */
    SVI_EPI_NO_MATCHES = 21,   /* :2361 "could not find any matches (empty matches pool)"                     */
    SVI_EPI_DIST = 22,         /* :2395 "could not find a matching descriptor"                                */
    SVI_EPI_ORIG_DIST = 23,    /* :2390 "... (ORIGINAL matching distance too big)"                            */
    SVI_EPI_NO_TRANSLATION = 24, /* :1804 detection pose == current pose: stage 3 is skipped for this landmark */
    SVI_SPARSE_NOT_MUTUAL = 25,  /* sparse frames with svi_sparse_band.mutual: not a reference path (no reference text) */
    SVI_SUBPIXEL_REJECTED = 26,  /* svi_params.subpixel_window: the SAD minimum lies on the edge of the search (no reference text) */
    SVI_LR_INCONSISTENT = 27     /* svi_params.lr_max_diff: the reverse search does not lead back to the LEFT key-point (no reference text) */
} svi_status;

/* src/vision/CPinholeCamera.h:16-64: the members the hot path reads
 * (m_uWidthPixel, m_uHeightPixel, m_matProjection row-major 3x4). */
typedef struct svi_camera {
    uint32_t width;
    uint32_t height;
    double P[12];
} svi_camera;

/* The reference's compile-time constants (SURVEY.md Appendix B); svi_params_default() fills in
 * exactly those values.  max_corners / search_range_px are parameters because the batch and
 * stress configurations of BASELINE.json raise them. */
typedef struct svi_params {
    double quality_level;      /* 0.01  src/core/CFundamentalMatcher.cpp:18 (cv::GFTTDetector takes doubles) */
    double min_distance;       /* 7.0   ibid. */
    double harris_k;           /* 0.04  OpenCV default for GFTTDetector */
    double min_disparity_px;   /* 0.01  src/core/CTriangulator.h:21; must be > 0 (svi_create refuses 0, negatives and NaN) */
    int32_t max_corners;       /* 1000  src/core/CFundamentalMatcher.cpp:18 */
    float keypoint_size;       /* 7.0   cv::KeyPoint::size GFTT reports (= blockSize) */
    float search_range_px;     /* 60.0  src/core/CTriangulator.h:20 */
    float match_cutoff;        /* 100.0 src/core/CTriangulator.cpp:13 */
    float cutoff_stage1;       /* 25.0  src/core/CFundamentalMatcher.cpp:23 */
    float cutoff_stage2;       /* 50.0  :24 */
    float cutoff_stage3;       /* 50.0  :25 */
    float cutoff_original;     /* 100.0 :26 */
    int32_t max_candidates;    /* per-frame capacity of the NMS candidate list (default 16384) */
    int32_t chunk_frames;      /* frames per kernel wave; 0 = library default */
    int32_t max_queries;       /* capacity of the per-query entry points (triangulate_*, describe, track) */
    /* optional detector mode (NOT a reference code path; SURVEY.md 8f rank 2): 0 = GFTT/Harris as the reference
     * (default), 1 = FAST-9/16 as cv::FastFeatureDetector(threshold, nonmaxSuppression, TYPE_9_16): every corner
     * in scan order, no maxCorners cut -- more corners than max_corners is SVI_ERR_CAPACITY */
    int32_t detector;
    int32_t fast_threshold;    /* 10 (cv default) */
    int32_t fast_nonmax;       /* 1 */
    /* optional sub-pixel disparity (NOT a reference code path; ORB-SLAM2's Frame::ComputeStereoMatches refinement): 0 = off
     * (default): every output is the reference's integer-disparity result.  w = subpixel_window > 0 refines the match of every
     * slot the new-landmark path reports SVI_OK (after the left-right check of lr_max_diff when it is on) --
     * svi_stereo_frames[_device] (both matchers), svi_stereo_frame_masked,
     * svi_stereo_frames_sparse[_device] (after the left-right check when it is on) and svi_multi_stereo_frames -- with
     * L = subpixel_search, on the images the detector read (the rectified planes while rectification is set):
     *   1. PL = the (2w+1)^2 LEFT patch centred on (xL, y) minus its centre pixel (integers);
     *   2. for k = -L .. L: PR(k) = the RIGHT patch centred on ((int)xR + k, y) minus its centre pixel, SAD(k) = sum |PL - PR(k)|
     *      (int32).  y is the LEFT row for both patches (rectified images): a sparse match on a neighbouring RIGHT row is
     *      refined on the LEFT row, and its uv_right.y stays the RIGHT key-point's row;
     *   3. k* = the first strict minimum in increasing k; k* = +-L is SVI_SUBPIXEL_REJECTED;
     *   4. s1, s2, s3 = SAD(k*-1), SAD(k*), SAD(k*+1); delta = float(s1 - s3) / (2 * float(s1 + s3 - 2 s2)) in fp32
     *      (the denominator is > 0, delta is in (-0.5, 0.5]);
     *   5. xR' = (xR + (float)k*) + delta, fp32, rounded after each addition;
     *   6. getPointInLEFT(uv_left, (xR', y)): SVI_TRI_ZERO_DISP, or SVI_OK with uv_right.x = xR' and xyz_left.
     * Status order: the integer path's statuses, SVI_SUBPIXEL_REJECTED, then step 6.  A slot the integer path reports
     * SVI_TRI_ZERO_DISP (only possible with min_disparity_px >= 1 or a sparse band admitting x_R >= x_L) is not refined.
     * Only uv_right.x, xyz_left and status change: distance, match_index, second_distance, every LEFT field and the counts are
     * byte-identical to the mode off, and desc_right stays the descriptor at the integer match.
     * svi_create refuses w < 0 and, for w > 0, L < 1 or w + L > 28.  BRIEF's 28-px border filter keeps every LEFT key-point
     * and every RIGHT position either matcher reports at least 28 px inside the image, so with w + L <= 28 every patch lies
     * inside the image: there is no border mode.  (A fractional keypoint_size or search_range_px can make the dense
     * matcher's uv_right.x fractional; a slot whose patches would then leave the image is SVI_SUBPIXEL_REJECTED.)
     * Not applied by the tracking cascade (svi_track_landmarks*), svi_track_frame_stereo_only or the per-query
     * svi_triangulate_* / svi_point_in_left. */
    int32_t subpixel_window;   /* 0 */
    int32_t subpixel_search;   /* 0 */
    /* optional left-right consistency check of the dense scan-line matches (NOT a reference code path; the convention of
     * cv::StereoSGBM's disp12MaxDiff): -1 = off (default): every output, launch and allocation is the reference path's.
     * With lr_max_diff = t >= 0, every slot the dense matcher reports SVI_OK, with LEFT key-point (xL, y), match (xR, y) and
     * RIGHT descriptor desc_right, is searched back with the reference's own reverse search, the 7-argument
     * CTriangulator::getPointTriangulatedInLEFT (CTriangulator.cpp:255-324, what svi_triangulate_left runs):
     *   r = getPointTriangulatedInLEFT(LEFT image, search_range_px, u_tl = xR - 4 * keypoint_size,
     *                                  v_tl = y - 4 * keypoint_size, keypoint_size, (xR, y), desc_right)   (fp32 corners)
     *   the slot stays SVI_OK iff r.status == SVI_OK and |r.uv.x - xL| <= t (fp32), otherwise it is SVI_LR_INCONSISTENT.
     * The LEFT image is the plane the detector read (the rectified one while rectification is set).  The reverse pool
     * xR+1 .. xR+search_range+1 holds xL, so the reverse minimum distance is at most the forward one; with the default
     * parameters the reverse search cannot fail the cut-off, and it fails only through the rule above (for example through
     * getPointInLEFT with a raised min_disparity_px).  Status order: every forward status unchanged, the check on forward
     * SVI_OK slots only, then the sub-pixel refinement (subpixel_window) on the slots that survive it.  status is the only
     * field the check writes: every other output byte is identical to the call with the check off.
     * Applied by svi_stereo_frames[_device] (both matchers, both detectors), svi_stereo_frame_masked and
     * svi_multi_stereo_frames.  Not applied by the sparse frames (svi_sparse_band.mutual is their check), the tracking
     * cascade (svi_track_landmarks*), svi_track_frame_stereo_only or the per-query svi_triangulate_* / svi_point_in_left.
     * svi_create refuses values below -1. */
    int32_t lr_max_diff;       /* -1 */
} svi_params;

enum { SVI_DETECTOR_GFTT_HARRIS = 0, SVI_DETECTOR_FAST_9_16 = 1 };

int svi_params_default(svi_params* p);
const char* svi_status_text(int status);

/* Which BRIEF-32 pair table this build of the library carries (the 256 test pairs are compile-time constants of the
 * match kernels): file name, its description line, number of distinct test points, FNV-1a hash of the offsets.
 * The table shipped in this repository is a STAND-IN, not opencv_contrib's generated_32.i behind
 * cv::xfeatures2d::BriefDescriptorExtractor::create(32) (src/core/CTriangulator.cpp:11): descriptors are bit-exact to
 * the CPU restatement with the same table, not to the reference's.  Another table: python -m svi_mapper_b200.build --table. */
const char* svi_brief_table_info(void);

/* Replaces the CTriangulator / CFundamentalMatcher constructors' OpenCV object creation
 * (src/core/CTriangulator.cpp:8-21, src/core/CFundamentalMatcher.cpp:14-28). */
int svi_create(const svi_camera* left, const svi_camera* right, const svi_params* params,
               int device, svi_ctx** out);
void svi_destroy(svi_ctx* ctx);
const char* svi_last_error(const svi_ctx* ctx); /* ctx may be NULL: last create error */
int svi_device_count(void);

/* SoA result of the new-landmark path, caller-owned.  Slot (f, i) lives at index
 * f*capacity_per_frame + i; only slots i < n_keypoints[f] carry results -- the content of the slots
 * behind them (up to max_corners per frame) is unspecified after the call.  113 bytes per key-point. */
typedef struct svi_stereo_result {
    int32_t capacity_per_frame; /* in: >= params.max_corners */
    int32_t* n_keypoints;       /* [n_frames] corners that survived BRIEF's 28-px border filter */
    int32_t* n_detected;        /* [n_frames] GFTT corners before that filter; may be NULL */
    float* uv_left;             /* [.. * 2] */
    float* uv_right;            /* [.. * 2] valid when status == SVI_OK */
    double* xyz_left;           /* [.. * 3] valid when status == SVI_OK */
    uint8_t* desc_left;         /* [.. * 32] */
    uint8_t* desc_right;        /* [.. * 32] valid when status == SVI_OK */
    int32_t* distance;          /* Hamming distance of the arg-min candidate, -1 if none evaluated */
    int32_t* match_index;       /* pool index (cv::DMatch::trainIdx), -1 if none */
    uint8_t* status;            /* svi_status */
} svi_stereo_result;

/* CFundamentalMatcher::addNewLandmarks (src/core/CFundamentalMatcher.cpp:83-193) minus landmark
 * bookkeeping, for a batch of independent stereo pairs: GFTT/Harris detect on LEFT (optional
 * u8 masks, 0 = blocked), BRIEF-32 on the kept corners, per corner the dense same-row search in
 * RIGHT (CTriangulator::getPointTriangulatedInRIGHTFull, src/core/CTriangulator.cpp:51-119),
 * Hamming arg-min, cut-off, closed-form triangulation.  Host buffers; images are n_frames
 * planes of height x pitch bytes, frame_stride bytes apart. */
int svi_stereo_frames(svi_ctx* ctx, const uint8_t* left, const uint8_t* right, size_t pitch,
                      size_t frame_stride, int n_frames, const uint8_t* masks_or_null,
                      svi_stereo_result* out);

/* Same, but every pointer (images, masks, and the arrays inside *out) is a DEVICE pointer on
 * ctx's GPU and the work is enqueued after everything already queued on `cuda_stream`
 * (a cudaStream_t; NULL = default stream); later work on that stream waits for it.
 * Returns without synchronising. */
int svi_stereo_frames_device(svi_ctx* ctx, const uint8_t* left, const uint8_t* right, size_t pitch,
                             size_t frame_stride, int n_frames, const uint8_t* masks_or_null,
                             const svi_stereo_result* out, void* cuda_stream);

/* Capacity check for work enqueued by svi_stereo_frames_device (every host-buffer entry point does it
 * itself before returning): waits for the ctx's streams, then returns SVI_ERR_CAPACITY (and clears the
 * condition) if any frame since the last check produced more candidates than svi_params.max_candidates
 * (or, in FAST mode, more corners than max_corners) -- the results of such a frame are zero key-points,
 * never a silently truncated list.  SVI_SUCCESS otherwise. */
int svi_check_overflow(svi_ctx* ctx);

/* CFundamentalMatcher::getMaskActiveLandmarks (src/core/CFundamentalMatcher.cpp:2043-2073) on the device: a
 * W x H plane of 255 with, per centre, the filled radius-7 disc of zeros that
 * cv::circle(mask, Point(cvRound(x), cvRound(y)), 7, Scalar(0), -1) draws (149 px; m_uFeatureRadiusForMask,
 * CFundamentalMatcher.h:70).  centres_xy = n_centres x (x, y): last LEFT detection of a visible landmark or the
 * projection of an invisible one (the caller's bookkeeping).  The plane is returned to `mask` (pitch bytes per
 * row) -- for display / inspection; the new-landmark path below never needs it on the host. */
int svi_mask_active_landmarks(svi_ctx* ctx, const float* centres_xy, int n_centres, uint8_t* mask, size_t pitch);

/* addNewLandmarks for ONE pair with the detection mask of getMaskActiveLandmarks built on the device from the
 * landmark centres: 8 bytes per active landmark go to the GPU instead of a W x H mask plane.  Same outputs as
 * svi_stereo_frames(..., n_frames = 1, mask, out). */
int svi_stereo_frame_masked(svi_ctx* ctx, const uint8_t* left, const uint8_t* right, size_t pitch,
                            const float* centres_xy, int n_centres, svi_stereo_result* out);

/* cv::cornerHarris(img, 7, 3, k) as GFTTDetector runs it (response plane, fp32, W*H). */
int svi_harris_response(svi_ctx* ctx, const uint8_t* img, size_t pitch, float* response);

/* cv::GFTTDetector::detect(img, kps, mask) (src/core/CFundamentalMatcher.cpp:101): integer corner
 * coordinates as floats in OpenCV's order; xy holds n_frames * params.max_corners * 2 floats. */
int svi_detect(svi_ctx* ctx, const uint8_t* img, size_t pitch, size_t frame_stride, int n_frames,
               const uint8_t* masks_or_null, float* xy, int32_t* counts);

/* cv::xfeatures2d::BriefDescriptorExtractor::compute(img, kps, desc) on a full image
 * (src/core/CFundamentalMatcher.cpp:106): kept[i] = 0 where OpenCV erases the key-point
 * (28-px border); desc32 rows are written for every i (zero where erased). */
int svi_describe(svi_ctx* ctx, const uint8_t* img, size_t pitch, const float* xy, int n,
                 uint8_t* desc32, uint8_t* kept);

/* cv::BFMatcher(NORM_HAMMING)::match(query, train) (src/core/CTriangulator.cpp:93): per query the
 * first arg-min train index and its distance; -1/-1 when n_train == 0. */
int svi_match_hamming(svi_ctx* ctx, const uint8_t* query32, int n_query, const uint8_t* train32,
                      int n_train, int32_t* index, int32_t* distance);

/* Sparse epipolar-band matcher (optional mode; not a reference code path -- the reference searches dense scan
 * lines, SURVEY.md fact 2; this is the key-point-to-key-point form BASELINE.json's stress configuration names and
 * what cv::BFMatcher::match(query, train, mask) computes with mask(q,t) = |yq - yt| <= band_v && min_disparity <=
 * xq - xt <= max_disparity).  Per query: first arg-min train index among the admissible trains, its Hamming
 * distance and the second-best distance (for a ratio test in the caller); -1 where no train is admissible. */
int svi_match_epipolar(svi_ctx* ctx, const uint8_t* query32, const float* query_xy, int n_query,
                       const uint8_t* train32, const float* train_xy, int n_train, float band_v,
                       float min_disparity, float max_disparity, int32_t* index, int32_t* distance,
                       int32_t* second_distance);

/* Sparse stereo frames (optional mode; not a reference code path -- the reference matches by dense scan lines, as
 * svi_stereo_frames does): addNewLandmarks with LEFT key-points matched against RIGHT key-points inside an epipolar row band,
 * for a batch of independent pairs in one call.  Per frame:
 *   - LEFT: detection (svi_params.detector, with the optional masks), selection, BRIEF's border filter and descriptors as in
 *     svi_stereo_frames: n_keypoints, n_detected, uv_left and desc_left are byte-identical to that call's;
 *   - RIGHT: the same detector without a mask, the same selection and border filter -- the list svi_detect(RIGHT) followed
 *     by svi_describe's `kept` filter gives; match_index indexes it;
 *   - per LEFT slot, the admissible RIGHT key-points are those svi_match_epipolar admits (fp32 tests as written there) for
 *     this band.  None: SVI_TRI_NO_MATCH, distance = match_index = second_distance = -1.  Otherwise the first arg-min
 *     (lowest index on ties) and the second-smallest admissible distance; !(float(distance) < params.match_cutoff) gives
 *     SVI_TRI_DISTANCE (distance and index still written); else getPointInLEFT(uv_left, uv_right) as svi_point_in_left
 *     gives SVI_TRI_ZERO_DISP or SVI_OK with xyz_left, uv_right and desc_right (the matched RIGHT key-point's).
 * No ratio test is applied: second_distance is there for the caller's.
 * Left-right check (band.mutual = 1, cv::BFMatcher(NORM_HAMMING, crossCheck = true)): for a slot matched to RIGHT key-point
 *     j that passes the cut-off, the reverse arg-min of j -- the first arg-min over the frame's LEFT key-points under the
 *     same admissibility relation, lowest LEFT slot on ties -- must be this slot, else SVI_SPARSE_NOT_MUTUAL.  Status order:
 *     SVI_TRI_NO_MATCH, SVI_TRI_DISTANCE, SVI_SPARSE_NOT_MUTUAL, getPointInLEFT.  Every other field (LEFT fields,
 *     n_keypoints_right, distance, match_index, second_distance) is byte-identical to mutual = 0; uv_right, xyz_left and
 *     desc_right are valid for SVI_OK only, as always.  The first call with mutual = 1 allocates the check's per-lane scratch.
 * While rectification is set both images are raw.
 * SVI_ERR_INVALID for a NaN band field, min_disparity > max_disparity or mutual other than 0 or 1.  A frame whose
 * candidate list overflows on either side gets zero key-points on that side and the call returns SVI_ERR_CAPACITY (FAST
 * mode: more corners than max_corners on either side is SVI_ERR_CAPACITY too).  The first call allocates the per-lane scratch of this mode. */
typedef struct svi_sparse_band {
    float band_v;          /* |y_L - y_R| <= band_v                       */
    float min_disparity;   /* min_disparity <= x_L - x_R <= max_disparity */
    float max_disparity;
    int32_t mutual;        /* 0: no left-right check; 1: left-right check (SVI_SPARSE_NOT_MUTUAL) */
} svi_sparse_band;
typedef struct svi_sparse_result {
    int32_t* second_distance;    /* [frames * capacity_per_frame] second-smallest admissible distance, -1 if < 2 admissible */
    int32_t* n_keypoints_right;  /* [frames] RIGHT key-points after BRIEF's border filter */
} svi_sparse_result;
int svi_stereo_frames_sparse(svi_ctx* ctx, const uint8_t* left, const uint8_t* right, size_t pitch, size_t frame_stride,
                             int n_frames, const uint8_t* masks_or_null, const svi_sparse_band* band,
                             svi_stereo_result* out, svi_sparse_result* sparse);

/* Same on DEVICE pointers (images, masks and every array of *out and *sparse), enqueued after the work on `cuda_stream`
 * like svi_stereo_frames_device; returns without synchronising.  Capacity overflows are reported by svi_check_overflow. */
int svi_stereo_frames_sparse_device(svi_ctx* ctx, const uint8_t* left, const uint8_t* right, size_t pitch,
                                    size_t frame_stride, int n_frames, const uint8_t* masks_or_null,
                                    const svi_sparse_band* band, const svi_stereo_result* out,
                                    const svi_sparse_result* sparse, void* cuda_stream);

/* Per-query results of the triangulating scan-line searches. */
typedef struct svi_tri_result {
    float* uv;          /* [n*2] matched point in the searched image */
    double* xyz_left;   /* [n*3] */
    uint8_t* desc;      /* [n*32] descriptor at the matched point */
    int32_t* distance;  /* [n] */
    int32_t* match_index; /* [n] */
    uint8_t* status;    /* [n] */
} svi_tri_result;

/* CTriangulator::getPointTriangulatedInRIGHT / ...Full (src/core/CTriangulator.cpp:51-119,185-253)
 * for n queries against one RIGHT image: top_left = (p_fUTopLeft, p_fVTopLeft) per query,
 * uv_left = p_ptUVLEFT, desc_left = p_matReferenceDescriptorLEFT, size = p_fKeyPointSizePixels. */
int svi_triangulate_right(svi_ctx* ctx, const uint8_t* img_right, size_t pitch, int n,
                          const float* top_left, const float* uv_left, const uint8_t* desc_left,
                          float keypoint_size, svi_tri_result* out);

/* CTriangulator::getPointTriangulatedInLEFT, 7-argument overload (src/core/CTriangulator.cpp:255-324). */
int svi_triangulate_left(svi_ctx* ctx, const uint8_t* img_left, size_t pitch, int n,
                         const float* search_range, const float* top_left, const float* uv_right,
                         const uint8_t* desc_right, float keypoint_size, svi_tri_result* out);

/* CTriangulator::getPointInLEFT (src/core/CTriangulator.cpp:326-356) in bulk. */
int svi_point_in_left(svi_ctx* ctx, int n, const float* uv_left, const float* uv_right,
                      double* xyz_left, uint8_t* status);

/* Landmark state the tracker hands over (fields of CLandmark the stage reads:
 * src/types/CLandmark.h:35-59, src/core/CFundamentalMatcher.cpp:1404-1413). */
typedef struct svi_landmarks {
    const double* xyz_world;      /* [n*3] vecPointXYZOptimized */
    const uint8_t* last_desc_left;  /* [n*32] getLastDescriptorLEFT() */
    const uint8_t* last_desc_right; /* [n*32] getLastDescriptorRIGHT() */
    const float* last_disparity;  /* [n] getLastDisparity() */
    const float* keypoint_size;   /* [n] dKeyPointSize */
    /* stage 3 only; all three NULL = stop after stage 2 */
    const double* uv_reference_left;      /* [n*2] vecUVReferenceLEFT (first LEFT detection) */
    const uint8_t* desc_reference_left;   /* [n*32] matDescriptorReferenceLEFT */
    const double* T_left_to_world_at_detection; /* [n*16] row-major matTransformationLEFTtoWORLD of the landmark's
                                                   detection point (CFundamentalMatcher.h:27) */
} svi_landmarks;

typedef struct svi_track_result {
    uint8_t* status;     /* [n] svi_status of the LAST stage tried */
    uint8_t* stage;      /* [n] 0 = not tracked, 1 / 2 = stage 1 LEFT / RIGHT, 3 / 4 = stage 2 LEFT / RIGHT, 5 = stage 3 */
    float* uv_left;      /* [n*2] */
    float* uv_right;     /* [n*2] */
    double* xyz_left;    /* [n*3] */
    uint8_t* desc_left;  /* [n*32] */
    uint8_t* desc_right; /* [n*32] */
} svi_track_result;

/* CFundamentalMatcher::trackManual, the reference's first-success cascade
 * (src/core/CFundamentalMatcher.cpp:1404-1993): stage 1 LEFT / RIGHT (descriptor exactly at the rounded
 * projection), stage 2 LEFT / RIGHT (GFTT inside the projection window of half size
 * round(round(w + scaling) * 15), BRIEF on the window grown by 28 px, 1 x K match, cut-off 50) and stage 3
 * (one key-point per pixel along the epipolar line F * uvReference in LEFT, clipped to the box around the
 * projection, BRIEF, 1 x N match, cut-offs 50 / 100, one retry 2 px off the line; :1786-1993, :2142-2397),
 * each followed by the scan-line triangulation in the other image.
 * T_world_to_left is the row-major 4x4 of p_matTransformationWORLDtoLEFT. */
int svi_track_landmarks(svi_ctx* ctx, const uint8_t* img_left, const uint8_t* img_right,
                        size_t pitch, const double* T_world_to_left, const svi_landmarks* lm, int n,
                        double motion_scaling, svi_track_result* out);

/* The same cascade restricted to some of its stages -- what the SV/SVI trackers call separately:
 *   CFundamentalMatcher::getPoseStereoPosit (src/core/CFundamentalMatcher.cpp:338-757): stages 1 and 2 on the
 *     optimal landmarks, feeding CSolverStereoPosit                      -> SVI_STAGE_1 | SVI_STAGE_2
 *   CFundamentalMatcher::trackEpipolar (:760-1332): for landmarks not seen yet in this frame, the epipolar
 *     search when the camera moved since their detection (:828-1020)     -> SVI_STAGE_3
 *     and the regional search otherwise (:1022-1290)                     -> SVI_STAGE_2
 * SVI_STAGE_2 without SVI_STAGE_1 keeps the reference's gate "both projections inside the field of view"
 * (status SVI_TRK_OUT_OF_FOV otherwise); SVI_STAGE_3 alone has no gate but its own "projection out of sight".
 * SVI_STAGE_3 needs the three reference arrays of svi_landmarks. */
enum { SVI_STAGE_1 = 1, SVI_STAGE_2 = 2, SVI_STAGE_3 = 4 };
int svi_track_landmarks_stages(svi_ctx* ctx, const uint8_t* img_left, const uint8_t* img_right,
                        size_t pitch, const double* T_world_to_left, const svi_landmarks* lm, int n,
                        double motion_scaling, uint32_t stage_mask, svi_track_result* out);

/* ---- landmark position refinement, batched.
 * Replaces the loop of CFundamentalMatcher::optimizeActiveLandmarks (src/core/CFundamentalMatcher.cpp:265-277) over
 * CLandmark::optimize (src/types/CLandmark.cpp:281-296) / _getOptimizedLandmarkSTEREOUV (:447-581): for each of n
 * landmarks a robust Gauss-Newton refinement of its WORLD position on the stereo re-projection error of all its
 * measurements (constants of CLandmark.h:90-98: at most 1000 iterations, convergence 1e-5 on the total squared error,
 * kernel 10 px^2, inlier ratio > 0.5, optimal below 9 px^2 average).  Measurements of landmark i are the entries
 * [first[i], first[i + 1]) of the measurement arrays; a measurement names the pose it was taken with by its row in the two
 * projection tables (matProjectionWORLDtoLEFT / RIGHT of CMeasurementLandmark, Types.h:79-121: one row per frame, 3 x 4
 * row-major).  Landmarks with <= 5 measurements are skipped as the reference does (bIsOptimal = true).
 * One GPU thread per landmark, reference operation order, fp64 without contraction: the results equal the C++ host
 * implementation of the same loop bit for bit. */
enum svi_optimize_outcome {
    SVI_OPT_SKIPPED = 0,        /* <= 5 measurements: position untouched, bIsOptimal = true */
    SVI_OPT_CONVERGED = 1,      /* ++uOptimizationsSuccessful, position updated, not optimal (average error >= 9 px^2) */
    SVI_OPT_OPTIMAL = 2,        /* ++uOptimizationsSuccessful, position updated, bIsOptimal = true */
    SVI_OPT_REJECTED = 3,       /* converged with too few inliers: ++uOptimizationsFailed, position kept */
    SVI_OPT_NOT_CONVERGED = 4   /* iteration cap reached: ++uOptimizationsFailed, position kept */
};
typedef struct svi_landmark_measurements {
    const double* xyz_world_guess;      /* n x 3: vecPointXYZOptimized before the call */
    const int32_t* first;               /* n + 1 */
    const int32_t* pose_index;          /* m = first[n] */
    const float* uv_left;               /* m x 2 */
    const float* uv_right;              /* m x 2 */
    const double* proj_world_to_left;   /* n_poses x 12 */
    const double* proj_world_to_right;  /* n_poses x 12 */
    int32_t n_poses;
} svi_landmark_measurements;
typedef struct svi_optimize_result {
    double* xyz_world;                  /* n x 3: the refined position, or the guess where the outcome keeps it */
    uint8_t* outcome;                   /* n: svi_optimize_outcome */
    double* average_squared_error;      /* n: dCurrentAverageSquaredError of a converged landmark (0 otherwise) */
    int32_t* iterations;                /* n, may be NULL */
} svi_optimize_result;
int svi_optimize_landmarks(svi_ctx* ctx, const svi_landmark_measurements* in, int n, svi_optimize_result* out);

/* ---- pose from the stereo measurements of one frame.
 * CSolverStereoPosit::getTransformationWORLDtoLEFT (src/optimization/CSolverStereoPosit.cpp:8-170), what
 * CFundamentalMatcher::getPoseStereoPosit hands the measurements of tracking stages 1 and 2 to: robust Gauss-Newton on the
 * stereo re-projection error of the WORLD->LEFT pose from the prior T_estimate (constants of CSolverStereoPosit.h:89-99: more
 * than 25 points, at most 1000 iterations, convergence 1e-5 on the total squared error, kernel 10 px^2; a converged pose with
 * an average error above 9 px^2 AND fewer than 15 inliers is inaccurate; a translation within 1 mm (squared 0.001 m^2) of
 * T_last keeps T_last's translation; a camera position more than 2 m^2 (squared) away from the prior's plus t_imu is a high
 * risk).  The projection matrices are the P of the ctx's two cameras.  One launch, the whole iteration loop on the device,
 * fp64 without contraction in the host's operation order: the results equal the C++ host implementation of the same loop bit
 * for bit.  Per-problem failures are the outcome, not the return code; n <= 25 is answered without touching the GPU. */
enum svi_posit_outcome {
    SVI_POSIT_OK = 0,               /* T_world_to_left is the solution                                              */
    SVI_POSIT_TOO_FEW_POINTS = 1,   /* "insufficient number of points: <n>"                                          */
    SVI_POSIT_INACCURATE = 2,       /* "insufficient accuracy (average error: <average_squared_error> inliers: <inliers>)" */
    SVI_POSIT_HIGH_RISK = 3,        /* "inconsistent with prior (HIGH RISK: <risk>)"                                 */
    SVI_POSIT_NOT_CONVERGED = 4     /* "system did not converge" (1000 iterations)                                   */
};
typedef struct svi_posit_problem {   /* one frame's CSolverStereoPosit::CMatch list + the solver's other arguments */
    int32_t n;                       /* measurements                                                               */
    const double* xyz_world;         /* n x 3 vecPointXYZWORLD                                                     */
    const float* uv_left;            /* n x 2 ptUVLEFT                                                             */
    const float* uv_right;           /* n x 2 ptUVRIGHT                                                            */
    double T_estimate[16];           /* p_matTransformationWORLDtoLEFTESTIMATE, row-major                          */
    double T_last[16];               /* p_matTransformationWORLDtoLEFTLAST                                         */
    double t_imu[3];                 /* p_vecTranslationIMU                                                        */
} svi_posit_problem;
typedef struct svi_posit_result {
    double T_world_to_left[16];      /* the solution when SVI_POSIT_OK, else T_estimate                            */
    uint8_t outcome;                 /* svi_posit_outcome                                                          */
    int32_t iterations;              /* iterations run (0 for SVI_POSIT_TOO_FEW_POINTS)                            */
    int32_t inliers;                 /* inliers of the last iteration                                              */
    double average_squared_error;    /* of the converged iteration (0 if it did not converge)                      */
    double risk;                     /* squared distance to the prior's position (0 unless the risk test ran)      */
} svi_posit_result;
int svi_solve_stereo_posit(svi_ctx* ctx, const svi_posit_problem* in, svi_posit_result* out);

/* ---- one frame of the stereo-only tracker in one call.
 * CTrackerSV::process (src/core/CTrackerSV.cpp:143-172, :234-552) between the pose prior and the landmark bookkeeping, with exactly
 * the semantics of the composed calls CFundamentalMatcher::getPoseStereoPosit / trackEpipolar make:
 *   1. stages 1 and 2 (svi_track_landmarks_stages, SVI_STAGE_1 | SVI_STAGE_2) around T_estimate on the pose candidates (flags bit 0,
 *      in caller order), then svi_solve_stereo_posit on their hits in that order;
 *   2. if that solve fails, the same with T_estimate_damped; if that fails too, the pose is T_estimate_damped;
 *   3. every landmark that is neither a pose hit of an accepted solve nor flagged bit 1 goes to the epipolar stage: stage 3 alone
 *      when the translation of T_world_to_left * T_left_to_world_at_detection has a non-zero squared norm (evaluated as the host's
 *      Isometry3d::operator* and CFundamentalMatcher.h:561-563 do it: fp64, no contraction), else, and for stage-3 items that come
 *      back SVI_EPI_NO_TRANSLATION, stage 2 alone (the regional search, behind its field-of-view gate).
 * The images are staged (and rectified, while svi_set_rectification is set) once, the landmark arrays go up in one copy and the
 * results come back in one copy.  The subsets are index lists built on the device.  The host waits for the outcome of each solve
 * that runs (a few hundred bytes: one or two waits), once for the size of the regional set, and once at the end for the results. */
enum { SVI_SV_POSE_CANDIDATE = 1,   /* flags bit 0: bIsOptimal                                                           */
       SVI_SV_LEAVES = 2 };         /* flags bit 1: leaves in trackEpipolar (uOptimizationsFailed > 0, or
                                       uOptimizationsSuccessful > 0 && !bIsOptimal, :808-825)                             */
enum svi_sv_source { SVI_SV_POSIT = 0, SVI_SV_POSIT_DAMPED = 1, SVI_SV_PRIOR = 2 };
enum svi_sv_route {                 /* one per landmark                                                                  */
    SVI_SV_ROUTE_POSE = 1,          /* stage-1/2 hit of the accepted solve: measured in the pose stage (also if bit 1)    */
    SVI_SV_ROUTE_EPIPOLAR = 2,      /* stage 3                                                                           */
    SVI_SV_ROUTE_REGIONAL = 3,      /* stage 2: no translation since detection                                          */
    SVI_SV_ROUTE_REGIONAL_NO_TRANSLATION = 4, /* stage 2 after stage 3 returned SVI_EPI_NO_TRANSLATION                    */
    SVI_SV_ROUTE_DROPPED = 5        /* bit 1 and not a pose hit: not tracked                                             */
};
typedef struct svi_sv_frame {
    svi_landmarks landmarks;        /* all active landmarks, in the tracker's order; the three stage-3 arrays are required */
    const uint8_t* flags;           /* [n] SVI_SV_POSE_CANDIDATE | SVI_SV_LEAVES; other bits are refused                 */
    double T_estimate[16];          /* constant-velocity prior, row-major                                               */
    double T_estimate_damped[16];   /* rotation-only prior: the second attempt, and the pose when both solves fail       */
    double T_last[16];              /* pose of the previous frame (the solver's translation clamp)                      */
    double t_imu[3];                /* the solver's risk test                                                           */
    double motion_scaling;
} svi_sv_frame;
typedef struct svi_sv_frame_result {
    double T_world_to_left[16];     /* the frame's pose                                                                 */
    uint8_t source;                 /* svi_sv_source                                                                    */
    int32_t attempts;               /* solves that ran: 1 or 2                                                          */
    svi_posit_result attempt[2];    /* as svi_solve_stereo_posit returns them; fields an outcome does not compute are 0  */
    int32_t measurements[2];        /* stage-1/2 hits of each attempt: the problem size of its solve                    */
    svi_track_result pose_stage;    /* [n] stages 1-2 of the LAST attempt that ran (all zero for non-candidates)        */
    uint8_t* route;                 /* [n] svi_sv_route                                                                 */
    svi_track_result epipolar_stage; /* [n] stage 3 or the regional stage 2 (all zero where neither ran)                */
} svi_sv_frame_result;
int svi_track_frame_stereo_only(svi_ctx* ctx, const uint8_t* img_left, const uint8_t* img_right, size_t pitch, const svi_sv_frame* in, int n,
                                svi_sv_frame_result* out);

/* Stage profiling: when enabled, every kernel of the new-landmark path is bracketed by CUDA events
 * on the stream it is launched on (the events come from a pool filled here, none is created while
 * work is being timed).  enable = 1: the lanes keep overlapping, a bracket also contains other lanes'
 * kernels; enable = 2: svi_stereo_frames_device runs every chunk on ONE lane, so each bracket is the
 * exclusive duration of one kernel (what the roofline record uses -- slower overall, not for timing
 * the step).  svi_set_profiling also clears the accumulators; svi_stage_timings waits for the ctx to
 * go idle and returns, per stage, the summed launch duration in ms and the number of launches
 * (arrays of length >= 6; returns the stage count; "describe_left" has launches only on the batch path, where the LEFT descriptors are a kernel of their own ahead of the matcher, and "subpixel" only while svi_params.subpixel_window > 0; "lr_check", listed between "stereo_match" and "subpixel", is
 * listed only while svi_params.lr_max_diff >= 0, so the arrays need length >= 7 then and the count is 6 otherwise). */
int svi_set_profiling(svi_ctx* ctx, int enable);
int svi_stage_timings(svi_ctx* ctx, const char** names, double* total_ms, int64_t* launches, int capacity);

/* Frame-partitioned batches over the GPUs of one box (SURVEY.md 8e; stereo pairs are independent:
 * CFundamentalMatcher::addNewLandmarks keeps no state between pairs, src/core/CFundamentalMatcher.cpp:83-193,
 * CTriangulator is const).  svi_multi owns one svi_ctx per listed device (devices == NULL: 0 .. n_devices-1; a
 * device may be listed more than once).  svi_multi_stereo_frames cuts the n_frames pairs into contiguous ranges
 * [g*F/G, (g+1)*F/G) (svi_multi_frame_range), runs every range through its own ctx on its own host thread and
 * writes disjoint slices of the caller's host arrays -- no collective, no peer access; the outputs are
 * byte-for-byte those of svi_stereo_frames on one device.  Pinned host buffers keep the copies asynchronous. */
typedef struct svi_multi svi_multi;
int svi_multi_create(const svi_camera* left, const svi_camera* right, const svi_params* params,
                     const int* devices, int n_devices, svi_multi** out);
void svi_multi_destroy(svi_multi* m);
const char* svi_multi_last_error(const svi_multi* m); /* m may be NULL: last create error */
int svi_multi_device_count(const svi_multi* m);
int svi_multi_frame_range(const svi_multi* m, int n_frames, int part, int* first, int* count);
int svi_multi_stereo_frames(svi_multi* m, const uint8_t* left, const uint8_t* right, size_t pitch,
                            size_t frame_stride, int n_frames, const uint8_t* masks_or_null,
                            svi_stereo_result* out);

/* How this ctx was configured: frames per kernel wave, number of stream lanes, whether corner
 * selection runs out of shared memory (1) or the global-memory variant for very large frames (0). */
int svi_config(const svi_ctx* ctx, int32_t* chunk_frames, int32_t* n_lanes, int32_t* select_in_smem);

/* Number of kernels the new-landmark path launches for one chunk of a call with n_frames frames: 4 (detector, RIGHT box
 * sums, corner selection, matcher) on the small-call path, 5 when the LEFT descriptors are a kernel of their own (batch
 * path), 6 when the batch path also sorts the key-points into image bins (dense frames); one more while rectification is
 * set (svi_set_rectification); one more while svi_params.subpixel_window > 0; one more while svi_params.lr_max_diff >= 0.
 * For launch accounting. */
int svi_kernels_per_chunk(const svi_ctx* ctx, int n_frames);

/* ---- undistortion + rectification of raw camera images (CStereoCamera.h:102-107, CStereoCameraIMU.h:36-51: the reference
 * builds cv::initUndistortRectifyMap(matIntrinsic, vecDistortionCoefficients, matRectification, matProjection, (W, H), m1type)
 * per camera and runs cv::remap(raw, rectified, map1, map2, INTER_LINEAR) on every frame).  The new camera matrix is the
 * first 3 x 3 of the svi_camera's P the ctx was created with. */
typedef struct svi_rectification {
    double K[9];          /* matIntrinsic, row-major                                                      */
    double D[4];          /* vecDistortionCoefficients k1 k2 p1 p2                                        */
    double R[9];          /* matRectification, row-major                                                  */
    int32_t float_maps;   /* 0: maps as cv::initUndistortRectifyMap(..., CV_16SC2) (default)               */
                          /* 1: CV_32FC1 maps handed to cv::remap (which rounds float32(u) * 32, not u * 32) */
} svi_rectification;

/* The map of one camera in cv2's CV_16SC2 layout: xy = W x H x 2 int16 (integer source column, row), frac = W x H uint16
 * (5-bit row fraction * 32 + 5-bit column fraction).  Host only, needs no ctx and no GPU; the library builds its device
 * maps with this function.  SVI_ERR_INVALID for a singular K or P[:3,:3] * R (e.g. an all-zero matIntrinsic). */
int svi_rectify_map(const svi_camera* cam, const svi_rectification* r, int16_t* xy, uint16_t* frac);

/* Switches rectification on (both non-NULL) or off (both NULL) for every later call on ctx.  Waits for the ctx to go idle,
 * builds both maps, uploads them and allocates the raw-image staging once.  While it is set, EVERY image argument of every
 * entry point is a RAW image of the camera it belongs to -- svi_stereo_frames, svi_stereo_frames_device,
 * svi_stereo_frame_masked, svi_triangulate_right (RIGHT), svi_triangulate_left (LEFT), svi_track_landmarks[_stages], and
 * svi_harris_response / svi_detect / svi_describe (LEFT) -- and is rectified on the device with cv::remap(INTER_LINEAR,
 * BORDER_CONSTANT 0) arithmetic, bit for bit.  Masks, key-point coordinates and every other coordinate in and out stay in
 * the RECTIFIED frame.  Off (the default) costs nothing: no launch, copy or allocation. */
int svi_set_rectification(svi_ctx* ctx, const svi_rectification* left, const svi_rectification* right);

/* The rectified images themselves (display, key-frame images, inspection): n_frames raw host images of camera `side`
 * (0 = LEFT, 1 = RIGHT), height x pitch bytes, frame_stride apart -> n_frames rectified images of height x out_pitch
 * bytes, densely stacked.  Needs svi_set_rectification. */
int svi_rectify(svi_ctx* ctx, int side, const uint8_t* raw, size_t pitch, size_t frame_stride, int n_frames, uint8_t* out,
                size_t out_pitch);

/* svi_set_rectification on every context of the multi-GPU driver. */
int svi_multi_set_rectification(svi_multi* m, const svi_rectification* left, const svi_rectification* right);

#ifdef __cplusplus
}
#endif
#endif /* SVI_GPU_H */
