/* svi_oracle.c -- plain-C restatement of the reference's CPU algorithm for the stereo front-end
 * hot path.  TEST INFRASTRUCTURE: only tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline / --impl reference legs load this library; libsvi_gpu never does.
 *
 * It follows the reference call-for-call (paths relative to the svi_mapper tree):
 *   CFundamentalMatcher::addNewLandmarks                  src/core/CFundamentalMatcher.cpp:83-193
 *     cv::GFTTDetector(1000,0.01,7,7,true)::detect        :18,:101   -> svo_gftt (cornerHarris, minMaxLoc,
 *                                                                        threshold, dilate, sort, bucket grid)
 *     BriefDescriptorExtractor::compute(imgL, kps)        :106       -> svo_brief32 (integral image of the
 *                                                                        whole input, border filter, 256 tests)
 *     per key-point getPointTriangulatedInRIGHTFull       src/core/CTriangulator.cpp:51-119
 *       one BRIEF::compute on the 57-row ROI (its own integral image), one BFMatcher::match,
 *       cut-off, getPointInLEFT :326-356
 *   CTriangulator::getPointTriangulatedInLEFT (7 args)    src/core/CTriangulator.cpp:255-324
 *   CLandmark::optimize / _getOptimizedLandmarkSTEREOUV    src/types/CLandmark.cpp:281-296, :447-581 -> svo_optimize_landmark
 *   (CFundamentalMatcher::trackManual stages 1-3           src/core/CFundamentalMatcher.cpp:1334-2027 -> svo_track_landmarks)
 * OpenCV arithmetic (not in the reference tree, un-versioned "trunk") is restated from its
 * published algorithms in the operation order validated against cv2 4.13 with optimisations off
 * (SURVEY.md Appendix A); tests/test_oracle.py pins this file against cv2 and against the numpy
 * oracle.  BRIEF: PARITY UNPINNED at pair-table level (opencv_contrib generated_32.i is absent);
 * the table is svi_mapper_b200/csrc/brief_pattern_32.h, shared with the CUDA kernels.
 *
 * Per-frame work allocates and frees its buffers like the OpenCV calls it stands for, and one
 * frame is processed by one thread (cv::setNumThreads(1), src/core/CTrackerGT.cpp:48-49);
 * svo_stereo_frames_mt runs independent frames on several threads for the all-cores baseline. */
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#ifdef SVI_BRIEF_PATTERN_HEADER   /* another pair table (tools/gen_pattern_header.py --table ... --out ...) */
#include SVI_BRIEF_PATTERN_HEADER
#else
#include "../svi_mapper_b200/csrc/brief_pattern_32.h"
#endif

static const signed char kPat[SVI_BRIEF_NTESTS][4] = SVI_BRIEF_PATTERN_INIT;

enum { ST_OK = 0, ST_TRI_RANGE = 1, ST_TRI_NO_DESC = 2, ST_TRI_NO_MATCH = 3, ST_TRI_DISTANCE = 4,
       ST_TRI_ZERO_DISP = 5, ST_TRI_BAD_ROI = 6 };

typedef struct svo_config {
    int32_t width, height;
    double P_left[12], P_right[12];
    double quality_level, min_distance, harris_k, min_disparity;
    int32_t max_corners;
    float keypoint_size, search_range, match_cutoff;
} svo_config;

static inline int reflect101(int i, int n) {
    if (i < 0) i = -i;
    if (i >= n) i = 2 * n - 2 - i;
    return i;
}
/* REFLECT_101 for windows that may be narrower than the filter reach (cv::borderInterpolate loops the same way) */
static inline int reflect_n(int i, int n) {
    if (n == 1) return 0;
    while (i < 0 || i >= n) i = i < 0 ? -i : 2 * n - 2 - i;
    return i;
}

/* ------------------------------------------------------------------ cv::cornerHarris(img(roi), 7, 3, k) */
/* The window (rx, ry, rw, rh) of a w x h image, as OpenCV filters an ROI view without BORDER_ISOLATED
 * (GFTTDetector::detect(img(roi)), src/core/CFundamentalMatcher.cpp:1566): the Sobel filters read the parent image's
 * real pixels around the window (REFLECT_101 only at the parent's own edge), the 7x7 box filter runs on the freshly
 * allocated product planes and reflects at the WINDOW edge.  The whole image is the window (0, 0, w, h). */
static int harris_roi(const uint8_t* img, int w, int h, int pitch, int rx, int ry, int rw, int rh, double k, float* out) {
    const double scale = 1.0 / (4.0 * 7.0 * 255.0);
    const float f1 = (float)scale, f0 = (float)(2.0 * scale), kf = (float)k;
    const size_t n = (size_t)rw * rh;
    float* r = (float*)malloc(sizeof(float) * (size_t)rw * (rh + 2));  /* row-filtered planes, window rows -1..rh */
    float* q = (float*)malloc(sizeof(float) * (size_t)rw * (rh + 2));
    float* cov = (float*)malloc(sizeof(float) * 3 * n);
    double* hs = (double*)malloc(sizeof(double) * 3 * n);
    double* col = (double*)malloc(sizeof(double) * 3 * rw);
    if (!r || !q || !cov || !hs || !col) { free(r); free(q); free(cov); free(hs); free(col); return -1; }
    /* Sobel row pass on every source row incl. the two rows above / below the window */
    for (int yy = -1; yy <= rh; ++yy) {
        const uint8_t* p = img + (size_t)reflect101(ry + yy, h) * pitch;
        float* rr = r + (size_t)(yy + 1) * rw;
        float* qq = q + (size_t)(yy + 1) * rw;
        for (int x = 0; x < rw; ++x) {
            const int gx = rx + x;
            const float a = (float)p[reflect101(gx - 1, w)], b = (float)p[gx], c = (float)p[reflect101(gx + 1, w)];
            rr[x] = c - a;
            float t0 = a * f1, t1 = b * f0, t2 = c * f1;
            float s = t0 + t1;
            qq[x] = s + t2;
        }
    }
    /* column pass + products */
    for (int y = 0; y < rh; ++y) {
        const float *r0 = r + (size_t)y * rw, *r1 = r0 + rw, *r2 = r1 + rw;
        const float *q0 = q + (size_t)y * rw, *q2 = q0 + 2 * (size_t)rw;
        float* c = cov + (size_t)y * rw * 3;
        for (int x = 0; x < rw; ++x) {
            float s = r0[x] + r2[x];
            float m0 = s * f1, m1 = r1[x] * f0;
            float dx = m0 + m1;
            float dy = q2[x] - q0[x];
            c[3 * x] = dx * dx;
            c[3 * x + 1] = dx * dy;
            c[3 * x + 2] = dy * dy;
        }
    }
    /* boxFilter 7x7, normalize=false: RowSum<float,double> then ColumnSum<double,float>, REFLECT_101 at the window edge.
     * (a window narrower or lower than 4 px would need repeated reflection: reflect_n below folds until inside) */
    for (int y = 0; y < rh; ++y) {
        const float* c = cov + (size_t)y * rw * 3;
        double* d = hs + (size_t)y * rw * 3;
        for (int ch = 0; ch < 3; ++ch) {
            double s = 0;
            for (int i = -3; i <= 3; ++i) s += (double)c[3 * reflect_n(i, rw) + ch];
            d[ch] = s;
            for (int x = 0; x < rw - 1; ++x) {
                s += (double)c[3 * reflect_n(x + 4, rw) + ch] - (double)c[3 * reflect_n(x - 3, rw) + ch];
                d[3 * (x + 1) + ch] = s;
            }
        }
    }
    /* calcHarris runs over the response as one row of rw*rh pixels (both planes are continuous): 4-lane fp32 vectors with
     * (float)k, then a scalar tail for the last n % 4 pixels that evaluates (float)(a*c - b*b - k*(a+c)*(a+c)) with the
     * double k (a*c, b*b, det and a+c in fp32, the rest in fp64) */
    const size_t tail = n - n % 4;
    for (int i = 0; i < 3 * rw; ++i) col[i] = 0;
    for (int yy = -3; yy < 3; ++yy) {
        const double* d = hs + (size_t)reflect_n(yy, rh) * rw * 3;
        for (int i = 0; i < 3 * rw; ++i) col[i] += d[i];
    }
    for (int y = 0; y < rh; ++y) {
        const double* dp = hs + (size_t)reflect_n(y + 3, rh) * rw * 3;
        const double* dm = hs + (size_t)reflect_n(y - 3, rh) * rw * 3;
        float* o = out + (size_t)y * rw;
        for (int x = 0; x < rw; ++x) {
            double s0 = col[3 * x] + dp[3 * x], s1 = col[3 * x + 1] + dp[3 * x + 1], s2 = col[3 * x + 2] + dp[3 * x + 2];
            float a = (float)s0, b = (float)s1, c = (float)s2;
            col[3 * x] = s0 - dm[3 * x];
            col[3 * x + 1] = s1 - dm[3 * x + 1];
            col[3 * x + 2] = s2 - dm[3 * x + 2];
            float ac = a * c, bb = b * b;
            float det = ac - bb;
            float tr = a + c;
            if ((size_t)y * rw + x >= tail) {
                o[x] = (float)((double)det - k * (double)tr * (double)tr);
                continue;
            }
            float kt = kf * tr;
            float ktt = kt * tr;
            o[x] = det - ktt;
        }
    }
    free(r); free(q); free(cov); free(hs); free(col);
    return 0;
}

int svo_harris_response(const uint8_t* img, int w, int h, int pitch, double k, float* out) {
    return harris_roi(img, w, h, pitch, 0, 0, w, h, k, out);
}

int svo_harris_response_roi(const uint8_t* img, int w, int h, int pitch, int rx, int ry, int rw, int rh, double k, float* out) {
    if (rx < 0 || ry < 0 || rw <= 0 || rh <= 0 || rx + rw > w || ry + rh > h) return -1;
    return harris_roi(img, w, h, pitch, rx, ry, rw, rh, k, out);
}

/* ------------------------------------------------------------------ cv::goodFeaturesToTrack (Harris) */
typedef struct { float v; int32_t addr; } cand_t;
static int cand_cmp(const void* pa, const void* pb) {
    const cand_t *a = (const cand_t*)pa, *b = (const cand_t*)pb;
    if (a->v > b->v) return -1;
    if (a->v < b->v) return 1;
    return (a->addr > b->addr) ? -1 : (a->addr < b->addr);
}

/* goodFeaturesToTrack after cornerHarris: `eig` (w x h floats, consumed) -> corners */
static int gftt_select(float* eig, int w, int h, const uint8_t* mask, int mask_pitch, int max_corners, double quality,
                       double min_distance, int32_t* xy, int cap) {
    const size_t n = (size_t)w * h;
    float* dil = (float*)malloc(sizeof(float) * n);
    if (!dil) { free(eig); return -1; }
    /* minMaxLoc over the mask */
    double max_val = 0;
    int have = 0;
    for (int y = 0; y < h; ++y)
        for (int x = 0; x < w; ++x)
            if (!mask || mask[(size_t)y * mask_pitch + x]) {
                float v = eig[(size_t)y * w + x];
                if (!have || v > max_val) { max_val = v; have = 1; }
            }
    /* threshold(eig, eig, maxVal*quality, 0, THRESH_TOZERO) */
    const float thr = (float)(max_val * quality);
    for (size_t i = 0; i < n; ++i) eig[i] = eig[i] > thr ? eig[i] : 0.f;
    /* dilate 3x3 */
    for (int y = 0; y < h; ++y)
        for (int x = 0; x < w; ++x) {
            float m = eig[(size_t)y * w + x];
            for (int dy = -1; dy <= 1; ++dy) {
                int yy = y + dy;
                if (yy < 0 || yy >= h) continue;
                for (int dx = -1; dx <= 1; ++dx) {
                    int xx = x + dx;
                    if (xx < 0 || xx >= w) continue;
                    float v = eig[(size_t)yy * w + xx];
                    if (v > m) m = v;
                }
            }
            dil[(size_t)y * w + x] = m;
        }
    size_t nc = 0, ccap = 4096;
    cand_t* c = (cand_t*)malloc(sizeof(cand_t) * ccap);
    for (int y = 1; y < h - 1; ++y)
        for (int x = 1; x < w - 1; ++x) {
            float v = eig[(size_t)y * w + x];
            if (v != 0 && v == dil[(size_t)y * w + x] && (!mask || mask[(size_t)y * mask_pitch + x])) {
                if (nc == ccap) { ccap *= 2; c = (cand_t*)realloc(c, sizeof(cand_t) * ccap); }
                c[nc].v = v;
                c[nc].addr = y * w + x;
                ++nc;
            }
        }
    free(eig); free(dil);
    qsort(c, nc, sizeof(cand_t), cand_cmp);
    int count = 0;
    if (min_distance >= 1) {
        const int cell = (int)lround(min_distance);
        const int gw = (w + cell - 1) / cell, gh = (h + cell - 1) / cell;
        int32_t* head = (int32_t*)malloc(sizeof(int32_t) * gw * gh);
        int32_t* next = (int32_t*)malloc(sizeof(int32_t) * (nc ? nc : 1));
        for (int i = 0; i < gw * gh; ++i) head[i] = -1;
        const double md2 = min_distance * min_distance;
        for (size_t i = 0; i < nc; ++i) {
            const int y = c[i].addr / w, x = c[i].addr - y * w;
            const int cx = x / cell, cy = y / cell;
            int good = 1;
            for (int yy = (cy > 0 ? cy - 1 : 0); good && yy <= (cy + 1 < gh ? cy + 1 : gh - 1); ++yy)
                for (int xx = (cx > 0 ? cx - 1 : 0); good && xx <= (cx + 1 < gw ? cx + 1 : gw - 1); ++xx)
                    for (int32_t j = head[yy * gw + xx]; j >= 0; j = next[j]) {
                        float dx = (float)(x - xy[2 * j]), dy = (float)(y - xy[2 * j + 1]);
                        if ((double)(dx * dx + dy * dy) < md2) { good = 0; break; }
                    }
            if (good) {
                if (count >= cap) break;
                xy[2 * count] = x;
                xy[2 * count + 1] = y;
                next[count] = head[cy * gw + cx];
                head[cy * gw + cx] = count;
                ++count;
                if (max_corners > 0 && count == max_corners) break;
            }
        }
        free(head); free(next);
    } else {
        for (size_t i = 0; i < nc && count < cap; ++i) {
            xy[2 * count] = c[i].addr % w;
            xy[2 * count + 1] = c[i].addr / w;
            ++count;
            if (max_corners > 0 && count == max_corners) break;
        }
    }
    free(c);
    return count;
}

int svo_gftt(const uint8_t* img, int w, int h, int pitch, const uint8_t* mask, int mask_pitch, int max_corners,
             double quality, double min_distance, double k, int32_t* xy, int cap) {
    float* eig = (float*)malloc(sizeof(float) * (size_t)w * h);
    if (!eig || svo_harris_response(img, w, h, pitch, k, eig) != 0) { free(eig); return -1; }
    return gftt_select(eig, w, h, mask, mask_pitch, max_corners, quality, min_distance, xy, cap);
}

/* GFTTDetector::detect(img(roi)): corners in window coordinates */
int svo_gftt_roi(const uint8_t* img, int w, int h, int pitch, int rx, int ry, int rw, int rh, int max_corners, double quality,
                 double min_distance, double k, int32_t* xy, int cap) {
    if (rw <= 0 || rh <= 0) return 0;
    float* eig = (float*)malloc(sizeof(float) * (size_t)rw * rh);
    if (!eig || svo_harris_response_roi(img, w, h, pitch, rx, ry, rw, rh, k, eig) != 0) { free(eig); return -1; }
    return gftt_select(eig, rw, rh, NULL, 0, max_corners, quality, min_distance, xy, cap);
}

/* ------------------------------------------------------------------ BriefDescriptorExtractor(32)::compute */
static inline long lrint_half_even(float v) { return lrintf(v); } /* cvRound, default rounding mode */

/* `img` is the (ROI) image BRIEF is called on: its own integral image is built here, as OpenCV does.
 * Returns the number of kept key-points; kept[i] = index into pts of the i-th surviving one. */
int svo_brief32(const uint8_t* img, int w, int h, int pitch, const float* pts, int n, uint8_t* desc, int32_t* kept) {
    int nk = 0;
    if (w <= 56 || h <= 56) return 0;
    for (int i = 0; i < n; ++i) {
        long rx = lrint_half_even(pts[2 * i]), ry = lrint_half_even(pts[2 * i + 1]);
        /* x.5 coordinates: cvRound and the sampling centre (int)(pt+0.5) can differ by one and the reference then
         * reads outside its integral image (undefined); defined here: such a key-point is erased */
        const int sx = (int)(pts[2 * i] + 0.5), sy = (int)(pts[2 * i + 1] + 0.5);
        if (rx >= 28 && rx < w - 28 && ry >= 28 && ry < h - 28 && sx >= 28 && sx < w - 28 && sy >= 28 && sy < h - 28) kept[nk++] = i;
    }
    if (!nk) return 0;
    const int sw = w + 1;
    int32_t* sum = (int32_t*)malloc(sizeof(int32_t) * (size_t)sw * (h + 1));
    if (!sum) return -1;
    memset(sum, 0, sizeof(int32_t) * sw);
    for (int y = 0; y < h; ++y) {
        const uint8_t* p = img + (size_t)y * pitch;
        int32_t* s = sum + (size_t)(y + 1) * sw;
        const int32_t* sp = s - sw;
        int32_t run = 0;
        s[0] = 0;
        for (int x = 0; x < w; ++x) { run += p[x]; s[x + 1] = sp[x + 1] + run; }
    }
    for (int kk = 0; kk < nk; ++kk) {
        const float* pt = pts + 2 * kept[kk];
        const int cx = (int)(pt[0] + 0.5), cy = (int)(pt[1] + 0.5);
        uint8_t* d = desc + (size_t)kk * 32;
        for (int j = 0; j < 32; ++j) {
            unsigned byte = 0;
            for (int i = 0; i < 8; ++i) {
                const signed char* t = kPat[8 * j + i];
                int y1 = cy + t[0], x1 = cx + t[1], y2 = cy + t[2], x2 = cx + t[3];
                int32_t s1 = sum[(size_t)(y1 + 5) * sw + x1 + 5] - sum[(size_t)(y1 + 5) * sw + x1 - 4] -
                             sum[(size_t)(y1 - 4) * sw + x1 + 5] + sum[(size_t)(y1 - 4) * sw + x1 - 4];
                int32_t s2 = sum[(size_t)(y2 + 5) * sw + x2 + 5] - sum[(size_t)(y2 + 5) * sw + x2 - 4] -
                             sum[(size_t)(y2 - 4) * sw + x2 + 5] + sum[(size_t)(y2 - 4) * sw + x2 - 4];
                byte |= (unsigned)(s1 < s2) << (7 - i);
            }
            d[j] = (uint8_t)byte;
        }
    }
    free(sum);
    return nk;
}

/* ------------------------------------------------------------------ BFMatcher(NORM_HAMMING)::match, 1 x N */
int svo_match(const uint8_t* q, const uint8_t* t, int n, int32_t* dist_out) {
    int best = -1, bd = 1 << 30;
    uint64_t qa[4];
    memcpy(qa, q, 32);
    for (int i = 0; i < n; ++i) {
        uint64_t ta[4];
        memcpy(ta, t + (size_t)i * 32, 32);
        int d = __builtin_popcountll(qa[0] ^ ta[0]) + __builtin_popcountll(qa[1] ^ ta[1]) +
                __builtin_popcountll(qa[2] ^ ta[2]) + __builtin_popcountll(qa[3] ^ ta[3]);
        if (d < bd) { bd = d; best = i; }
    }
    *dist_out = best >= 0 ? bd : -1;
    return best;
}

/* ------------------------------------------------------------------ CTriangulator */
typedef struct { double f_inv, pu, pv, du_r, du_r_flipped, min_disp; float width; float cutoff; } tri_t;

static void tri_init(tri_t* t, const svo_config* c) {
    t->f_inv = 1.0 / c->P_left[0];
    t->pu = c->P_left[2];
    t->pv = c->P_left[6];
    t->du_r = c->P_right[3];
    t->du_r_flipped = -t->du_r;
    t->min_disp = c->min_disparity;
    t->width = (float)c->width;
    t->cutoff = c->match_cutoff;
}

int svo_point_in_left(const svo_config* c, const float* uvl, const float* uvr, double* xyz) {
    tri_t t;
    tri_init(&t, c);
    const float d = uvl[0] - uvr[0];
    if ((double)d < t.min_disp) return ST_TRI_ZERO_DISP;
    const double z = t.du_r_flipped / (double)d;
    const double fz = t.f_inv * z;
    xyz[0] = fz * ((double)uvl[0] - t.pu);
    xyz[1] = fz * ((double)uvl[1] - t.pv);
    xyz[2] = z;
    return ST_OK;
}

/* shared body of CTriangulator.cpp:59-117 / :264-322 */
static int search(const svo_config* c, const uint8_t* img, int pitch, float u_tl, float v_tl, float size, int first,
                  int n_pool, const uint8_t* ref, float* uv, uint8_t* desc_out, int32_t* dist, int32_t* idx) {
    const float border = 4 * size, full_h = 8 * size + 1;
    float wroi = (float)n_pool + full_h;
    const float wmax = (float)c->width - u_tl;
    if (wmax < wroi) wroi = wmax;
    const int rx = (int)u_tl, ry = (int)v_tl, rw = (int)wroi, rh = (int)full_h;
    *dist = -1;
    *idx = -1;
    if (rx < 0 || ry < 0 || rw < 0 || rh < 0 || rx + rw > c->width || ry + rh > c->height) return ST_TRI_BAD_ROI;
    if (n_pool <= 0) return ST_TRI_NO_DESC;
    float* pool = (float*)malloc(sizeof(float) * 2 * n_pool);
    uint8_t* pd = (uint8_t*)malloc((size_t)32 * n_pool);
    int32_t* kept = (int32_t*)malloc(sizeof(int32_t) * n_pool);
    for (int i = 0; i < n_pool; ++i) {
        pool[2 * i] = (border + (float)i) + (float)first;
        pool[2 * i + 1] = border;
    }
    const int nk = svo_brief32(img + (size_t)ry * pitch + rx, rw, rh, pitch, pool, n_pool, pd, kept);
    int st;
    if (nk <= 0) st = ST_TRI_NO_DESC;
    else {
        int32_t d;
        const int m = svo_match(ref, pd, nk, &d);
        if (m < 0) st = ST_TRI_NO_MATCH;
        else {
            *dist = d;
            *idx = m;
            if (c->match_cutoff > (float)d) {
                uv[0] = pool[2 * kept[m]] + u_tl;
                uv[1] = pool[2 * kept[m] + 1] + v_tl;
                memcpy(desc_out, pd + (size_t)m * 32, 32);
                st = ST_OK;
            } else st = ST_TRI_DISTANCE;
        }
    }
    free(pool); free(pd); free(kept);
    return st;
}

int svo_triangulate_right(const svo_config* c, const uint8_t* img_r, int pitch, float u_tl, float v_tl, float size,
                          const float* uvl, const uint8_t* desc_l, float* uv, double* xyz, uint8_t* desc, int32_t* dist,
                          int32_t* idx) {
    const float border = 4 * size;
    *dist = -1;
    *idx = -1;
    if (uvl[0] <= u_tl + border) return ST_TRI_RANGE;
    const int n_pool = (int)ceilf(uvl[0] - u_tl - border);
    int st = search(c, img_r, pitch, u_tl, v_tl, size, 0, n_pool, desc_l, uv, desc, dist, idx);
    if (st == ST_OK) st = svo_point_in_left(c, uvl, uv, xyz);
    return st;
}

int svo_triangulate_left(const svo_config* c, const uint8_t* img_l, int pitch, float search_range, float u_tl, float v_tl,
                         float size, const float* uvr, const uint8_t* desc_r, float* uv, double* xyz, uint8_t* desc,
                         int32_t* dist, int32_t* idx) {
    *dist = -1;
    *idx = -1;
    if (0 >= search_range) return ST_TRI_RANGE;
    float m = search_range;
    const float wl = (float)c->width - u_tl;
    if (wl < m) m = wl;
    const int n_pool = (int)ceilf(m) + 1;
    int st = search(c, img_l, pitch, u_tl, v_tl, size, 1, n_pool, desc_r, uv, desc, dist, idx);
    if (st == ST_OK) st = svo_point_in_left(c, uv, uvr, xyz);
    return st;
}

/* ------------------------------------------------------------------ addNewLandmarks, one pair */
typedef struct svo_result {
    int32_t capacity;
    float* uv_left; float* uv_right; double* xyz_left; uint8_t* desc_left; uint8_t* desc_right;
    int32_t* distance; int32_t* match_index; uint8_t* status;
} svo_result;

int svo_add_new_landmarks(const svo_config* c, const uint8_t* left, const uint8_t* right, int pitch, const uint8_t* mask,
                          const svo_result* out, size_t o0, int32_t* n_detected) {
    const int cap = c->max_corners > 0 ? c->max_corners : out->capacity;
    int32_t* xy = (int32_t*)malloc(sizeof(int32_t) * 2 * cap);
    const int nd = svo_gftt(left, c->width, c->height, pitch, mask, pitch, c->max_corners, c->quality_level, c->min_distance,
                            c->harris_k, xy, cap);
    if (nd < 0) { free(xy); return -1; }
    if (n_detected) *n_detected = nd;
    float* pts = (float*)malloc(sizeof(float) * 2 * (nd ? nd : 1));
    int32_t* kept = (int32_t*)malloc(sizeof(int32_t) * (nd ? nd : 1));
    uint8_t* dl = (uint8_t*)malloc((size_t)32 * (nd ? nd : 1));
    for (int i = 0; i < nd; ++i) { pts[2 * i] = (float)xy[2 * i]; pts[2 * i + 1] = (float)xy[2 * i + 1]; }
    const int nk = svo_brief32(left, c->width, c->height, pitch, pts, nd, dl, kept);
    const float size = c->keypoint_size;
    for (int u = 0; u < nk && u < out->capacity; ++u) {
        const size_t o = o0 + u;
        const float x = pts[2 * kept[u]], y = pts[2 * kept[u] + 1];
        float u_tl = x - c->search_range - 4 * size;
        if (u_tl < 0.0f) u_tl = 0.0f;
        const float v_tl = y - 4 * size;
        float uvl[2] = {x, y}, uvr[2] = {0, 0};
        double xyz[3] = {0, 0, 0};
        uint8_t dr[32];
        int32_t dist, idx;
        memset(dr, 0, 32);
        const int st = svo_triangulate_right(c, right, pitch, u_tl, v_tl, size, uvl, dl + (size_t)u * 32, uvr, xyz, dr, &dist, &idx);
        out->uv_left[2 * o] = x; out->uv_left[2 * o + 1] = y;
        memcpy(out->desc_left + o * 32, dl + (size_t)u * 32, 32);
        out->status[o] = (uint8_t)st;
        out->distance[o] = dist;
        out->match_index[o] = idx;
        if (st == ST_OK) {
            out->uv_right[2 * o] = uvr[0]; out->uv_right[2 * o + 1] = uvr[1];
            out->xyz_left[3 * o] = xyz[0]; out->xyz_left[3 * o + 1] = xyz[1]; out->xyz_left[3 * o + 2] = xyz[2];
            memcpy(out->desc_right + o * 32, dr, 32);
        }
    }
    free(xy); free(pts); free(kept); free(dl);
    return nk;
}

/* ------------------------------------------------------------------ batch driver (frame-parallel) */
typedef struct {
    const svo_config* c; const uint8_t* left; const uint8_t* right; const uint8_t* masks;
    int pitch; size_t stride; int n_frames; const svo_result* out; int32_t* n_kp; int32_t* n_det;
    int next; pthread_mutex_t mu; int error;
} job_t;

static void* worker(void* arg) {
    job_t* j = (job_t*)arg;
    for (;;) {
        pthread_mutex_lock(&j->mu);
        const int f = j->next++;
        pthread_mutex_unlock(&j->mu);
        if (f >= j->n_frames) break;
        int32_t nd = 0;
        const int nk = svo_add_new_landmarks(j->c, j->left + f * j->stride, j->right + f * j->stride, j->pitch,
                                             j->masks ? j->masks + f * j->stride : NULL, j->out,
                                             (size_t)f * j->out->capacity, &nd);
        if (nk < 0) j->error = 1;
        j->n_kp[f] = nk;
        if (j->n_det) j->n_det[f] = nd;
    }
    return NULL;
}

int svo_stereo_frames_mt(const svo_config* c, const uint8_t* left, const uint8_t* right, int pitch, size_t frame_stride,
                         int n_frames, const uint8_t* masks, const svo_result* out, int32_t* n_keypoints,
                         int32_t* n_detected, int n_threads) {
    job_t j;
    j.c = c; j.left = left; j.right = right; j.masks = masks; j.pitch = pitch; j.stride = frame_stride;
    j.n_frames = n_frames; j.out = out; j.n_kp = n_keypoints; j.n_det = n_detected; j.next = 0; j.error = 0;
    pthread_mutex_init(&j.mu, NULL);
    if (n_threads < 1) n_threads = 1;
    if (n_threads > n_frames) n_threads = n_frames > 0 ? n_frames : 1;
    pthread_t* th = (pthread_t*)malloc(sizeof(pthread_t) * n_threads);
    for (int i = 1; i < n_threads; ++i) pthread_create(&th[i], NULL, worker, &j);
    worker(&j);
    for (int i = 1; i < n_threads; ++i) pthread_join(th[i], NULL);
    free(th);
    pthread_mutex_destroy(&j.mu);
    return j.error ? -1 : 0;
}

/* ================================================================== CFundamentalMatcher::trackManual
 * src/core/CFundamentalMatcher.cpp:1334-2027 restated per landmark, call for call:
 *   stage 1 LEFT / RIGHT   :1404-1538   descriptor exactly at the rounded projection (one BRIEF::compute on the
 *                                       (8*size+1)^2 ROI), cut-off 25, scan-line triangulation in the other image
 *   stage 2 LEFT / RIGHT   :1545-1785   GFTTDetector::detect on the projection window, BRIEF on the window grown by
 *                                       4*size, 1 x K match, cut-off 50, triangulation
 *   stage 3                :1786-1993   epipolar line F * uvReference in LEFT, _getMatchSampleRecursiveU/V + _getMatch
 *                                       (:2142-2397), cut-offs 50 / 100, one retry 2 px off the line,
 *                                       _addMeasurementToLandmarkLEFT (:2399-2453)
 * and getPoseStereoPosit (:338-757) / trackEpipolar (:760-1332) as subsets of the same cascade (stage_mask).
 * Status values: include/svi_gpu.h svi_status.  The arithmetic (float / double, operation order, roundings) is the one
 * oracle/frontend_np.py states line by line; tests/test_oracle.py pins this file against it. */
enum { ST_TRK_DEPTH = 7, ST_TRK_STAGE1_DIST = 8, ST_TRK_TRI_DESC = 9, ST_TRK_OUT_OF_FOV = 10, ST_TRK_NO_FEATURES = 11,
       ST_TRK_NO_MATCHES = 12, ST_TRK_DESC = 13, ST_TRK_RANGE = 14, ST_EPI_OUT_OF_SIGHT = 15, ST_EPI_VERTICAL = 16,
       ST_EPI_NEG_SLOPE = 17, ST_EPI_POS_SLOPE = 18, ST_EPI_ZERO_LEN = 19, ST_EPI_POOL_EMPTY = 20, ST_EPI_NO_MATCHES = 21,
       ST_EPI_DIST = 22, ST_EPI_ORIG_DIST = 23, ST_EPI_NO_TRANSLATION = 24 };

typedef struct svo_track_params {
    float cutoff_stage1, cutoff_stage2, cutoff_stage3, cutoff_original;   /* 25 / 50 / 50 / 100  :23-26 */
    double epipolar_base_length;                                          /* 15  CFundamentalMatcher.h:92 */
    int32_t block_size_stage2;                                            /* 15  CFundamentalMatcher.h:95 */
} svo_track_params;

typedef struct svo_landmarks {
    const double* xyz_world; const uint8_t* last_desc_left; const uint8_t* last_desc_right;
    const float* last_disparity; const float* keypoint_size;
    const double* uv_reference_left; const uint8_t* desc_reference_left; const double* T_left_to_world_at_detection;
} svo_landmarks;

typedef struct svo_track_result {
    uint8_t* status; uint8_t* stage; float* uv_left; float* uv_right; double* xyz_left; uint8_t* desc_left; uint8_t* desc_right;
} svo_track_result;

static int hamming32(const uint8_t* a, const uint8_t* b) {
    uint64_t x[4], y[4];
    memcpy(x, a, 32);
    memcpy(y, b, 32);
    return __builtin_popcountll(x[0] ^ y[0]) + __builtin_popcountll(x[1] ^ y[1]) + __builtin_popcountll(x[2] ^ y[2]) +
           __builtin_popcountll(x[3] ^ y[3]);
}

/* CPinholeCamera::getProjectionRounded (src/vision/CPinholeCamera.h:202-210): std::round on the float quotient */
static void projection_rounded(const double* P, const double* p, float* u, float* v) {
    const double h0 = ((P[0] * p[0] + P[1] * p[1]) + P[2] * p[2]) + P[3];
    const double h1 = ((P[4] * p[0] + P[5] * p[1]) + P[6] * p[2]) + P[7];
    const double h2 = ((P[8] * p[0] + P[9] * p[1]) + P[10] * p[2]) + P[11];
    *u = roundf((float)(h0 / h2));
    *v = roundf((float)(h1 / h2));
}
static int fov_contains(const svo_config* c, float u, float v) {   /* m_cFieldOfView(28, 28, W-56, H-56) :61 */
    return u >= 28.f && u < (float)(c->width - 28) && v >= 28.f && v < (float)(c->height - 28);
}
static void to_camera(const double* T, const double* w, double* p) {   /* Isometry3d * Vector3d */
    for (int r = 0; r < 3; ++r) p[r] = ((T[4 * r] * w[0] + T[4 * r + 1] * w[1]) + T[4 * r + 2] * w[2]) + T[4 * r + 3];
}

typedef struct { float uv_l[2], uv_r[2]; double xyz[3]; uint8_t desc_l[32], desc_r[32]; int stage; } track_hit;

/* BRIEF at the single key-point (half, half) of the (8*size+1)^2 ROI whose corner is (roi_x, roi_y) (:1423-1428) */
static int describe_at_projection(const svo_config* c, const uint8_t* img, int pitch, float roi_x, float roi_y, float size,
                                  uint8_t* desc, int* roi_ok) {
    const int len = (int)(8.f * size + 1.f), rx = (int)roi_x, ry = (int)roi_y;
    *roi_ok = rx >= 0 && ry >= 0 && rx + len <= c->width && ry + len <= c->height;
    if (!*roi_ok) return 0;
    const float pt[2] = {4.f * size, 4.f * size};
    int32_t kept;
    return svo_brief32(img + (size_t)ry * pitch + rx, len, len, pitch, pt, 1, desc, &kept) == 1;
}

static int depth_ok(const svo_config* c, double z) {
    const double du = -c->P_right[3];
    return !(du / (double)c->width > z || du / c->min_disparity < z);
}

/* stage 1, both sides; returns the status of the last attempt, fills *hit on success */
static int track_stage1(const svo_config* c, const svo_track_params* tp, const uint8_t* img_l, const uint8_t* img_r, int pitch,
                        float ul, float vl, float ur, float vr, float size, float search, const uint8_t* last_l,
                        const uint8_t* last_r, track_hit* hit) {
    const float half = 4.f * size;
    uint8_t d[32], dr[32];
    float uv[2];
    double xyz[3];
    int32_t dist, idx;
    int st, roi_ok;
    {   /* LEFT :1419-1476 */
        const float roi_x = ul - half, roi_y = vl - half;
        const int have = describe_at_projection(c, img_l, pitch, roi_x, roi_y, size, d, &roi_ok);
        st = roi_ok ? ST_TRK_STAGE1_DIST : ST_TRI_BAD_ROI;
        if (have && tp->cutoff_stage1 > (float)hamming32(last_l, d)) {
            float u_tl = roi_x - search;
            if (u_tl < 0.f) u_tl = 0.f;
            const float uvl[2] = {roi_x + half, roi_y + half};
            st = svo_triangulate_right(c, img_r, pitch, u_tl, roi_y, size, uvl, d, uv, xyz, dr, &dist, &idx);
            if (st == ST_OK) {
                if (!depth_ok(c, xyz[2])) st = ST_TRK_DEPTH;
                else if (tp->cutoff_stage1 < (float)hamming32(last_r, dr)) st = ST_TRK_TRI_DESC;
                else {
                    hit->stage = 1;
                    hit->uv_l[0] = ul; hit->uv_l[1] = vl; hit->uv_r[0] = uv[0]; hit->uv_r[1] = uv[1];
                    memcpy(hit->xyz, xyz, sizeof(xyz)); memcpy(hit->desc_l, d, 32); memcpy(hit->desc_r, dr, 32);
                    return ST_OK;
                }
            }
        }
    }
    {   /* RIGHT :1480-1538 */
        const float roi_x = ur - half, roi_y = vr - half;
        const int have = describe_at_projection(c, img_r, pitch, roi_x, roi_y, size, d, &roi_ok);
        st = roi_ok ? ST_TRK_STAGE1_DIST : ST_TRI_BAD_ROI;
        if (have && tp->cutoff_stage1 > (float)hamming32(last_r, d)) {
            const float uvr[2] = {roi_x + half, roi_y + half};
            st = svo_triangulate_left(c, img_l, pitch, search, roi_x, roi_y, size, uvr, d, uv, xyz, dr, &dist, &idx);
            if (st == ST_OK) {
                if (!depth_ok(c, xyz[2])) st = ST_TRK_DEPTH;
                else if (tp->cutoff_stage1 < (float)hamming32(last_l, dr)) st = ST_TRK_TRI_DESC;
                else {
                    hit->stage = 2;
                    hit->uv_l[0] = uv[0]; hit->uv_l[1] = uv[1]; hit->uv_r[0] = ur; hit->uv_r[1] = vr;
                    memcpy(hit->xyz, xyz, sizeof(xyz)); memcpy(hit->desc_l, dr, 32); memcpy(hit->desc_r, d, 32);
                    return ST_OK;
                }
            }
        }
    }
    return st;
}

static long cv_round_f(float v) { return lrintf(v); }   /* saturate_cast<int>(float) = cvRound, half to even */

/* one side of stage 2 (LEFT :1545-1665, RIGHT :1669-1785) */
static int track_stage2_side(const svo_config* c, const svo_track_params* tp, const uint8_t* img_this, const uint8_t* img_other,
                             int pitch, const double* P_this, float u, float v, const uint8_t* last_this,
                             const uint8_t* last_other, float search, float size, double motion_scaling, int left, track_hit* hit) {
    const float half = 4.f * size;
    const int W = c->width, H = c->height;
    /* :1548-1558 half sizes round(round(w + scaling) * block), corners clamped, cv::Rect(Point2f, Point2f) */
    const double wu = sqrt(fabs((double)u - P_this[2])) / 10.0, wv = sqrt(fabs((double)v - P_this[6])) / 10.0;
    const double hw = round(round(wu + motion_scaling) * tp->block_size_stage2), hh = round(round(wv + motion_scaling) * tp->block_size_stage2);
    const float ul_x = (float)fmax((double)u - hw, 0.0), ul_y = (float)fmax((double)v - hh, 0.0);
    const float lr_x = (float)fmin((double)u + hw, (double)W), lr_y = (float)fmin((double)v + hh, (double)H);
    const int rx = (int)cv_round_f(ul_x), ry = (int)cv_round_f(ul_y);
    const int rw = (int)cv_round_f(lr_x) - rx, rh = (int)cv_round_f(lr_y) - ry;
    if (rw <= 0 || rh <= 0 || rx < 0 || ry < 0 || rx + rw > W || ry + rh > H) return ST_TRK_NO_FEATURES;
    const int cap = c->max_corners > 0 ? c->max_corners : rw * rh;
    int32_t* xy = (int32_t*)malloc(sizeof(int32_t) * 2 * (size_t)cap);
    const int nd = svo_gftt_roi(img_this, W, H, pitch, rx, ry, rw, rh, c->max_corners, c->quality_level, c->min_distance, c->harris_k, xy, cap);   /* :1566 */
    if (nd <= 0) { free(xy); return ST_TRK_NO_FEATURES; }
    /* :1572-1575 window grown by 4*size and clamped */
    const float g_ulx = fmaxf(ul_x - half, 0.f), g_uly = fmaxf(ul_y - half, 0.f);
    const float g_lrx = fminf(lr_x + half, (float)W), g_lry = fminf(lr_y + half, (float)H);
    const int gx = (int)cv_round_f(g_ulx), gy = (int)cv_round_f(g_uly);
    const int gw = (int)cv_round_f(g_lrx) - gx, gh = (int)cv_round_f(g_lry) - gy;
    float* pts = (float*)malloc(sizeof(float) * 2 * (size_t)nd);
    uint8_t* desc = (uint8_t*)malloc((size_t)32 * nd);
    int32_t* kept = (int32_t*)malloc(sizeof(int32_t) * (size_t)nd);
    for (int i = 0; i < nd; ++i) { pts[2 * i] = (float)xy[2 * i] + half; pts[2 * i + 1] = (float)xy[2 * i + 1] + half; }   /* :1579 */
    const int nk = (gw > 0 && gh > 0) ? svo_brief32(img_this + (size_t)gy * pitch + gx, gw, gh, pitch, pts, nd, desc, kept) : 0;   /* :1580 */
    int st;
    int32_t dist = -1;
    const int m = nk > 0 ? svo_match(last_this, desc, nk, &dist) : -1;   /* :1584 */
    if (m < 0) st = ST_TRK_NO_MATCHES;
    else if (!(tp->cutoff_stage2 > (float)dist)) st = ST_TRK_DESC;
    else {
        const float bx = pts[2 * kept[m]], by = pts[2 * kept[m] + 1];
        const float in_cam[2] = {(ul_x + bx) - half, (ul_y + by) - half};   /* :1592 */
        const uint8_t* d_this = desc + (size_t)m * 32;
        const float v_ref = in_cam[1] - half;
        if (!(0.0f <= v_ref)) st = ST_TRK_RANGE;
        else {
            float uv[2];
            double xyz[3];
            uint8_t d_other[32];
            int32_t d2, i2;
            if (left) st = svo_triangulate_right(c, img_other, pitch, fmaxf(0.f, (in_cam[0] - search) - half), v_ref, size, in_cam, d_this, uv, xyz, d_other, &d2, &i2);
            else st = svo_triangulate_left(c, img_other, pitch, search, fmaxf(0.f, in_cam[0] - half), v_ref, size, in_cam, d_this, uv, xyz, d_other, &d2, &i2);
            if (st == ST_OK) {
                if (!depth_ok(c, xyz[2])) st = ST_TRK_DEPTH;
                else if (!(tp->cutoff_stage2 > (float)hamming32(last_other, d_other))) st = ST_TRK_TRI_DESC;
                else {
                    hit->stage = left ? 3 : 4;
                    float* uv_this = left ? hit->uv_l : hit->uv_r;
                    float* uv_oth = left ? hit->uv_r : hit->uv_l;
                    uv_this[0] = in_cam[0]; uv_this[1] = in_cam[1]; uv_oth[0] = uv[0]; uv_oth[1] = uv[1];
                    memcpy(hit->xyz, xyz, sizeof(xyz));
                    memcpy(left ? hit->desc_l : hit->desc_r, d_this, 32);
                    memcpy(left ? hit->desc_r : hit->desc_l, d_other, 32);
                }
            }
        }
    }
    free(xy); free(pts); free(desc); free(kept);
    return st;
}

/* ---- stage 3 geometry (:1795-1947), plain double arithmetic */
static void mul3(const double A[3][3], const double B[3][3], double C[3][3]) {
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) C[i][j] = (A[i][0] * B[0][j] + A[i][1] * B[1][j]) + A[i][2] * B[2][j];
}
static double cof3(const double m[3][3], int i, int j) {
    const int i1 = (i + 1) % 3, i2 = (i + 2) % 3, j1 = (j + 1) % 3, j2 = (j + 2) % 3;
    return m[i1][j1] * m[i2][j2] - m[i1][j2] * m[i2][j1];
}
static void inv3(const double m[3][3], double out[3][3]) {   /* adjugate / determinant (Eigen's fixed 3x3 closed form) */
    const double c0 = cof3(m, 0, 0), c1 = cof3(m, 1, 0), c2 = cof3(m, 2, 0);
    const double det = (c0 * m[0][0] + c1 * m[1][0]) + c2 * m[2][0];
    const double inv_det = 1.0 / det;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) out[i][j] = cof3(m, j, i) * inv_det;
}

typedef struct { int along_u, count; double start, c0, c1, c2; } epi_plan;

static int epipolar_plan(const svo_config* cfg, const svo_track_params* tp, const double* Tw, const double* Td, const double* uv_ref,
                         const double* pw, double motion_scaling, epi_plan* it) {
    double R[3][3], t[3];
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) R[i][j] = (Tw[4 * i] * Td[j] + Tw[4 * i + 1] * Td[4 + j]) + Tw[4 * i + 2] * Td[8 + j];
        t[i] = ((Tw[4 * i] * Td[3] + Tw[4 * i + 1] * Td[7]) + Tw[4 * i + 2] * Td[11]) + Tw[4 * i + 3];
    }
    if (!(0.0 < (t[0] * t[0] + t[1] * t[1]) + t[2] * t[2])) return ST_EPI_NO_TRANSLATION;
    const double S[3][3] = {{0.0, -t[2], t[1]}, {t[2], 0.0, -t[0]}, {-t[1], t[0], 0.0}};   /* CMiniVisionToolbox::getSkew */
    double E[3][3], K[3][3], Ki[3][3], KiT[3][3], A[3][3], F[3][3];
    mul3(R, S, E);                                                                          /* :1800 */
    const double* P = cfg->P_left;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) K[i][j] = P[4 * i + j];
    inv3(K, Ki);
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) KiT[i][j] = Ki[j][i];
    mul3(KiT, E, A);
    mul3(A, Ki, F);                                                                         /* :1801 */
    double c[3];
    for (int i = 0; i < 3; ++i) c[i] = (F[i][0] * uv_ref[0] + F[i][1] * uv_ref[1]) + F[i][2] * 1.0;   /* :1818 */
    double p[3];
    to_camera(Tw, pw, p);
    float pu, pv;
    projection_rounded(P, p, &pu, &pv);                                                     /* :1807 */
    if (!fov_contains(cfg, pu, pv)) return ST_EPI_OUT_OF_SIGHT;
    const double W = (double)cfg->width, H = (double)cfg->height;
    const double half = 10.0 * motion_scaling;                                              /* :1362 */
    const double wu = sqrt(fabs((double)pu - P[2])) / 10.0, wv = sqrt(fabs((double)pv - P[6])) / 10.0;
    const double hl_u = tp->epipolar_base_length + wu * half, hl_v = tp->epipolar_base_length + wv * half;   /* :1821-1822 */
#define CURVE_V(u_) (-(c[0] * (u_) + c[2]) / c[1])
#define CURVE_U(v_) (-(c[1] * (v_) + c[2]) / c[0])
    const double u_min_raw = fmax((double)pu - hl_u, 0.0), u_max_raw = fmin((double)pu + hl_u, W);
    const double v_min_raw = CURVE_V(u_min_raw), v_max_raw = CURVE_V(u_max_raw);
    if ((0.0 > v_min_raw && 0.0 > v_max_raw) || (H < v_min_raw && H < v_max_raw)) return ST_EPI_VERTICAL;
    const double v_lim_min = fmax((double)pv - hl_v, 0.0), v_lim_max = fmin((double)pv + hl_v, H);
    double u_min = u_min_raw, u_max = u_max_raw, v_for_min, v_for_max;
    if (v_min_raw < v_max_raw) {
        if (v_lim_min > v_max_raw || v_lim_max < v_min_raw) return ST_EPI_NEG_SLOPE;
        if (v_lim_min > v_min_raw) { v_for_min = v_lim_min; u_min = CURVE_U(v_for_min); } else v_for_min = v_min_raw;
        if (v_lim_max < v_max_raw) { v_for_max = v_lim_max; u_max = CURVE_U(v_for_max); } else v_for_max = v_max_raw;
    } else {
        if (v_lim_min > v_min_raw || v_lim_max < v_max_raw) return ST_EPI_POS_SLOPE;
        if (v_lim_min > v_max_raw) { v_for_min = v_lim_min; u_max = CURVE_U(v_for_min); } else v_for_min = v_max_raw;
        if (v_lim_max < v_min_raw) { v_for_max = v_lim_max; u_min = CURVE_U(v_for_max); } else v_for_max = v_min_raw;
    }
#undef CURVE_V
#undef CURVE_U
    const double du = u_max - u_min, dv = v_for_max - v_for_min;
    /* the reference converts these to uint32_t (:1933-1934); negative / non-finite values are undefined there */
    if (!(isfinite(du) && isfinite(dv)) || du < 0.0 || dv < 0.0 || du >= 65536.0 || dv >= 65536.0) return ST_EPI_ZERO_LEN;
    const int delta_u = (int)du, delta_v = (int)dv;
    if (delta_u == 0 && delta_v == 0) return ST_EPI_ZERO_LEN;
    it->along_u = delta_v < delta_u ? 1 : 0;
    it->count = it->along_u ? delta_u : delta_v;
    it->start = it->along_u ? u_min : v_for_min;
    it->c0 = c[0]; it->c1 = c[1]; it->c2 = c[2];
    return ST_OK;
}

/* _getMatchSampleRecursiveU/V + _getMatch (:2142-2397): one key-point per pixel along the line, BRIEF in the bounding
 * ROI, 1 x N match, cut-offs 50 (last) / 100 (original); one retry with the samples moved by +2 px */
static int epipolar_match(const svo_config* cfg, const svo_track_params* tp, const uint8_t* img, int pitch, const epi_plan* it,
                          float size, const uint8_t* last_desc, const uint8_t* orig_desc, float* uv, uint8_t* desc_out) {
    const int n = it->count;
    const float wf = (float)cfg->width, hf = (float)cfg->height;
    float* pool = (float*)malloc(sizeof(float) * 2 * (size_t)n);
    float* local = (float*)malloc(sizeof(float) * 2 * (size_t)n);
    uint8_t* desc = (uint8_t*)malloc((size_t)32 * n);
    int32_t* kept = (int32_t*)malloc(sizeof(int32_t) * (size_t)n);
    int status = ST_EPI_POOL_EMPTY;
    for (int attempt = 0; attempt < 2; ++attempt) {
        const double off = attempt ? 2.0 : 0.0;   /* recursion depth 0, then 2 (limit 2, step 2) */
        for (int i = 0; i < n; ++i) {
            double du, dv;
            if (it->along_u) { du = it->start + (double)i; dv = (-(it->c0 * du + it->c2) / it->c1) + off; }
            else { dv = it->start + (double)i; du = (-(it->c1 * dv + it->c2) / it->c0) + off; }
            pool[2 * i] = (float)du; pool[2 * i + 1] = (float)dv;
        }
        const float* ctr = pool + 2 * (n / 2);
        const float f_du = fabsf(pool[0] - pool[2 * (n - 1)]) + 16.f * size, f_dv = fabsf(pool[1] - pool[2 * (n - 1) + 1]) + 16.f * size;
        const float u_tl = fmaxf(ctr[0] - f_du / 2.f, 0.f), v_tl = fmaxf(ctr[1] - f_dv / 2.f, 0.f);
        const float width = fminf(f_du, wf - u_tl), height = fminf(f_dv, hf - v_tl);
        status = ST_EPI_POOL_EMPTY;
        if (!(isfinite(u_tl) && isfinite(v_tl) && isfinite(width) && isfinite(height))) continue;
        const int rx = (int)u_tl, ry = (int)v_tl, rw = (int)width, rh = (int)height;   /* cv::Rect(float...) truncates */
        if (rw <= 0 || rh <= 0 || rx + rw > cfg->width || ry + rh > cfg->height) continue;
        for (int i = 0; i < n; ++i) { local[2 * i] = pool[2 * i] - u_tl; local[2 * i + 1] = pool[2 * i + 1] - v_tl; }
        const int nk = svo_brief32(img + (size_t)ry * pitch + rx, rw, rh, pitch, local, n, desc, kept);
        if (nk <= 0) continue;
        int32_t dist;
        const int m = svo_match(last_desc, desc, nk, &dist);
        status = ST_EPI_DIST;
        if (!(tp->cutoff_stage3 > (float)dist)) continue;
        status = ST_EPI_ORIG_DIST;
        if (!(tp->cutoff_original > (float)hamming32(orig_desc, desc + (size_t)m * 32))) continue;
        uv[0] = local[2 * kept[m]] + u_tl;
        uv[1] = local[2 * kept[m] + 1] + v_tl;
        memcpy(desc_out, desc + (size_t)m * 32, 32);
        status = ST_OK;
        break;
    }
    free(pool); free(local); free(desc); free(kept);
    return status;
}

static int track_stage3(const svo_config* c, const svo_track_params* tp, const uint8_t* img_l, const uint8_t* img_r, int pitch,
                        const double* Tw, const svo_landmarks* lm, int q, double motion_scaling, track_hit* hit) {
    epi_plan it;
    int st = epipolar_plan(c, tp, Tw, lm->T_left_to_world_at_detection + 16 * (size_t)q, lm->uv_reference_left + 2 * (size_t)q,
                           lm->xyz_world + 3 * (size_t)q, motion_scaling, &it);
    if (st != ST_OK) return st;
    const float size = lm->keypoint_size[q];
    float uv[2];
    uint8_t d[32];
    st = epipolar_match(c, tp, img_l, pitch, &it, size, lm->last_desc_left + 32 * (size_t)q, lm->desc_reference_left + 32 * (size_t)q, uv, d);
    if (st != ST_OK) return st;
    const float search = (float)((1.0 + motion_scaling) * (double)lm->last_disparity[q]);   /* :2415 double product, then float */
    float uvr[2];
    double xyz[3];
    uint8_t dr[32];
    int32_t dist, idx;
    st = svo_triangulate_right(c, img_r, pitch, fmaxf(0.f, (uv[0] - search) - 4.f * size), uv[1] - 4.f * size, size, uv, d, uvr, xyz, dr, &dist, &idx);
    if (st != ST_OK) return st;
    if (!depth_ok(c, xyz[2])) return ST_TRK_DEPTH;
    hit->stage = 5;
    hit->uv_l[0] = uv[0]; hit->uv_l[1] = uv[1]; hit->uv_r[0] = uvr[0]; hit->uv_r[1] = uvr[1];
    memcpy(hit->xyz, xyz, sizeof(xyz)); memcpy(hit->desc_l, d, 32); memcpy(hit->desc_r, dr, 32);
    return ST_OK;
}

/* the cascade for landmark q; stage_mask bit 0 = stage 1, bit 1 = stage 2, bit 2 = stage 3 (svi_track_landmarks_stages) */
static void track_one(const svo_config* c, const svo_track_params* tp, const uint8_t* img_l, const uint8_t* img_r, int pitch,
                      const double* Tw, const svo_landmarks* lm, int q, double motion_scaling, unsigned stage_mask,
                      const svo_track_result* out) {
    track_hit hit;
    memset(&hit, 0, sizeof(hit));
    int status = ST_TRK_STAGE1_DIST;
    const float size = lm->keypoint_size[q];
    const uint8_t *last_l = lm->last_desc_left + 32 * (size_t)q, *last_r = lm->last_desc_right + 32 * (size_t)q;
    if (stage_mask & 3u) {
        double p[3];
        to_camera(Tw, lm->xyz_world + 3 * (size_t)q, p);                                   /* :1404 */
        float ul, vl, ur, vr;
        projection_rounded(c->P_left, p, &ul, &vl);
        projection_rounded(c->P_right, p, &ur, &vr);
        const float search = (float)(1.0 + motion_scaling) * lm->last_disparity[q];        /* :1363, :1413 */
        if (!(fov_contains(c, ul, vl) && fov_contains(c, ur, vr))) status = ST_TRK_OUT_OF_FOV;   /* :1416 */
        else {
            if (stage_mask & 1u) status = track_stage1(c, tp, img_l, img_r, pitch, ul, vl, ur, vr, size, search, last_l, last_r, &hit);
            if (!hit.stage && (stage_mask & 2u)) {
                status = track_stage2_side(c, tp, img_l, img_r, pitch, c->P_left, ul, vl, last_l, last_r, search, size, motion_scaling, 1, &hit);
                if (!hit.stage)
                    status = track_stage2_side(c, tp, img_r, img_l, pitch, c->P_right, ur, vr, last_r, last_l, search, size, motion_scaling, 0, &hit);
            }
        }
    }
    if (!hit.stage && status != ST_TRK_OUT_OF_FOV && (stage_mask & 4u))
        status = track_stage3(c, tp, img_l, img_r, pitch, Tw, lm, q, motion_scaling, &hit);
    out->status[q] = (uint8_t)(hit.stage ? ST_OK : status);
    out->stage[q] = (uint8_t)hit.stage;
    if (hit.stage) {
        memcpy(out->uv_left + 2 * (size_t)q, hit.uv_l, sizeof(hit.uv_l));
        memcpy(out->uv_right + 2 * (size_t)q, hit.uv_r, sizeof(hit.uv_r));
        memcpy(out->xyz_left + 3 * (size_t)q, hit.xyz, sizeof(hit.xyz));
        memcpy(out->desc_left + 32 * (size_t)q, hit.desc_l, 32);
        memcpy(out->desc_right + 32 * (size_t)q, hit.desc_r, 32);
    }
}

typedef struct {
    const svo_config* c; const svo_track_params* tp; const uint8_t* img_l; const uint8_t* img_r; int pitch; const double* Tw;
    const svo_landmarks* lm; int n; double motion_scaling; unsigned stage_mask; const svo_track_result* out;
    int next; pthread_mutex_t mu;
} track_job;

static void* track_worker(void* arg) {
    track_job* j = (track_job*)arg;
    for (;;) {
        pthread_mutex_lock(&j->mu);
        const int q0 = j->next;
        j->next += 16;
        pthread_mutex_unlock(&j->mu);
        if (q0 >= j->n) break;
        for (int q = q0; q < q0 + 16 && q < j->n; ++q)
            track_one(j->c, j->tp, j->img_l, j->img_r, j->pitch, j->Tw, j->lm, q, j->motion_scaling, j->stage_mask, j->out);
    }
    return NULL;
}

int svo_track_params_default(svo_track_params* tp) {
    tp->cutoff_stage1 = 25.f; tp->cutoff_stage2 = 50.f; tp->cutoff_stage3 = 50.f; tp->cutoff_original = 100.f;
    tp->epipolar_base_length = 15.0;
    tp->block_size_stage2 = 15;
    return 0;
}

/* trackManual for n landmarks of one stereo pair.  The reference walks them on one thread (n_threads = 1); more threads
 * split the landmarks (they are independent within a frame) for the all-cores baseline. */
int svo_track_landmarks(const svo_config* c, const svo_track_params* tp, const uint8_t* img_left, const uint8_t* img_right, int pitch,
                        const double* T_world_to_left, const svo_landmarks* lm, int n, double motion_scaling, unsigned stage_mask,
                        const svo_track_result* out, int n_threads) {
    if ((stage_mask & 4u) && !(lm->uv_reference_left && lm->desc_reference_left && lm->T_left_to_world_at_detection)) return -1;
    track_job j;
    j.c = c; j.tp = tp; j.img_l = img_left; j.img_r = img_right; j.pitch = pitch; j.Tw = T_world_to_left; j.lm = lm; j.n = n;
    j.motion_scaling = motion_scaling; j.stage_mask = stage_mask; j.out = out; j.next = 0;
    pthread_mutex_init(&j.mu, NULL);
    if (n_threads < 1) n_threads = 1;
    if (n_threads > (n + 15) / 16) n_threads = n > 0 ? (n + 15) / 16 : 1;
    pthread_t* th = (pthread_t*)malloc(sizeof(pthread_t) * n_threads);
    for (int i = 1; i < n_threads; ++i) pthread_create(&th[i], NULL, track_worker, &j);
    track_worker(&j);
    for (int i = 1; i < n_threads; ++i) pthread_join(th[i], NULL);
    free(th);
    pthread_mutex_destroy(&j.mu);
    return 0;
}

/* ---- CLandmark::optimize / _getOptimizedLandmarkSTEREOUV (src/types/CLandmark.cpp:281-296, :447-581): robust Gauss-Newton
 * refinement of one landmark's WORLD position on the stereo re-projection error of its measurements; constants of
 * CLandmark.h:90-98.  Written from the reference's loop: per measurement the two projections, the error, the Jacobian of the
 * homogeneous division times the projection, the weight, the accumulation of H and b; then
 * H.block<4,3>(0,0).householderQr().solve(-b) restated as three Householder reflections and a back substitution (Eigen's
 * result up to rounding), the convergence test on the total squared error and the inlier / average-error verdicts.
 * m measurements: proj_left / proj_right m x 12 (row-major 3 x 4), uv_left / uv_right m x 2.
 * outcome: 0 skipped (m <= 5: position kept, optimal), 1 converged, 2 converged and optimal, 3 rejected (inlier ratio),
 * 4 not converged in 1000 iterations.  xyz_out = refined position for 1 / 2, the guess otherwise. */
static void svo_ls_4x3(double H[4][4], const double b[4], double x[3]) {
    double A[4][3], y[4];
    for (int i = 0; i < 4; ++i) { for (int j = 0; j < 3; ++j) A[i][j] = H[i][j]; y[i] = -b[i]; }
    for (int c = 0; c < 3; ++c) {
        double norm = 0.0;
        for (int r = c; r < 4; ++r) norm += A[r][c] * A[r][c];
        norm = sqrt(norm);
        if (norm == 0.0) continue;
        const double alpha = A[c][c] > 0.0 ? -norm : norm;
        double v[4] = {0.0, 0.0, 0.0, 0.0};
        v[c] = A[c][c] - alpha;
        for (int r = c + 1; r < 4; ++r) v[r] = A[r][c];
        double vv = 0.0;
        for (int r = c; r < 4; ++r) vv += v[r] * v[r];
        if (vv == 0.0) continue;
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
        double s = y[r];
        for (int j = r + 1; j < 3; ++j) s -= A[r][j] * x[j];
        x[r] = A[r][r] != 0.0 ? s / A[r][r] : 0.0;
    }
}

int svo_optimize_landmark(const double* xyz_guess, int m, const double* proj_left, const double* proj_right, const float* uv_left,
                          const float* uv_right, double* xyz_out, int32_t* outcome, double* average_squared_error, int32_t* iterations) {
    const double kernel = 10.0, delta = 1e-5, min_ratio = 0.5, max_avg = 9.0;
    xyz_out[0] = xyz_guess[0]; xyz_out[1] = xyz_guess[1]; xyz_out[2] = xyz_guess[2];
    *average_squared_error = 0.0;
    *iterations = 0;
    if (!(5 < m)) { *outcome = 0; return 0; }
    double X[4] = {xyz_guess[0], xyz_guess[1], xyz_guess[2], 1.0};
    double prev = 0.0;
    for (int it = 0; it < 1000; ++it) {
        double H[4][4] = {{0}}, b[4] = {0, 0, 0, 0}, total = 0.0;
        int inliers = 0;
        for (int k = 0; k < m; ++k) {
            const double* P[2] = {proj_left + 12 * (size_t)k, proj_right + 12 * (size_t)k};
            const float* uv[2] = {uv_left + 2 * (size_t)k, uv_right + 2 * (size_t)k};
            double J[4][4], e[4];
            for (int s = 0; s < 2; ++s) {
                const double* p = P[s];
                double a[3];
                for (int r = 0; r < 3; ++r) a[r] = p[4 * r] * X[0] + p[4 * r + 1] * X[1] + p[4 * r + 2] * X[2] + p[4 * r + 3] * X[3];
                const double c = a[2];
                e[2 * s] = a[0] / c - uv[s][0];
                e[2 * s + 1] = a[1] / c - uv[s][1];
                for (int q = 0; q < 4; ++q) {
                    J[2 * s][q] = p[q] / c - a[0] / (c * c) * p[8 + q];
                    J[2 * s + 1][q] = p[4 + q] / c - a[1] / (c * c) * p[8 + q];
                }
            }
            const double e2 = e[0] * e[0] + e[1] * e[1] + e[2] * e[2] + e[3] * e[3];
            double w = 1.0;
            if (kernel < e2) w = kernel / e2; else ++inliers;
            total += w * e2;
            for (int r = 0; r < 4; ++r) {
                for (int q = 0; q < 4; ++q) H[r][q] += w * (J[0][r] * J[0][q] + J[1][r] * J[1][q] + J[2][r] * J[2][q] + J[3][r] * J[3][q]);
                b[r] += w * (J[0][r] * e[0] + J[1][r] * e[1] + J[2][r] * e[2] + J[3][r] * e[3]);
            }
        }
        double dx[3];
        svo_ls_4x3(H, b, dx);
        X[0] += dx[0]; X[1] += dx[1]; X[2] += dx[2];
        *iterations = it + 1;
        if (delta > fabs(prev - total)) {
            const double avg = total / (double)m;
            if (min_ratio < (double)inliers / (double)m) {
                xyz_out[0] = X[0]; xyz_out[1] = X[1]; xyz_out[2] = X[2];
                *average_squared_error = avg;
                *outcome = max_avg > avg ? 2 : 1;
            } else {
                *outcome = 3;
            }
            return 0;
        }
        prev = total;
    }
    *outcome = 4;
    return 0;
}

/* ---- CSolverStereoPosit::getTransformationWORLDtoLEFT (src/optimization/CSolverStereoPosit.cpp:8-170): robust Gauss-Newton on
 * the four-dimensional stereo re-projection error of the WORLD->LEFT pose, constants of CSolverStereoPosit.h:89-99.  Written
 * from the reference's loop: per measurement the transform into the LEFT frame (points with z <= 0 contribute nothing but still
 * count in the average), both projections, the error, the robust weight, the 4 x 6 Jacobian of the increment (translation,
 * quaternion vector part of CMiniVisionToolbox::getTransformationFromVector, src/vision/CMiniVisionToolbox.cpp:354-377) and the
 * accumulation of the normal equations; then H dx = -b by Gaussian elimination with partial pivoting, the pose update
 * T = T(dx) * T, the re-orthonormalisation R -= 0.5 R (R^T R - I), and at convergence (1e-5 on the total weighted error) the
 * accuracy verdict, the translation clamp against T_last and the risk test against the prior's position plus t_imu.
 * Every sum runs in measurement order and every operation rounds on its own (-ffp-contract=off), so the result is the C++ host
 * layer's (host/CSolverStereoPosit.h) to the last bit.
 * P_left / P_right / T_estimate / T_last row-major (3 x 4, 4 x 4); n measurements: xyz_world n x 3, uv_left / uv_right n x 2.
 * Outputs as svi_posit_result: T_out = the solution for outcome 0, else T_estimate; outcome 0 ok / 1 too few points (n <= 25) /
 * 2 inaccurate / 3 high risk / 4 not converged in 1000 iterations; iterations run (0 for 1); inliers of the last iteration;
 * average_squared_error of the converged iteration (else 0); risk (0 unless the risk test ran). */
static void svo_iso_mul(const double* A, const double* B, double* C) {   /* Isometry3d * Isometry3d: bottom row (0 0 0 1) */
    for (int k = 0; k < 16; ++k) C[k] = (k % 5 == 0) ? 1.0 : 0.0;
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 4; ++c) {
            double s = 0.0;
            for (int k = 0; k < 3; ++k) s += A[4 * r + k] * B[4 * k + c];
            C[4 * r + c] = s + (c == 3 ? A[4 * r + 3] : 0.0);
        }
}

static void svo_posit_rows(const double* P, const double a[3], double c, const double Jt[3][6], double* rowU, double* rowV) {
    for (int k = 0; k < 6; ++k) {
        double PJ[3];
        for (int r = 0; r < 3; ++r) PJ[r] = P[4 * r] * Jt[0][k] + P[4 * r + 1] * Jt[1][k] + P[4 * r + 2] * Jt[2][k];
        rowU[k] = PJ[0] / c - a[0] / (c * c) * PJ[2];
        rowV[k] = PJ[1] / c - a[1] / (c * c) * PJ[2];
    }
}

static void svo_posit_solve(const double H[6][6], const double b[6], double x[6]) {
    double A[6][7];
    for (int i = 0; i < 6; ++i) { for (int j = 0; j < 6; ++j) A[i][j] = H[i][j]; A[i][6] = -b[i]; }
    for (int c = 0; c < 6; ++c) {
        int piv = c;
        for (int r = c + 1; r < 6; ++r) if (fabs(A[r][c]) > fabs(A[piv][c])) piv = r;
        if (piv != c) for (int j = 0; j < 7; ++j) { const double t = A[c][j]; A[c][j] = A[piv][j]; A[piv][j] = t; }
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

int svo_solve_stereo_posit(const double* P_left, const double* P_right, const double* T_estimate, const double* T_last, const double* t_imu,
                           int n, const double* xyz_world, const float* uv_left, const float* uv_right, double* T_out, int32_t* outcome,
                           int32_t* iterations, int32_t* inliers_out, double* average_squared_error, double* risk_out) {
    const double kernel = 10.0, max_avg = 9.0, max_risk = 2.0, delta = 1e-5, min_t2 = 0.001;
    const int min_points = 25, min_inliers = 15, cap = 1000;
    memcpy(T_out, T_estimate, 16 * sizeof(double));
    *iterations = 0; *inliers_out = 0; *average_squared_error = 0.0; *risk_out = 0.0;
    if (!(min_points < n)) { *outcome = 1; return 0; }
    double T[16];
    memcpy(T, T_estimate, sizeof(T));
    double prev = 0.0;
    for (int it = 0; it < cap; ++it) {
        double H[6][6] = {{0}}, b[6] = {0, 0, 0, 0, 0, 0}, total = 0.0;
        int inliers = 0;
        for (int m = 0; m < n; ++m) {
            const double* X = xyz_world + 3 * (size_t)m;
            const double p[3] = {T[0] * X[0] + T[1] * X[1] + T[2] * X[2] + T[3], T[4] * X[0] + T[5] * X[1] + T[6] * X[2] + T[7],
                                 T[8] * X[0] + T[9] * X[1] + T[10] * X[2] + T[11]};
            if (!(0.0 < p[2])) continue;
            double aL[3], aR[3];
            for (int r = 0; r < 3; ++r) {
                aL[r] = P_left[4 * r] * p[0] + P_left[4 * r + 1] * p[1] + P_left[4 * r + 2] * p[2] + P_left[4 * r + 3];
                aR[r] = P_right[4 * r] * p[0] + P_right[4 * r + 1] * p[1] + P_right[4 * r + 2] * p[2] + P_right[4 * r + 3];
            }
            const double cL = aL[2], cR = aR[2];
            const double e[4] = {aL[0] / cL - (double)uv_left[2 * (size_t)m], aL[1] / cL - (double)uv_left[2 * (size_t)m + 1],
                                 aR[0] / cR - (double)uv_right[2 * (size_t)m], aR[1] / cR - (double)uv_right[2 * (size_t)m + 1]};
            const double e2 = e[0] * e[0] + e[1] * e[1] + e[2] * e[2] + e[3] * e[3];
            double w = 1.0;
            if (kernel < e2) w = kernel / e2; else ++inliers;
            total += w * e2;
            const double Jt[3][6] = {{1, 0, 0, 0, 2 * p[2], -2 * p[1]}, {0, 1, 0, -2 * p[2], 0, 2 * p[0]}, {0, 0, 1, 2 * p[1], -2 * p[0], 0}};
            double J[4][6];
            svo_posit_rows(P_left, aL, cL, Jt, J[0], J[1]);
            svo_posit_rows(P_right, aR, cR, Jt, J[2], J[3]);
            for (int i = 0; i < 6; ++i) {
                for (int j = 0; j < 6; ++j) H[i][j] += w * (J[0][i] * J[0][j] + J[1][i] * J[1][j] + J[2][i] * J[2][j] + J[3][i] * J[3][j]);
                b[i] += w * (J[0][i] * e[0] + J[1][i] * e[1] + J[2][i] * e[2] + J[3][i] * e[3]);
            }
        }
        double dx[6], D[16], Tn[16];
        svo_posit_solve(H, b, dx);
        for (int k = 0; k < 16; ++k) D[k] = (k % 5 == 0) ? 1.0 : 0.0;
        D[3] = dx[0]; D[7] = dx[1]; D[11] = dx[2];
        const double x = dx[3], y = dx[4], z = dx[5], n2 = x * x + y * y + z * z;
        if (1.0 > n2) {
            const double qw = sqrt(1.0 - n2);
            D[0] = 1 - 2 * (y * y + z * z); D[1] = 2 * (x * y - z * qw);     D[2] = 2 * (x * z + y * qw);
            D[4] = 2 * (x * y + z * qw);     D[5] = 1 - 2 * (x * x + z * z); D[6] = 2 * (y * z - x * qw);
            D[8] = 2 * (x * z - y * qw);     D[9] = 2 * (y * z + x * qw);     D[10] = 1 - 2 * (x * x + y * y);
        }
        svo_iso_mul(D, T, Tn);
        double RtR[3][3], R[3][3];
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) RtR[i][j] = Tn[i] * Tn[j] + Tn[4 + i] * Tn[4 + j] + Tn[8 + i] * Tn[8 + j] - (i == j ? 1.0 : 0.0);
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) R[i][j] = Tn[4 * i + j] - 0.5 * (Tn[4 * i] * RtR[0][j] + Tn[4 * i + 1] * RtR[1][j] + Tn[4 * i + 2] * RtR[2][j]);
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) Tn[4 * i + j] = R[i][j];
        memcpy(T, Tn, sizeof(T));
        *iterations = it + 1;
        *inliers_out = inliers;
        if (delta > fabs(prev - total)) {
            const double avg = total / (double)n;
            *average_squared_error = avg;
            if (max_avg < avg && min_inliers > inliers) { *outcome = 2; return 0; }
            double d2 = 0.0;
            for (int r = 0; r < 3; ++r) { const double d = T[4 * r + 3] - T_last[4 * r + 3]; d2 += d * d; }
            if (min_t2 > d2)
                for (int r = 0; r < 3; ++r) T[4 * r + 3] = T_last[4 * r + 3];   /* the translational part is not integrated */
            double risk = 0.0;
            for (int r = 0; r < 3; ++r) {   /* position of the solution minus the prior's, minus t_imu (inverseIsometry's translation) */
                const double ti = -(T[r] * T[3] + T[4 + r] * T[7] + T[8 + r] * T[11]);
                const double te = -(T_estimate[r] * T_estimate[3] + T_estimate[4 + r] * T_estimate[7] + T_estimate[8 + r] * T_estimate[11]);
                const double d = ti - te - t_imu[r];
                risk += d * d;
            }
            *risk_out = risk;
            if (max_risk < risk) { *outcome = 3; return 0; }
            memcpy(T_out, T, sizeof(T));
            *outcome = 0;
            return 0;
        }
        prev = total;
    }
    *outcome = 4;
    return 0;
}
