// harris.cuh -- detection front half: Harris response (bit-exact to cv::cornerHarris with
// optimisations off), 9x9 box-sum images for BRIEF, 3x3 NMS candidate extraction -- one kernel, the
// response never leaves the SM.
//
// Replaces, for cv::GFTTDetector::create(1000, 0.01, 7.0, 7, true)->detect
// (reference src/core/CFundamentalMatcher.cpp:18,101), the OpenCV calls cornerHarris
// (Sobel x2, covariance products, 7x7 boxFilter), minMaxLoc, threshold(TOZERO), dilate 3x3 and
// the candidate collection loop of goodFeaturesToTrack; arithmetic order from SURVEY.md App. A.
//
// goodFeaturesToTrack's candidate test "R' != 0 and R' == dilate3x3(R')" with R' = TOZERO(R, thr),
// thr = float(double(max R) * quality), equals "R > thr and R >= its 8 raw neighbours" (thresholding is
// monotone), and thr > 0 whenever there is a candidate at all.  A CTA therefore emits the local maxima
// of its response tile that exceed the threshold of the TILE's own maximum (<= the frame's, so nothing
// is lost, and the emitted list is deterministic); the exact frame threshold is applied to the keys by
// select_corners_kernel once the frame maximum is final.  Response tiles overlap by one pixel on each
// side (stride 62 x 30 for a 64 x 32 tile) so that every candidate sees its 8 neighbours on chip.
#pragma once
#include "common.cuh"

namespace svi {

// Tile width: 64 (CTAs of 256 threads, four per SM).  -DHARRIS_TILE_W=128 builds CTAs of 512 threads, two per SM: the
// 6-px Sobel/box halo and the 2-px candidate overlap spread over twice the columns (1.35 instead of 1.43 pixels of work
// per useful pixel, 10 instead of 21 tiles per 1241-px row) -- measured SLOWER (C2: harris_box 20.0 vs 17.7 ms per 64
// launches, 97.3 k vs 103.9 k frames/s; C4 124.9 k vs 136.0 k): the kernel has seven barrier phases, and two big CTAs per
// SM leave fewer independent CTAs to fill them than four small ones.  Kept as a build option, parity-tested at both widths.
#ifndef HARRIS_TILE_W
#define HARRIS_TILE_W 64
#endif
constexpr int HT_W = HARRIS_TILE_W, HT_H = 32, HT_THREADS = HT_W * 4;
static_assert(HT_W == 64 || HT_W == 128, "tile width");
#ifndef HARRIS_CTAS_PER_SM
#define HARRIS_CTAS_PER_SM (HT_W == 64 ? 4 : 2)
#endif
constexpr int HT_SX = HT_W - 2, HT_SY = HT_H - 2;   // tile stride of the Harris kernel: candidates = tile interior
constexpr int HT_MAX_KEYS = HT_SX * HT_SY;          // a plateau can make every interior pixel a local maximum
constexpr int U8_W = HT_W + 8;       // u8 tile: 4-px halo (1 Sobel + 3 box; also the 9x9 box sum)
constexpr int U8_P = U8_W + 4;       // 19 words per row: row-per-lane walks are bank-conflict free
constexpr int H9_P = HT_W + 2;       // 33 words per row, same reason
constexpr int U8_ROWS = HT_H + 8;
constexpr int COV_W = HT_W + 6;      // covariance products: 3-px halo
constexpr int COV_ROWS = HT_H + 6;
constexpr int COV_P = HT_W == 64 ? 73 : 139;   // odd pitches: row-per-lane accesses are bank-conflict free
constexpr int HS_P = HT_W + 1;
constexpr int COV_SEG_ROWS = 13;     // 38 rows = 3 segments for the sliding Sobel
constexpr int HS_SEG = 11;           // horizontal box sums: 11 outputs per work item, 6 segments x 38 rows = 228 items
constexpr int HS_NSEG = (HT_W + HS_SEG - 1) / HS_SEG;
static_assert(HS_NSEG * COV_ROWS <= HT_THREADS, "one horizontal work item per thread");
static_assert((HS_NSEG - 1) * HS_SEG + HS_SEG + 6 <= COV_P, "the last segment's loads stay inside the padded row");
static_assert(COV_ROWS > 32 && COV_ROWS <= 64, "row mapping of the horizontal pass");

struct __align__(16) HarrisSmem {
    double hs[COV_ROWS][HS_P];        // horizontal 7-sums of ONE product plane, fp64
    float cov[3][COV_ROWS][COV_P];    // Dx*Dx, Dx*Dy, Dy*Dy (fp32); reused as the 9-sum rows (u16)
    uint8_t tile[U8_ROWS][U8_P];
    uint32_t red[HT_THREADS / 32];
    int key_count, key_base;
};
static_assert(sizeof(float) * 3 * COV_ROWS * COV_P >= sizeof(uint16_t) * U8_ROWS * H9_P, "h9 alias");
static_assert(sizeof(float) * 3 * COV_ROWS * COV_P >= sizeof(float) * HT_H * HT_W, "response tile alias");
static_assert(sizeof(double) * COV_ROWS * HS_P >= sizeof(unsigned long long) * HT_MAX_KEYS, "key list alias");

// Stage the (HT_H+8) x (HT_W+8) u8 tile with REFLECT_101 at the image border.  A warp copies whole rows: lane l
// moves bytes l, l+32, l+64 of a row, so every load instruction of the warp touches one or two 128-byte lines
// (image rows have no alignment: the pitch is the image width) and every shared store is one wavefront.
__device__ __forceinline__ void load_tile_u8(uint8_t (*tile)[U8_P], const uint8_t* __restrict__ img,
                                             int pitch, int W, int H, int x0, int y0) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gx0 = x0 - 4, gy0 = y0 - 4;
    const bool inside_x = gx0 >= 0 && gx0 + U8_W <= W;        // CTA-uniform
    const bool inside_y = gy0 >= 0 && gy0 + U8_ROWS <= H;     // CTA-uniform
    constexpr int NW = HT_THREADS / 32, RPW = (U8_ROWS + NW - 1) / NW;   // rows per warp
    // all loads of the thread are issued before the first store: the global round trip is paid once.
    // 32-bit element offsets inside the frame; the three loads of a row share one address register.
    constexpr int NG = (U8_W + 31) / 32;          // 32-byte column groups of a row; only the last one is partial
    const bool last_ok = lane < U8_W - 32 * (NG - 1);
    uint8_t v[RPW][NG];
    if (inside_x) {
        const uint8_t* col = img + gx0 + lane;
#pragma unroll
        for (int k = 0; k < RPW; ++k) {
            const int ly = min(warp + k * NW, U8_ROWS - 1);
            const int ry = inside_y ? gy0 + ly : reflect101(gy0 + ly, H);
            const uint8_t* src = col + ry * pitch;
#pragma unroll
            for (int c = 0; c < NG; ++c) v[k][c] = (c < NG - 1 || last_ok) ? __ldg(src + 32 * c) : (uint8_t)0;
        }
    } else {
        int cx[NG];
#pragma unroll
        for (int c = 0; c < NG; ++c) cx[c] = reflect101(gx0 + lane + 32 * c, W);
#pragma unroll
        for (int k = 0; k < RPW; ++k) {
            const int ly = min(warp + k * NW, U8_ROWS - 1);
            const uint8_t* row = img + reflect101(gy0 + ly, H) * pitch;
#pragma unroll
            for (int c = 0; c < NG; ++c) v[k][c] = (c < NG - 1 || last_ok) ? __ldg(row + cx[c]) : (uint8_t)0;
        }
    }
#pragma unroll
    for (int k = 0; k < RPW; ++k) {
        const int ly = warp + k * NW;
        if (ly < U8_ROWS) {
            uint8_t* dst = &tile[ly][lane];
#pragma unroll
            for (int c = 0; c < NG; ++c)
                if (c < NG - 1 || last_ok) dst[32 * c] = v[k][c];
        }
    }
}

// 9x9 box sums (u16, max 81*255 = 20655) of the 64x32 tile from its u8 tile with 4-px halo.
// S(y,x) = sum over [y-4,y+4]x[x-4,x+4]; equals the 4-corner integral-image expression of
// OpenCV BRIEF's smoothedSum.  Values within 4 px of the image border are never sampled.
// `box_shift` (optional) receives the same plane stored one element to the left,
// box_shift[y][x] = S(y, x+1): TMA tile loads must start on a 16-byte boundary, so the match
// kernels fetch their odd-aligned copy of a window from this plane at the same aligned address.
__device__ __forceinline__ void box9_rows(const uint8_t (*tile)[U8_P], uint16_t (*h9)[H9_P]) {
    // horizontal 9-sums: one work item = 16 outputs of one tile row; its 24 source bytes arrive as six 32-bit loads
    // (one shared-memory wavefront each instead of one per byte), the 16 sums leave as eight packed stores
    for (int item = threadIdx.x; item < U8_ROWS * (HT_W / 16); item += HT_THREADS) {
        const int r = item % U8_ROWS, c0 = (item / U8_ROWS) * 16;
        const uint32_t* row32 = reinterpret_cast<const uint32_t*>(tile[r] + c0);   // U8_P and c0 are multiples of 4
        uint32_t w[6];
#pragma unroll
        for (int i = 0; i < 6; ++i) w[i] = row32[i];
        uint32_t b[24];
#pragma unroll
        for (int i = 0; i < 24; ++i) b[i] = __byte_perm(w[i >> 2], 0u, 0x4440u + (i & 3));
        uint32_t s = 0;
#pragma unroll
        for (int i = 0; i < 9; ++i) s += b[i];
        uint32_t* out32 = reinterpret_cast<uint32_t*>(&h9[r][c0]);                  // H9_P and c0 are even
#pragma unroll
        for (int j = 0; j < 16; j += 2) {
            if (j > 0) s += b[j + 8] - b[j - 1];
            const uint32_t s1 = s + b[j + 9] - b[j];
            out32[j >> 1] = s | (s1 << 16);
            s = s1;
        }
    }
}
// (a __syncthreads() separates the two halves)
__device__ __forceinline__ void box9_cols(const uint16_t (*h9)[H9_P], uint16_t* __restrict__ box,
                                          uint16_t* __restrict__ box_shift, int box_pitch, int W, int H, int x0, int y0) {
    // vertical 9-sums, two columns per thread as packed u16 pairs (sums <= 20655, so s + new - old never carries
    // or borrows across the halves): one 32-bit store per plane and row.  thread = (column pair, 8-row group)
    if (threadIdx.x < (HT_W / 2) * (HT_H / 8)) {
        const int xp = (threadIdx.x % (HT_W / 2)) * 2, oy0 = (threadIdx.x / (HT_W / 2)) * 8;
        const int gx = x0 + xp, rows = min(8, H - (y0 + oy0));
        if (gx < W && rows > 0) {
            constexpr int HP = H9_P / 2;   // 33 words per row: conflict-free across the lanes of a warp
            const uint32_t* col = reinterpret_cast<const uint32_t*>(&h9[0][0]) + oy0 * HP + (xp >> 1);
            const bool pair2 = xp + 2 < HT_W;   // columns xp+2, xp+3 (for the shifted plane) are inside this tile
            uint32_t s0 = 0u, s1 = 0u;          // (S(xp), S(xp+1)), (S(xp+2), S(xp+3))
#pragma unroll
            for (int i = 0; i < 9; ++i) { s0 += col[i * HP]; s1 += col[i * HP + 1]; }
            uint16_t* brow = box + (size_t)(y0 + oy0) * box_pitch + gx;
            uint16_t* srow = box_shift ? box_shift + (size_t)(y0 + oy0) * box_pitch + gx : nullptr;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                if (k < rows) {
                    if (k > 0) {
                        s0 = s0 + col[(k + 8) * HP] - col[(k - 1) * HP];
                        s1 = s1 + col[(k + 8) * HP + 1] - col[(k - 1) * HP + 1];
                    }
                    *reinterpret_cast<uint32_t*>(brow) = s0;
                    if (srow) {
                        // srow[j] = S(gx + j + 1)
                        if (pair2) *reinterpret_cast<uint32_t*>(srow) = __byte_perm(s0, s1, 0x5432);
                        else srow[0] = (uint16_t)(s0 >> 16);
                        if (xp == 0 && gx > 0) srow[-1] = (uint16_t)s0;   // the previous tile's last element
                        srow += box_pitch;
                    }
                    brow += box_pitch;
                }
            }
        }
    }
}

// K2: box-sum image of one plane per blockIdx.z (used for the RIGHT image, and for both images
// on the per-query entry points).
__global__ void __launch_bounds__(HT_THREADS)
boxsum9_kernel(const uint8_t* __restrict__ img, FrameGeom g, uint16_t* __restrict__ box, uint16_t* __restrict__ box_shift) {
    __shared__ __align__(16) uint8_t tile[U8_ROWS][U8_P];
    __shared__ __align__(16) uint16_t h9[U8_ROWS][H9_P];
    const int f = blockIdx.z, x0 = blockIdx.x * HT_W, y0 = blockIdx.y * HT_H;
    load_tile_u8(tile, img + (size_t)f * g.img_stride, g.img_pitch, g.W, g.H, x0, y0);
    __syncthreads();
    const size_t fo = (size_t)f * g.H * g.box_pitch;
    box9_rows(tile, h9);
    __syncthreads();
    box9_cols(h9, box + fo, box_shift ? box_shift + fo : nullptr, g.box_pitch, g.W, g.H, x0, y0);
}

// K1: Harris response + per-frame masked maximum + 3x3 NMS candidates + LEFT box-sum image; one 64x32 response
// tile per CTA, tiles HT_SX x HT_SY apart (the tile interior is the CTA's share of the candidates).
//   Sobel (SURVEY.md A.1):  r = p[x+1]-p[x-1];  Dx = (r[y-1]+r[y+1])*f1 + r[y]*f0
//                           q = (p[x-1]*f1 + p[x]*f0) + p[x+1]*f1;  Dy = q[y+1]-q[y-1]
//   every op rounded to fp32 on its own (explicit _rn intrinsics, never an FMA).
//   Box 7x7 (A.2): products accumulated in fp64, REFLECT_101 on the PRODUCT planes, one rounding
//   to fp32.  Harris (A.3): R = (a*c - b*b) - (k*(a+c))*(a+c) in fp32 (the last (W*H) % 4 pixels: k*(a+c)*(a+c) and
//   the difference in fp64 with the double k, as calcHarris's scalar tail).
//   Candidates (A.4): R > 0, R > thr(tile max), R >= its 8 neighbours (neighbours outside the image are
//   ignored, as cv::dilate does), mask != 0, 1-px image border excluded.
//   key = ordered(R) << 32 | y << 16 | x ; descending key order == cv's greaterThanPtr order
//   (value desc, then larger address first).
// With `rois` the z-th CTA layer works on the window rois[z] of image plane rois[z].plane instead of
// frame z: the Sobel filters still read the real pixels around the window (OpenCV ROI semantics without
// BORDER_ISOLATED), while the product planes reflect at the WINDOW edge and the maximum / NMS are window-local
// -- exactly what cv::cornerHarris / goodFeaturesToTrack do on img(roi); key coordinates are window-local.
// `n_rois` (optional) points at the number of valid window items.
// `resp` (optional, svi_harris_response only) receives the response plane, `out_rows` rows per z.
__global__ void __launch_bounds__(HT_THREADS, HARRIS_CTAS_PER_SM)
harris_box_kernel(const uint8_t* __restrict__ img, const uint8_t* __restrict__ mask, FrameGeom g,
                  float f1, float f0, double k, double quality, float* __restrict__ resp, uint16_t* __restrict__ box,
                  uint16_t* __restrict__ box_shift, uint32_t* __restrict__ frame_max,
                  unsigned long long* __restrict__ cand, int* __restrict__ cand_count, int cand_cap,
                  const RoiItem* __restrict__ rois, const int* __restrict__ n_rois, int out_rows) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    HarrisSmem& sm = *reinterpret_cast<HarrisSmem*>(smem_raw);
    const int f = blockIdx.z, x0 = blockIdx.x * HT_SX, y0 = blockIdx.y * HT_SY;
    const int tid = threadIdx.x;
    // W x H is the rectangle the detector sees (frame or window), (ox, oy) its origin in the image
    int W = g.W, H = g.H, ox = 0, oy = 0;
    const uint8_t* im = img + (size_t)f * g.img_stride;
    if (rois) {
        if (n_rois && f >= *n_rois) return;   // the item list was compacted on the device: layers past its end are idle
        const RoiItem it = rois[f];
        W = it.rw; H = it.rh; ox = it.rx; oy = it.ry;
        im = img + (size_t)it.plane * g.img_stride;
    }
    // a tile without interior pixels inside the 1-px border has no candidates, and every pixel it holds also
    // belongs to a neighbouring tile (maximum, box sums); tile (0, 0) always runs
    if ((blockIdx.x > 0 && x0 + 1 > W - 2) || (blockIdx.y > 0 && y0 + 1 > H - 2)) return;
    if (tid == 0) sm.key_count = 0;

    load_tile_u8(sm.tile, im, g.img_pitch, g.W, g.H, ox + x0, oy + y0);
    __syncthreads();

    // ---- covariance products on the (HT_H+6) x (HT_W+6) region, sliding down columns
    if (tid < COV_W * 3) {
        const int c = tid % COV_W, seg = tid / COV_W;
        const int ly0 = seg * COV_SEG_ROWS, ly1 = min(ly0 + COV_SEG_ROWS, COV_ROWS);
        const int gx = x0 - 3 + c, tx = c + 1;
        if (gx >= 0 && gx < W) {
            float r_m, r_c, q_m, q_c;
            {
                const uint8_t* t = sm.tile[ly0];  // tile row of cov row ly0-1 (tile row = cov row + 1)
                float a = u8_to_float(t[tx - 1]), b = u8_to_float(t[tx]), d = u8_to_float(t[tx + 1]);
                r_m = __fsub_rn(d, a);
                q_m = __fadd_rn(__fadd_rn(__fmul_rn(a, f1), __fmul_rn(b, f0)), __fmul_rn(d, f1));
                t = sm.tile[ly0 + 1];
                a = u8_to_float(t[tx - 1]); b = u8_to_float(t[tx]); d = u8_to_float(t[tx + 1]);
                r_c = __fsub_rn(d, a);
                q_c = __fadd_rn(__fadd_rn(__fmul_rn(a, f1), __fmul_rn(b, f0)), __fmul_rn(d, f1));
            }
            for (int ly = ly0; ly < ly1; ++ly) {
                const uint8_t* t = sm.tile[ly + 2];
                float a = u8_to_float(t[tx - 1]), b = u8_to_float(t[tx]), d = u8_to_float(t[tx + 1]);
                float r_p = __fsub_rn(d, a);
                float q_p = __fadd_rn(__fadd_rn(__fmul_rn(a, f1), __fmul_rn(b, f0)), __fmul_rn(d, f1));
                int gy = y0 - 3 + ly;
                if (gy >= 0 && gy < H) {
                    float dx = __fadd_rn(__fmul_rn(__fadd_rn(r_m, r_p), f1), __fmul_rn(r_c, f0));
                    float dy = __fsub_rn(q_p, q_m);
                    sm.cov[0][ly][c] = __fmul_rn(dx, dx);
                    sm.cov[1][ly][c] = __fmul_rn(dx, dy);
                    sm.cov[2][ly][c] = __fmul_rn(dy, dy);
                }
                r_m = r_c; r_c = r_p; q_m = q_c; q_c = q_p;
            }
        }
    }
    __syncthreads();
    // ---- REFLECT_101 of the product planes for halo positions outside the image (border tiles only):
    // at most 3 columns left/right and 3 rows above/below the image are ever read by an in-image output
    {
        const int nlc = max(0, 3 - x0), cr0 = W - x0 + 3, nrc = min(max(COV_W - cr0, 0), 3);
        const int ntr = max(0, 3 - y0), rb0 = H - y0 + 3, nbr = min(max(COV_ROWS - rb0, 0), 3);
        if (nlc + nrc + ntr + nbr > 0) {
            auto fix = [&](int ly, int c) {
                const int gy = y0 - 3 + ly, gx = x0 - 3 + c;
                const int sy = reflect101(gy, H) - (y0 - 3), sx = reflect101(gx, W) - (x0 - 3);
                const bool ok = sy >= 0 && sy < COV_ROWS && sx >= 0 && sx < COV_W;
#pragma unroll
                for (int p = 0; p < 3; ++p) sm.cov[p][ly][c] = ok ? sm.cov[p][sy][sx] : 0.f;
            };
            const int i8 = tid & 7;            // outside columns of every row: 8 lanes per row
            if (i8 < nlc + nrc) {
                const int c = i8 < nlc ? i8 : cr0 + (i8 - nlc);
                for (int ly = tid >> 3; ly < COV_ROWS; ly += HT_THREADS / 8) {
                    const int gy = y0 - 3 + ly;
                    if (gy >= 0 && gy < H) fix(ly, c);
                }
            }
            // outside rows, every column (corners included)
            for (int i = tid; i < (ntr + nbr) * COV_W; i += HT_THREADS) {
                const int r = i / COV_W;
                fix(r < ntr ? r : rb0 + (r - ntr), i - r * COV_W);
            }
            __syncthreads();
        }
    }
    // ---- 7x7 box sums in fp64, one product plane at a time through ONE plane of horizontal sums (the three planes
    //      at once would be 59 KB and hold the SM at two CTAs; this way four fit):
    //        horizontal 7-sums: work item = (row, HS_SEG-output segment), a warp takes 32 consecutive rows of one
    //          segment -- the row pitches are odd, so its loads and 64-bit stores are free of bank conflicts; the six
    //          rows past 32 follow in the seventh warp
    //        vertical 7-sums:   thread = (column, 8-row segment); the seven rows of the first window stay in
    //          registers: they are exactly the rows that leave the window while it slides over the eight outputs
    const int x = tid % HT_W, oy0 = (tid / HT_W) * 8;
    const int gx = x0 + x;
    float bsum[3][8];
#pragma unroll
    for (int p = 0; p < 3; ++p) {
        if (p > 0) __syncthreads();   // every thread has finished reading the previous plane's sums
        if (tid < HS_NSEG * COV_ROWS) {
            const int sgm = tid < HS_NSEG * 32 ? tid >> 5 : (tid - HS_NSEG * 32) / (COV_ROWS - 32);
            const int r = tid < HS_NSEG * 32 ? tid & 31 : 32 + (tid - HS_NSEG * 32) % (COV_ROWS - 32);
            SVI_CHECK(1, r < COV_ROWS && sgm < HS_NSEG);
            const float* src = &sm.cov[p][r][sgm * HS_SEG];
            double v[HS_SEG + 6];
#pragma unroll
            for (int i = 0; i < HS_SEG + 6; ++i) v[i] = (double)src[i];   // the last segment reads into the row padding: unused sums
            double s = v[0];
#pragma unroll
            for (int i = 1; i < 7; ++i) s = __dadd_rn(s, v[i]);
            double* dst = &sm.hs[r][sgm * HS_SEG];
            dst[0] = s;
#pragma unroll
            for (int j = 1; j < HS_SEG; ++j) {
                s = __dadd_rn(s, __dsub_rn(v[j + 6], v[j - 1]));
                if (sgm * HS_SEG + j < HT_W) dst[j] = s;
            }
        }
        __syncthreads();
        double rw[7];
#pragma unroll
        for (int i = 0; i < 7; ++i) rw[i] = sm.hs[oy0 + i][x];
        double sv = rw[0];
#pragma unroll
        for (int i = 1; i < 7; ++i) sv = __dadd_rn(sv, rw[i]);
        bsum[p][0] = __double2float_rn(sv);
#pragma unroll
        for (int k = 1; k < 8; ++k) {
            sv = __dadd_rn(sv, __dsub_rn(sm.hs[oy0 + k + 6][x], rw[k - 1]));
            bsum[p][k] = __double2float_rn(sv);
        }
    }
    // ---- Harris; the responses stay in registers and go to a shared tile (the product planes are dead) for the
    //      neighbourhood test
    float lmax = -INFINITY;
    float rv[8];
    unsigned mbits = 0u;   // pixels of this thread that the mask admits
    float (*Rs)[HT_W] = reinterpret_cast<float(*)[HT_W]>(&sm.cov[0][0][0]);
    {
        float* rrow = resp ? resp + ((size_t)f * out_rows) * g.resp_pitch : nullptr;
        const uint8_t* mrow = mask ? mask + (size_t)f * g.img_stride : nullptr;
        const int rows_in = min(8, H - (y0 + oy0));   // rows of this thread inside the image (<= 0: none)
        // cv::cornerHarris (calcHarris) evaluates the response plane as ONE row of W*H pixels: 4-lane fp32 vectors with
        // (float)k, and a scalar tail for the last (W*H) % 4 pixels (the end of the last row) that computes
        // (float)(a*c - b*b - k*(a+c)*(a+c)) with the double k: det and a+c in fp32, the rest in fp64
        const float kf = (float)k;
        const long long tail_start = (long long)W * H - (((W & 3) * (H & 3)) & 3);
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            float R = -INFINITY;   // outside the image: ignored by the neighbourhood maximum
            if (gx < W && r < rows_in) {
                const float a = bsum[0][r], b = bsum[1][r], c = bsum[2][r];
                const float det = __fsub_rn(__fmul_rn(a, c), __fmul_rn(b, b));
                const float tr = __fadd_rn(a, c);
                const int gy = y0 + oy0 + r;
                if ((long long)gy * W + gx < tail_start)
                    R = __fsub_rn(det, __fmul_rn(__fmul_rn(kf, tr), tr));
                else
                    R = __double2float_rn(__dsub_rn((double)det, __dmul_rn(__dmul_rn(k, (double)tr), (double)tr)));
                if (rrow) rrow[(size_t)gy * g.resp_pitch + gx] = R;
                if (!mrow || mrow[(size_t)gy * g.img_pitch + gx]) {
                    lmax = fmaxf(lmax, R);
                    mbits |= 1u << r;
                }
            }
            rv[r] = R;
            SVI_CHECK(1, oy0 + r < HT_H && x < HT_W);
            Rs[oy0 + r][x] = R;
        }
    }
    uint32_t local_max = lmax == -INFINITY ? 0u : float_to_ordered(lmax);   // 0 = no admitted pixel
    local_max = warp_max_u32(local_max);
    if ((tid & 31) == 0) sm.red[tid >> 5] = local_max;
    __syncthreads();   // response tile complete; hs and the product planes are dead
    uint32_t tile_max = 0u;
#pragma unroll
    for (int i = 0; i < HT_THREADS / 32; ++i) tile_max = max(tile_max, sm.red[i]);
    if (tid == 0 && tile_max) atomicMax(frame_max + f, tile_max);

    // ---- 3x3 non-maximum suppression on the tile interior.  A thread owns 8 rows of one column: the vertical
    //      3-maxima come from its registers plus the rows above / below in the shared tile, the horizontal ones
    //      from the neighbouring lanes by shuffle (the column across the warp boundary from the shared tile).
    unsigned long long* s_keys = reinterpret_cast<unsigned long long*>(&sm.hs[0][0]);
    if (cand) {
        const int lane = tid & 31;
        const float thr = gftt_threshold(tile_max, quality);
        const float up = oy0 > 0 ? Rs[oy0 - 1][x] : -INFINITY;
        const float dn = oy0 + 8 < HT_H ? Rs[oy0 + 8][x] : -INFINITY;
        float c3[8], e3[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            c3[k] = fmaxf(fmaxf(k > 0 ? rv[k - 1] : up, rv[k]), k < 7 ? rv[k + 1] : dn);
            e3[k] = -INFINITY;
        }
        if (lane == 0 || lane == 31) {
            const int xn = lane == 0 ? x - 1 : x + 1;
            if (xn >= 0 && xn < HT_W) {
                float t[10];
#pragma unroll
                for (int i = 0; i < 10; ++i) {
                    const int row = oy0 - 1 + i;
                    t[i] = (row >= 0 && row < HT_H) ? Rs[row][xn] : -INFINITY;
                }
#pragma unroll
                for (int k = 0; k < 8; ++k) e3[k] = fmaxf(fmaxf(t[k], t[k + 1]), t[k + 2]);
            }
        }
        // candidate rows of this thread: tile interior (rows 1 .. HT_H-2) inside the image minus its 1-px border
        // (y <= H-2); bit k = row oy0 + k.  Columns: tile interior, x <= W-2 (x >= 1 and y >= 1 follow from the tile).
        unsigned allowed = 0u;
        {
            const int k_lo = oy0 == 0 ? 1 : 0;
            const int k_hi = min(min(7, HT_H - 2 - oy0), H - 2 - y0 - oy0);
            if (k_hi >= k_lo && x >= 1 && x <= HT_W - 2 && gx <= W - 2) allowed = (0xFFu >> (7 - k_hi)) & (0xFFu << k_lo);
        }
        allowed &= mbits;
        const float thr0 = fmaxf(thr, 0.f);   // a candidate has R' = R > thr and R' != 0; thr >= 0 whenever max R > 0
        unsigned mine = 0u;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            float l3 = __shfl_up_sync(0xFFFFFFFFu, c3[k], 1), r3 = __shfl_down_sync(0xFFFFFFFFu, c3[k], 1);
            if (lane == 0) l3 = e3[k];
            if (lane == 31) r3 = e3[k];
            const float v = rv[k];
            if (v > thr0 && v == fmaxf(fmaxf(l3, c3[k]), r3)) mine |= 1u << k;
        }
        mine &= allowed;
        // same-address atomics serialise: aggregate per warp (one scan of the per-thread counts), then per CTA
        // (shared counter); the CTA claims its slice of the frame's list with ONE global atomic below
        if (__any_sync(0xFFFFFFFFu, mine != 0u)) {
            const int cnt = __popc(mine);
            int incl = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int u = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                if (lane >= o) incl += u;
            }
            int base = 0;
            if (lane == 31) base = atomicAdd(&sm.key_count, incl);
            base = __shfl_sync(0xFFFFFFFFu, base, 31) + incl - cnt;
            const unsigned yx0 = ((unsigned)(y0 + oy0) << 16) | (unsigned)gx;
            while (mine) {   // a thread rarely holds more than one local maximum
                const int k = __ffs(mine) - 1;
                mine &= mine - 1u;
                float v = rv[0];
#pragma unroll
                for (int i = 1; i < 8; ++i) v = (k == i) ? rv[i] : v;
                SVI_CHECK(1, base >= 0 && base < HT_MAX_KEYS);
                s_keys[base++] = ((unsigned long long)float_to_ordered(v) << 32) | (yx0 + ((unsigned)k << 16));
            }
        }
    }
    __syncthreads();   // key list complete; the response tile is dead -> its memory becomes the 9-sum rows
    const int n_keys = sm.key_count;
    if (tid == 0 && n_keys) sm.key_base = atomicAdd(cand_count + f, n_keys);
    uint16_t (*h9)[H9_P] = reinterpret_cast<uint16_t(*)[H9_P]>(&sm.cov[0][0][0]);
    if (box) box9_rows(sm.tile, h9);   // whole-frame mode only
    __syncthreads();
    if (n_keys) {
        const int base = sm.key_base;
        unsigned long long* dst = cand + (size_t)f * cand_cap;
        for (int i = tid; i < n_keys; i += HT_THREADS)
            if (base + i < cand_cap) dst[base + i] = s_keys[i];   // an overflowing list is reported by select_corners_kernel
    }
    if (box) {
        const size_t fo = (size_t)f * H * g.box_pitch;
        box9_cols(h9, box + fo, box_shift ? box_shift + fo : nullptr, g.box_pitch, W, H, x0, y0);
    }
}

// ------------------------------------------------------------------ FAST-9/16 (optional detector mode)
// cv::FAST(img, kps, threshold, nonmax, TYPE_9_16) (OpenCV fast.cpp FAST_t<16>, cornerScore<16>): corner test on
// the 16-pixel circle, score = largest threshold that keeps the corner, 3x3 non-max suppression with strict >,
// 3-px image border excluded.  Same 64x32 tile + 4-px halo staging as the Harris kernel; the scores of the tile
// and a 1-px ring around it live in shared memory for the suppression.  Emits keys whose descending order is
// OpenCV's output order (scan order): high word = ~(y << 16 | x), low word = y << 16 | x.
__device__ __forceinline__ int fast_ring(const uint8_t (*tile)[U8_P], int ty, int tx, int k) {
    // (dx, dy) of OpenCV's makeOffsets(), k taken modulo 16
    constexpr signed char DX[16] = {0, 1, 2, 3, 3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1};
    constexpr signed char DY[16] = {3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1, 0, 1, 2, 3};
    return tile[ty + DY[k & 15]][tx + DX[k & 15]];
}

__device__ __forceinline__ int fast_corner_score(const uint8_t (*tile)[U8_P], int ty, int tx, int threshold) {
    const int v = tile[ty][tx];
    int d[25];
#pragma unroll
    for (int k = 0; k < 25; ++k) d[k] = v - fast_ring(tile, ty, tx, k);
    int a0 = threshold;
#pragma unroll
    for (int k = 0; k < 16; k += 2) {
        int a = min(min(d[k + 1], d[k + 2]), d[k + 3]);
        if (a <= a0) continue;
        a = min(min(min(a, d[k + 4]), min(d[k + 5], d[k + 6])), min(d[k + 7], d[k + 8]));
        a0 = max(a0, min(a, d[k]));
        a0 = max(a0, min(a, d[k + 9]));
    }
    int b0 = -a0;
#pragma unroll
    for (int k = 0; k < 16; k += 2) {
        int b = max(max(max(d[k + 1], d[k + 2]), max(d[k + 3], d[k + 4])), d[k + 5]);
        if (b >= b0) continue;
        b = max(max(b, d[k + 6]), max(d[k + 7], d[k + 8]));
        b0 = min(b0, max(b, d[k]));
        b0 = min(b0, max(b, d[k + 9]));
    }
    return -b0 - 1;
}

__global__ void __launch_bounds__(HT_THREADS)
fast_candidates_kernel(const uint8_t* __restrict__ img, const uint8_t* __restrict__ mask, FrameGeom g, int threshold, int nonmax,
                       unsigned long long* __restrict__ cand, int* __restrict__ cand_count, int cand_cap) {
    __shared__ __align__(16) uint8_t tile[U8_ROWS][U8_P];
    __shared__ uint16_t score[HT_H + 2][HT_W + 2];      // bit 8 = corner, low byte = score stored as uchar like OpenCV
    __shared__ unsigned long long s_keys[512];
    __shared__ int s_count, s_base;
    const int f = blockIdx.z, x0 = blockIdx.x * HT_W, y0 = blockIdx.y * HT_H, tid = threadIdx.x;
    if (tid == 0) s_count = 0;
    load_tile_u8(tile, img + (size_t)f * g.img_stride, g.img_pitch, g.W, g.H, x0, y0);
    __syncthreads();
    const int t = min(max(threshold, 0), 255);
    for (int idx = tid; idx < (HT_H + 2) * (HT_W + 2); idx += HT_THREADS) {
        const int ly = idx / (HT_W + 2), lx = idx - ly * (HT_W + 2);
        const int gx = x0 - 1 + lx, gy = y0 - 1 + ly;
        uint16_t sc = 0;
        if (gx >= 3 && gx < g.W - 3 && gy >= 3 && gy < g.H - 3) {
            const int ty = ly + 3, tx = lx + 3;        // tile origin is (x0 - 4, y0 - 4)
            const int v = tile[ty][tx];
            uint32_t dark = 0u, bright = 0u;
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                const int p = fast_ring(tile, ty, tx, k);
                dark |= (uint32_t)(p < v - t) << k;
                bright |= (uint32_t)(p > v + t) << k;
            }
            // >= 9 contiguous set bits on the circle: AND of 9 rotations of the doubled mask
            uint32_t r = dark | (dark << 16), x = r & (r >> 1);
            x &= x >> 2; x &= x >> 4; x &= r >> 8;
            uint32_t r2 = bright | (bright << 16), y = r2 & (r2 >> 1);
            y &= y >> 2; y &= y >> 4; y &= r2 >> 8;
            if ((x | y) & 0xFFFFu) sc = 0x100u | (uint16_t)(uint8_t)fast_corner_score(tile, ty, tx, t);
        }
        score[ly][lx] = sc;
    }
    __syncthreads();
    for (int idx = tid; idx < HT_H * HT_W; idx += HT_THREADS) {
        const int ly = idx / HT_W, lx = idx - ly * HT_W;
        const int gx = x0 + lx, gy = y0 + ly;
        const uint16_t c = score[ly + 1][lx + 1];
        if (!(c & 0x100u) || gx >= g.W || gy >= g.H) continue;
        bool keep = true;
        if (nonmax) {
            const int sv = c & 0xFF;
#pragma unroll
            for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                for (int dx = 0; dx < 3; ++dx)
                    if (dy != 1 || dx != 1) keep &= sv > (score[ly + dy][lx + dx] & 0xFF);
        }
        if (keep && mask && !mask[(size_t)f * g.img_stride + (size_t)gy * g.img_pitch + gx]) keep = false;
        if (keep) {
            const int pos = atomicAdd(&s_count, 1);
            const unsigned xy = ((unsigned)gy << 16) | (unsigned)gx;
            if (pos < 512) s_keys[pos] = ((unsigned long long)(0xFFFFFFFFu - xy) << 32) | xy;
            else {   // more than 512 corners in one tile (cannot happen with nonmax): straight to the global list
                const int gp = atomicAdd(cand_count + f, 1);
                if (gp < cand_cap) cand[(size_t)f * cand_cap + gp] = ((unsigned long long)(0xFFFFFFFFu - xy) << 32) | xy;
            }
        }
    }
    __syncthreads();
    const int n = min(s_count, 512);
    if (n == 0) return;
    if (tid == 0) s_base = atomicAdd(cand_count + f, n);
    __syncthreads();
    for (int i = tid; i < n; i += HT_THREADS)
        if (s_base + i < cand_cap) cand[(size_t)f * cand_cap + s_base + i] = s_keys[i];
}

}  // namespace svi
