// K3: pyramidal Lucas-Kanade, one warp per feature point, all levels and iterations, forward and
// backward pass plus the forward-backward check in one launch (SURVEY.md A.5, A.7).
// Replaces the two cv2.calcOpticalFlowPyrLK calls and the numpy FB arithmetic at
// s1_lucaskanade_tracking.py:323-333 (s0_1_test_lucaskanade_tracking.py:92-102).
//
// Per level a warp
//  (a) stages everything the level can touch into its private shared-memory slab in one burst: three TMA bulk tensor
//      copies (per-warp mbarriers; box origins on 16-byte boundaries) bring the I window, its Scharr planes (TMA zero
//      fill = OpenCV's zero-padded derivative planes) and the J search patch around the propagated guess (window + 1 +
//      2*MARGIN px).  Intensity patches that overhang the image are mirrored (REFLECT_101) inside shared memory after the
//      zero-filling copy; cp.async / gather paths remain for far-out windows and images that are not 16-byte aligned;
//  (b) builds the template: lane = window column, rows walked top to bottom.  Per window pixel the slab keeps only the
//      int16 pair (Ix, Iy) -- 4 bytes, Ix and Iy of 4 columns grouped (tmpl_store) -- and the pass accumulates, exactly,
//      the structure tensor and the two constants C1 = sum(Iw*Ix), C2 = sum(Iw*Iy).  The template rows overwrite the
//      Scharr patch rows already consumed;
//  (c) runs the Newton iterations out of shared memory with a different lane mapping: lane = (row group, column quad),
//      4 adjacent columns x RG consecutive rows.  Per row a lane loads the two aligned words that hold its 5 J bytes,
//      two PRMTs (warp-uniform selectors) turn them into the byte windows (b0..b3), (b1..b4), and dp2a.lo / dp2a.hi on
//      those against OpenCV's packed 14-bit weights give the four bilinear samples; one 16-byte load brings the four
//      template entries, and the products with them run on dp2a as well (samples split into bytes).  The mismatch vector
//      is  b = sum(Jw*Ix) - C1  (sum(Jw*Iy) - C2): identical, as an exact integer, to OpenCV's sum((Jw - Iw)*Ix), and it
//      halves the template.  Template entries outside the window are zero, so the iteration loop carries no masks.
// Multi-channel frames (cv2 takes 3- and 4-channel images) run the same solver with every window sum taken over the channel
// planes as well, on the runtime-window kernel without tensor maps.
// All sums are exact integers (int32 per lane, REDUX across the warp, int64 totals) rounded to float once; OpenCV
// accumulates in float SIMD lanes, which differs in the last bits only.  Float arithmetic that OpenCV does unfused is
// compiled with -fmad=false.
#include "common.cuh"
#include <stdlib.h>
#include <string.h>
#include <type_traits>
#include <mutex>
#include <vector>

namespace ibt {

constexpr int LK_MARGIN = 3;        // px the window may drift inside a staged patch, each direction

// ---- slab geometry as a function of the window size (shared by host launch code and the specialised kernels) ----------
// Newton mapping: NL lanes per row group (4 columns each), NG row groups of RG rows; the template is TROWS x TCOLS.
__host__ __device__ constexpr int lk_nl(int w) { return (w + 3) / 4; }
__host__ __device__ constexpr int lk_tcols(int w) { return 4 * lk_nl(w); }
__host__ __device__ constexpr int lk_ng0(int w, int h) { return (32 / lk_nl(w)) < h ? (32 / lk_nl(w)) : h; }
__host__ __device__ constexpr int lk_rg(int w, int h) { return (h + lk_ng0(w, h) - 1) / lk_ng0(w, h); }
__host__ __device__ constexpr int lk_ng(int w, int h) { return (h + lk_rg(w, h) - 1) / lk_rg(w, h); }
__host__ __device__ constexpr int lk_trows(int w, int h) { return lk_ng(w, h) * lk_rg(w, h); }
// template-build mapping: lane = column of a strip of <= 32 of the TCOLS template columns
__host__ __device__ constexpr int lk_nstrips(int w) { return (lk_tcols(w) + 31) / 32; }
__host__ __device__ constexpr int lk_strip_cols(int w) { return (lk_tcols(w) + lk_nstrips(w) - 1) / lk_nstrips(w); }
// window widths whose compiled-in kernel builds the template with build_template_split (columns 32.. spread over the lanes)
__host__ __device__ constexpr bool lk_split(int w) { return w == 35; }
// every lane of every strip reads two adjacent elements per row, active or not: pitches keep those reads in the slab
__host__ __device__ constexpr int lk_reach(int w) { return lk_split(w) ? lk_tcols(w) + 1 : (lk_nstrips(w) - 1) * lk_strip_cols(w) + 33; }
__host__ __device__ constexpr int lk_dpitch(int w) { return (lk_reach(w) + 6) & ~3; }                 // words; rows are 16-byte multiples (TMA box); + window offset 0..3
// TMA boxes start on 16-byte boundaries of the image row: up to 15 extra columns on the left
__host__ __device__ constexpr int lk_ipitch(int w) { return (15 + lk_reach(w) + 15) & ~15; }
// Newton lanes read the two aligned words around bytes [ox + 4c, ox + 4c + 4], ox <= 15 + 2*MARGIN
__host__ __device__ constexpr int lk_jpitch(int w) { return (15 + 2 * LK_MARGIN + lk_tcols(w) + 4 + 15) & ~15; }

struct LKLevel {
    const uint8_t *img;
    const uint32_t *deriv;      // packed (dx | dy << 16), may be null for a J-only pyramid
    int img_pitch;              // bytes
    int deriv_pitch;            // 4-byte elements
    int rows, cols;
    int word_ok;                // img and img_pitch are 4-byte aligned: patch staging may use 4-byte cp.async
    int tma_img, tma_der;       // tensor maps exist for this level (16-byte aligned base and pitch)
};
struct LKPyr {
    LKLevel lv[IBT_MAX_LEVELS];
    int nlevels;
};
// tensor maps of both pyramids: [pyramid][level]; boxes = I window, J search patch, Scharr window
struct LKMaps {
    CUtensorMap imgI[2][IBT_MAX_LEVELS], imgJ[2][IBT_MAX_LEVELS], der[2][IBT_MAX_LEVELS];
};
// Multi-channel frames (ibt_lk_multichannel): cn single-channel pyramids per frame, one per channel plane (built by the
// single-channel kernels).  OpenCV sums every window quantity (structure tensor, mismatch vector, residual) over the window
// pixels AND the channels; the min-eigenvalue test and the Newton update are unchanged, err is divided by 32 * winW * cn * winH.
// These pyramids carry no tensor maps, so they are staged by cp.async and the gather.
constexpr int LK_MC_MAX = 4;
struct LKMcPyr {
    LKPyr I[LK_MC_MAX], J[LK_MC_MAX];
    int cn;
};

struct LKArgs {
    LKPyr pyr[2];               // [0] = prev, [1] = next
    const float *p0;
    int n;
    int winW, winH;
    int nl, ng, rg, trows, tcols;           // Newton mapping / template shape
    int nstrips, strip_cols;                // template-build mapping
    // per-warp shared-memory slab: [template (Ix,Iy) words, overlaid on the Scharr patch][I patch][J patch]
    int dpitch;                 // deriv patch row pitch, words
    int ipitch;                 // I patch row pitch, bytes (multiple of 16)
    int jpitch, jrows;          // J patch row pitch (bytes, multiple of 16) and staged rows (window + 1 + 2*MARGIN)
    unsigned int *work_counter; // [0] next point index (dynamic point -> warp assignment), [1] warps that have left
    unsigned int total_warps;
    int off_ipatch, off_jpatch, warp_smem;     // bytes (template and Scharr patch start at 0)
    int maxCount;
    float eps2, minEigThr;
    int flags;
    int fb;                     // 0: single pass A->B ; 1: forward + backward + FB check
    float fb_thresh;
    float *p1; uint8_t *st1; float *err1;
    float *p0r; uint8_t *st0; float *err0;
    float *fbdist; uint8_t *alive; int32_t *iters; unsigned long long *iter_total;
};

// exact warp sum of int32 lane values (|v| < 2^31) as int64: two REDUX instead of ten shuffles
__device__ __forceinline__ long long warp_sum_wide(int v)
{
    const int lo = __reduce_add_sync(0xffffffffu, v & 0xffff);
    const int hi = __reduce_add_sync(0xffffffffu, v >> 16);
    return ((long long)hi << 16) + lo;
}

__device__ __forceinline__ int cv_floor(float v) { return __float2int_rd(v); }
// OpenCV's cvFloor gives INT_MIN for NaN on x86, so cv2 finds the window of a NaN point or guess out of bounds at every level
// (status 0, err 0, nextPts = the propagated input).  PTX converts NaN to 0, which would put that window at the origin.  The
// coordinates that can be NaN -- the point and the guess at each level, the final position -- pass through no_nan before they
// are floored (-inf floors to INT_MIN); the Newton iterates of a finite guess stay finite, so the iteration loop needs no test.
// +-inf and |v| >= 2^31 saturate to INT_MIN / INT_MAX (INT_MIN on x86): out of bounds either way.
__device__ __forceinline__ float no_nan(float v) { return v == v ? v : __int_as_float(0xff800000); }

// The FB distance as numpy's float32 hypot computes it (s1:330): glibc's hypotf, the double square root of the exact double
// sum of squares rounded to float, and +inf if either input is infinite even when the other is NaN (the sum alone would
// give NaN there; a NaN otherwise propagates).  CUDA's hypotf differs in the last bit, and dist < fb_thresh and the
// trackquality files rest on these bits.
__device__ __forceinline__ float glibc_hypotf(float x, float y)
{
    if (isinf(x) || isinf(y)) return __int_as_float(0x7f800000);
    const double a = x, b = y;
    return __double2float_rn(__dsqrt_rn(__dadd_rn(__dmul_rn(a, a), __dmul_rn(b, b))));
}

// d = c + a.lo16 * b.byte0 + a.hi16 * b.byte1 (.lo) / b.byte2, b.byte3 (.hi) with SIGNED 16-bit weights (iw11 = 2^14 - iw00 -
// iw01 - iw10 can be -1 after rounding) and UNSIGNED pixel bytes.
__device__ __forceinline__ uint32_t dp2a_lo(uint32_t a, uint32_t b, uint32_t c)
{
    int d;
    asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"((int)c));
    return (uint32_t)d;
}
__device__ __forceinline__ uint32_t dp2a_hi(uint32_t a, uint32_t b, uint32_t c)
{
    int d;
    asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"((int)c));
    return (uint32_t)d;
}

__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async4(unsigned smem_dst, const void *gsrc)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async4_zfill(unsigned smem_dst, const void *gsrc, int src_size)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(smem_dst), "l"(gsrc), "r"(src_size) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// OpenCV's integer bilinear weights, packed for dp2a: wtop = iw00 | iw01 << 16, wbot = iw10 | iw11 << 16.
__device__ __forceinline__ void bilinear_weights(float a, float b, uint32_t &wtop, uint32_t &wbot,
                                                 int &iw00, int &iw01, int &iw10, int &iw11)
{
    const float oa = __fsub_rn(1.f, a), ob = __fsub_rn(1.f, b);
    iw00 = __float2int_rn(__fmul_rn(__fmul_rn(oa, ob), 16384.f));
    iw01 = __float2int_rn(__fmul_rn(__fmul_rn(a, ob), 16384.f));
    iw10 = __float2int_rn(__fmul_rn(__fmul_rn(oa, b), 16384.f));
    iw11 = 16384 - iw00 - iw01 - iw10;
    wtop = ((uint32_t)iw00 & 0xffffu) | ((uint32_t)iw01 << 16);
    wbot = ((uint32_t)iw10 & 0xffffu) | ((uint32_t)iw11 << 16);
}

__device__ __forceinline__ bool window_oob(int ix, int iy, int winW, int winH, int rows, int cols)
{
    return ix < -winW || ix >= cols || iy < -winH || iy >= rows;
}

// ---- staging ---------------------------------------------------------------------------------------------
// Border variant of stage_bytes: REFLECT_101 gather (column indices resolved once per lane, rows batched four at a time).
// Kept out of line: it is rare and would otherwise bloat the hot instruction stream.
__device__ __noinline__ void stage_bytes_border(const LKLevel &L, int x0a, int y0, int nrows, int pitch, uint8_t *dst, int lane)
{
    for (int c = lane; c < pitch; c += 32) {
        const uint8_t *s = L.img + r101(x0a + c, L.cols);
        uint8_t *d = dst + c;
        int r = 0;
        for (; r + 4 <= nrows; r += 4) {
            const uint8_t v0 = __ldg(s + (int64_t)r101(y0 + r, L.rows) * L.img_pitch);
            const uint8_t v1 = __ldg(s + (int64_t)r101(y0 + r + 1, L.rows) * L.img_pitch);
            const uint8_t v2 = __ldg(s + (int64_t)r101(y0 + r + 2, L.rows) * L.img_pitch);
            const uint8_t v3 = __ldg(s + (int64_t)r101(y0 + r + 3, L.rows) * L.img_pitch);
            d[r * pitch] = v0; d[(r + 1) * pitch] = v1; d[(r + 2) * pitch] = v2; d[(r + 3) * pitch] = v3;
        }
        for (; r < nrows; r++) d[r * pitch] = __ldg(s + (int64_t)r101(y0 + r, L.rows) * L.img_pitch);
    }
}

// Stage image rows [y0, y0+nrows) x bytes [x0a, x0a+pitch) (x0a a multiple of 4) into dst (row pitch `pitch`).
// Interior patches go as 4-byte cp.async (lane -> (row sr + k*rpp, word sw)); patches that touch the border are
// gathered through REFLECT_101.  The caller commits / waits.
__device__ __forceinline__ void stage_bytes(const LKLevel &L, int x0a, int y0, int nrows, int pitch, int lane, uint8_t *dst)
{
    const bool interior = L.word_ok && x0a >= 0 && y0 >= 0 && y0 + nrows <= L.rows && x0a + pitch <= L.cols;
    if (interior) {
        const int ppw = pitch >> 2;                 // words per row (<= 32: pitches are at most 128 bytes)
        const int rpp = 32 / ppw;                   // rows covered per pass
        const int sr = lane / ppw, sw = lane - sr * ppw;
        if (sr < rpp) {
            const uint8_t *src = L.img + (int64_t)(y0 + sr) * L.img_pitch + x0a + 4 * sw;
            unsigned d = smem_u32(dst) + sr * pitch + 4 * sw;
            const int64_t sstep = (int64_t)rpp * L.img_pitch;
            const int dstep = rpp * pitch;
#pragma unroll 4
            for (int r = sr; r < nrows; r += rpp) {
                cp_async4(d, src);
                src += sstep; d += dstep;
            }
        }
    } else {
        stage_bytes_border(L, x0a, y0, nrows, pitch, dst, lane);
    }
}

// REFLECT_101 of a TMA-staged intensity patch inside shared memory.  The bulk tensor copy zero-fills what lies outside
// the image; when every mirror source of the needed region [nx0, nx1] x [y0, y0 + nrows) lies inside that region (and
// inside the image) the out-of-image rows, then columns, are copied from the patch itself.  patch_reflectable() is the
// warp-uniform test; windows further out take the gather path.
__device__ __forceinline__ bool patch_reflectable(int nx0, int nx1, int y0, int nrows, int rows, int cols)
{
    const int y1 = y0 + nrows - 1;
    return -nx0 <= nx1 && -nx0 < cols && 2 * (cols - 1) - nx1 >= nx0 && 2 * (cols - 1) - nx1 >= 0 &&
           -y0 <= y1 && -y0 < rows && 2 * (rows - 1) - y1 >= y0 && 2 * (rows - 1) - y1 >= 0;
}
__device__ __noinline__ void patch_reflect(uint8_t *patch, int pitch, int x0a, int nx0, int nx1, int y0, int nrows, int rows,
                                           int cols, int lane)
{
    __syncwarp();
    const int pw = pitch >> 2;
    const int ntop = min(nrows, max(0, -y0));                     // patch rows above the image
    const int rbot = max(0, rows - y0);                           // first patch row below the image
    for (int i = lane; i < (ntop + max(0, nrows - rbot)) * pw; i += 32) {       // rows first (whole staged width)
        int r = i / pw;
        const int c = i - r * pw;
        if (r >= ntop) r = rbot + (r - ntop);
        const int y = y0 + r;
        const int rs = (y < 0 ? -y : 2 * (rows - 1) - y) - y0;
        reinterpret_cast<uint32_t *>(patch + r * pitch)[c] = reinterpret_cast<const uint32_t *>(patch + rs * pitch)[c];
    }
    __syncwarp();
    const int nleft = min(nx1 - nx0 + 1, max(0, -nx0));           // needed columns left of the image
    const int xright = max(nx0, cols);                            // first needed column right of the image
    const int ncol = nleft + max(0, nx1 - xright + 1);
    for (int i = lane; i < ncol * nrows; i += 32) {               // then the needed columns outside the image
        int k = i / nrows;
        const int r = i - k * nrows;
        const int x = k < nleft ? nx0 + k : xright + (k - nleft);
        const int xs = (x < 0 ? -x : 2 * (cols - 1) - x) - x0a, xd = x - x0a;
        patch[r * pitch + xd] = patch[r * pitch + xs];
    }
    __syncwarp();
}

// Re-stage the J patch synchronously (the window drifted out of the prefetched patch): rare, kept out of line.
__device__ __noinline__ void restage_sync(const LKLevel &L, int x0a, int y0, int nrows, int pitch, uint8_t *dst, int lane)
{
    __syncwarp();
    stage_bytes(L, x0a, y0, nrows, pitch, lane, dst);
    cp_async_commit();
    cp_async_wait<0>();
    __syncwarp();
}

// Stage the Scharr planes of the template window: rows [y0, y0+winH], columns [x0, x0+winW]; zero outside the image.
template <int WW, int WH>
__device__ __forceinline__ void stage_deriv(const LKLevel &L, const LKArgs &a, int x0, int y0, uint32_t *dst, int lane)
{
    const int winW = WW ? WW : a.winW, winH = WH ? WH : a.winH;
    const int DP = WW ? lk_dpitch(WW) : a.dpitch;
    const bool interior = x0 >= 0 && y0 >= 0 && x0 + winW < L.cols && y0 + winH < L.rows;
    for (int c = lane; c <= winW; c += 32) {
        const uint32_t *src = L.deriv + (int64_t)y0 * L.deriv_pitch + x0 + c;
        unsigned d = smem_u32(dst + c);
        if (interior) {
#pragma unroll 8
            for (int r = 0; r <= winH; r++) {
                cp_async4(d, src);
                src += L.deriv_pitch; d += DP * 4;
            }
        } else {
            const bool xin = (unsigned)(x0 + c) < (unsigned)L.cols;
            for (int r = 0; r <= winH; r++) {
                const bool ok = xin && (unsigned)(y0 + r) < (unsigned)L.rows;
                cp_async4_zfill(d, ok ? src : L.deriv, ok ? 4 : 0);
                src += L.deriv_pitch; d += DP * 4;
            }
        }
    }
}

// ---- template --------------------------------------------------------------------------------------------
// Template layout: a row is TCOLS int16 pairs (4 * TCOLS bytes), in quads of 4 columns.  A quad's 16 bytes hold
// Ix0 Ix1 Ix2 Ix3 Iy0 Iy1 Iy2 Iy3 (int16), so the Newton lane's one 16-byte load gives dp2a-ready pairs: x = (Ix0, Ix1),
// y = (Ix2, Ix3), z = (Iy0, Iy1), w = (Iy2, Iy3).  Column c keeps Ix at halfword (c >> 2) * 8 + (c & 3) of its row, Iy 4
// halfwords later.
__device__ __forceinline__ void tmpl_store(uint32_t *tmpl, int row, int tc, int c, int Ix, int Iy)
{
    int16_t *h = reinterpret_cast<int16_t *>(tmpl) + 2 * row * tc + (c >> 2) * 8 + (c & 3);
    h[0] = (int16_t)Ix;
    h[4] = (int16_t)Iy;
}

// lane = template column (strips of <= 32 columns), rows top to bottom.  Writes column col of row r (tmpl_store) for the
// TROWS x TCOLS template (zero outside the window) and returns the exact sums
//   A11 = sum Ix^2, A12 = sum Ix*Iy, A22 = sum Iy^2, C1 = sum Iw*Ix, C2 = sum Iw*Iy.
// The template row r overwrites Scharr patch bytes below row r+1 only (TCOLS <= DPITCH), which every lane has consumed
// by then (one __syncwarp per row keeps the lanes within a row of each other).
// Windows 33 .. 36 px wide (the reference's own 35 x 35): a second 32-lane strip would run the whole row loop again for 1 .. 4
// columns.  Instead the columns 32 .. TCOLS-1 are spread over the 32 lanes as (column, row phase): a lane handles rows
// ph, ph + PH, ... of one of them (5 pixels at 35 x 35) without a row-to-row carry.  That pass runs FIRST (the template overlays
// the Scharr patch and would overwrite what it reads), keeps its results in registers, and stores them after the main strip.
template <int WW, int WH>
__device__ __forceinline__ void build_template_split(const uint8_t *ip0, const uint32_t *dp0, uint32_t *tmpl, uint32_t wtop,
                                                     uint32_t wbot, int iw00, int iw01, int iw10, int iw11, int lane,
                                                     long long &sA11, long long &sA12, long long &sA22, long long &sC1, long long &sC2)
{
    constexpr int TC = lk_tcols(WW), TR = lk_trows(WW, WH), IP = lk_ipitch(WW), DP = lk_dpitch(WW);
    constexpr int C1 = TC - 32, PH = 32 / C1, NR = (WH + PH - 1) / PH;
    static_assert(C1 >= 1 && C1 <= 4 && (32 % C1) == 0 || C1 == 3, "split template: 1, 2 or 4 extra columns");
    // ---- the extra columns ------------------------------------------------------------------------------------------------------
    const int xc = 32 + lane % C1, ph = lane / C1;
    const bool lane1 = ph < PH;
    uint32_t tv[NR];
    int e11 = 0, e12 = 0, e22 = 0, ec1 = 0, ec2 = 0;
#pragma unroll
    for (int i = 0; i < NR; i++) {
        const int r = ph + PH * i;
        const bool act = lane1 && r < WH && xc < WW;
        const int rr = act ? r : 0;                              // (idle lanes read row 0: any staged address will do)
        const uint8_t *ip = ip0 + rr * IP + xc;
        const uint32_t *dp = dp0 + rr * DP + xc;
        const uint32_t p0 = (uint32_t)ip[0] | ((uint32_t)ip[1] << 8), p1 = (uint32_t)ip[IP] | ((uint32_t)ip[IP + 1] << 8);
        const uint32_t q00 = dp[0], q01 = dp[1], q10 = dp[DP], q11 = dp[DP + 1];
        const uint32_t v = dp2a_lo(wbot, p1, dp2a_lo(wtop, p0, 256u));
        int Iw = (int)(v >> 9);
        int Ix = ((int)(short)(q00 & 0xffffu) * iw00 + (int)(short)(q01 & 0xffffu) * iw01 + (int)(short)(q10 & 0xffffu) * iw10 +
                  (int)(short)(q11 & 0xffffu) * iw11 + 8192) >> 14;
        int Iy = (((int)q00 >> 16) * iw00 + ((int)q01 >> 16) * iw01 + ((int)q10 >> 16) * iw10 + ((int)q11 >> 16) * iw11 + 8192) >> 14;
        if (!act) { Iw = 0; Ix = 0; Iy = 0; }
        tv[i] = ((uint32_t)Ix << 16) | ((uint32_t)Iy & 0xffffu);
        e11 += Ix * Ix; e12 += Ix * Iy; e22 += Iy * Iy; ec1 += Iw * Ix; ec2 += Iw * Iy;
    }
    __syncwarp();
    // ---- the main strip: columns 0 .. 31, one per lane, rows top to bottom (all inside the window) ----------------------------------
    int a11 = 0, a12 = 0, a22 = 0, c1 = 0, c2 = 0;
    const uint8_t *ipl = ip0 + lane;
    const uint32_t *dpl = dp0 + lane;
    uint32_t ipair = (uint32_t)ipl[0] | ((uint32_t)ipl[1] << 8);
    int d00x, d00y, d01x, d01y;
    {
        const uint32_t dc = dpl[0], dcr = dpl[1];
        d00x = (int)(short)(dc & 0xffffu); d00y = (int)dc >> 16;
        d01x = (int)(short)(dcr & 0xffffu); d01y = (int)dcr >> 16;
    }
#pragma unroll 4
    for (int r = 0; r < WH; r++) {
        const uint8_t *ip = ipl + (r + 1) * IP;
        const uint32_t *dp = dpl + (r + 1) * DP;
        const uint32_t cpair = (uint32_t)ip[0] | ((uint32_t)ip[1] << 8);
        const uint32_t dc = dp[0], dcr = dp[1];
        const int d10x = (int)(short)(dc & 0xffffu), d10y = (int)dc >> 16;
        const int d11x = (int)(short)(dcr & 0xffffu), d11y = (int)dcr >> 16;
        uint32_t v = dp2a_lo(wtop, ipair, 256u);
        v = dp2a_lo(wbot, cpair, v);
        const int Iw = (int)(v >> 9);
        const int Ix = (d00x * iw00 + d01x * iw01 + d10x * iw10 + d11x * iw11 + 8192) >> 14;
        const int Iy = (d00y * iw00 + d01y * iw01 + d10y * iw10 + d11y * iw11 + 8192) >> 14;
        tmpl_store(tmpl, r, TC, lane, Ix, Iy);
        a11 += Ix * Ix; a12 += Ix * Iy; a22 += Iy * Iy;
        c1 += Iw * Ix; c2 += Iw * Iy;
        ipair = cpair; d00x = d10x; d00y = d10y; d01x = d11x; d01y = d11y;
        __syncwarp();            // the template overlays the Scharr patch rows already consumed (see launch_lk)
    }
    // ---- the extra columns' entries, the template rows below the window -------------------------------------------------------------
#pragma unroll
    for (int i = 0; i < NR; i++) {
        const int r = ph + PH * i;
        if (lane1 && r < WH) tmpl_store(tmpl, r, TC, xc, (int)tv[i] >> 16, (int)(short)(tv[i] & 0xffffu));
    }
    for (int i = WH * TC + lane; i < TR * TC; i += 32) tmpl[i] = 0u;
    sA11 = warp_sum_wide(a11) + warp_sum_wide(e11); sA12 = warp_sum_wide(a12) + warp_sum_wide(e12);
    sA22 = warp_sum_wide(a22) + warp_sum_wide(e22);
    sC1 = warp_sum_wide(c1) + warp_sum_wide(ec1); sC2 = warp_sum_wide(c2) + warp_sum_wide(ec2);
    __syncwarp();
}

template <int WW, int WH>
__device__ __forceinline__ void build_template(const LKArgs &a, const uint8_t *ip0, const uint32_t *dp0, uint32_t *tmpl,
                                               uint32_t wtop, uint32_t wbot, int iw00, int iw01, int iw10, int iw11, int lane,
                                               long long &sA11, long long &sA12, long long &sA22, long long &sC1, long long &sC2)
{
    if (WW > 0 && WH > 0 && lk_split(WW)) {
        build_template_split<lk_split(WW) ? WW : 35, WH ? WH : 35>(ip0, dp0, tmpl, wtop, wbot, iw00, iw01, iw10, iw11, lane,
                                                                             sA11, sA12, sA22, sC1, sC2);
        return;
    }
    const int winW = WW ? WW : a.winW, winH = WH ? WH : a.winH;
    constexpr int NS = WW ? lk_nstrips(WW) : 2;                 // strips held in registers (generic kernel: at most 2)
    const int nstrips = WW ? lk_nstrips(WW) : a.nstrips, SC = WW ? lk_strip_cols(WW) : a.strip_cols;
    const int TC = WW ? lk_tcols(WW) : a.tcols, TR = (WW && WH) ? lk_trows(WW, WH) : a.trows;
    const int IP = WW ? lk_ipitch(WW) : a.ipitch, DP = WW ? lk_dpitch(WW) : a.dpitch;
    int a11[NS], a12[NS], a22[NS], c1[NS], c2[NS];
    uint32_t ipair[NS];
    int d00x[NS], d00y[NS], d01x[NS], d01y[NS];
    // lanes beyond the window take all-zero weights: Iw = Ix = Iy = 0 there without a per-row select, which is exactly what the
    // template must hold outside the window
    uint32_t mtop[NS], mbot[NS];
    int m00[NS], m01[NS], m10[NS], m11[NS];
#pragma unroll
    for (int s = 0; s < NS; s++) {
        a11[s] = a12[s] = a22[s] = c1[s] = c2[s] = 0;
        ipair[s] = 0; d00x[s] = d00y[s] = d01x[s] = d01y[s] = 0;
        const bool active = s < nstrips && lane < SC && s * SC + lane < winW;
        mtop[s] = active ? wtop : 0u; mbot[s] = active ? wbot : 0u;
        m00[s] = active ? iw00 : 0; m01[s] = active ? iw01 : 0; m10[s] = active ? iw10 : 0; m11[s] = active ? iw11 : 0;
        if (s < nstrips) {
            const uint8_t *ip = ip0 + s * SC + lane;
            const uint32_t *dp = dp0 + s * SC + lane;
            ipair[s] = (uint32_t)ip[0] | ((uint32_t)ip[1] << 8);
            const uint32_t dc = dp[0], dcr = dp[1];
            d00x[s] = (int)(short)(dc & 0xffffu); d00y[s] = (int)dc >> 16;
            d01x[s] = (int)(short)(dcr & 0xffffu); d01y[s] = (int)dcr >> 16;
        }
    }
#pragma unroll 4
    for (int r = 0; r < winH; r++) {
#pragma unroll
        for (int s = 0; s < NS; s++) {
            if (s < nstrips) {
                const int col = s * SC + lane;
                const uint8_t *ip = ip0 + (r + 1) * IP + col;
                const uint32_t *dp = dp0 + (r + 1) * DP + col;
                const uint32_t cpair = (uint32_t)ip[0] | ((uint32_t)ip[1] << 8);
                const uint32_t dc = dp[0], dcr = dp[1];
                const int d10x = (int)(short)(dc & 0xffffu), d10y = (int)dc >> 16;
                const int d11x = (int)(short)(dcr & 0xffffu), d11y = (int)dcr >> 16;
                uint32_t v = dp2a_lo(mtop[s], ipair[s], 256u);
                v = dp2a_lo(mbot[s], cpair, v);                        // v = taps + 256; Iw = v >> 9
                const int Iw = (int)(v >> 9);
                const int Ix = (d00x[s] * m00[s] + d01x[s] * m01[s] + d10x * m10[s] + d11x * m11[s] + 8192) >> 14;
                const int Iy = (d00y[s] * m00[s] + d01y[s] * m01[s] + d10y * m10[s] + d11y * m11[s] + 8192) >> 14;
                // (compile-time window sizes fold these guards away where every lane owns a template column)
                if ((SC >= 32 || lane < SC) && (NS * SC <= TC || col < TC))
                    tmpl_store(tmpl, r, TC, col, Ix, Iy);
                a11[s] += Ix * Ix; a12[s] += Ix * Iy; a22[s] += Iy * Iy;
                c1[s] += Iw * Ix; c2[s] += Iw * Iy;
                ipair[s] = cpair; d00x[s] = d10x; d00y[s] = d10y; d01x[s] = d11x; d01y[s] = d11y;
            }
        }
        __syncwarp();            // the template overlays the Scharr patch rows already consumed (see launch_lk)
    }
    for (int i = winH * TC + lane; i < TR * TC; i += 32) tmpl[i] = 0u;       // template rows below the window
    sA11 = sA12 = sA22 = sC1 = sC2 = 0;
#pragma unroll
    for (int s = 0; s < NS; s++) {
        if (s < nstrips) {
            sA11 += warp_sum_wide(a11[s]); sA12 += warp_sum_wide(a12[s]); sA22 += warp_sum_wide(a22[s]);
            sC1 += warp_sum_wide(c1[s]); sC2 += warp_sum_wide(c2[s]);
        }
    }
    __syncwarp();
}

// ---- Newton pass ---------------------------------------------------------------------------------------------
// Lane = (row group, column quad): rows [rowbase, rowbase + RG), template columns [4*cq, 4*cq + 4).
// S1 = sum Jw * Ix, S2 = sum Jw * Iy over the window, Jw = DESCALE(bilinear J at byte offset (ox, oy) inside the patch, 9).
// The products run on dp2a too: the four samples j0..j3 (0 <= j <= 255 * 32 = 8160) are split into bytes, jb01 = (lo0, lo1,
// hi0, hi1), jb23 likewise, and dp2a.lo / dp2a.hi against the template pairs give sum lo * Ix and sum hi * Ix separately;
// S1 = sum(lo * Ix) + 256 * sum(hi * Ix), the same integer as sum j * Ix.
// Headroom: |Ix|, |Iy| <= 16 * 255 = 4080 (Scharr of u8, bilinear weights summing to 2^14), lo <= 255, hi <= 31.  A lane
// flushes every 16 rows of its 4 columns, at most 64 pixels whatever the window, so a lo sum is within 64 * 4080 * 255 =
// 66 585 600 and the 32-lane total within 2 130 739 200 < 2^31: one plain REDUX per sum.
template <int WW, int WH>
__device__ __forceinline__ void newton_sums(const LKArgs &a, const uint8_t *__restrict__ patch, int ox, int oy, uint32_t wtop,
                                            uint32_t wbot, const uint32_t *__restrict__ tmpl, int rowbase, int cq, bool lane_on,
                                            long long &S1, long long &S2)
{
    const int RG = (WW && WH) ? lk_rg(WW, WH) : a.rg;
    const int JP = WW ? lk_jpitch(WW) : a.jpitch, TC = WW ? lk_tcols(WW) : a.tcols;
    const uint32_t al = (uint32_t)ox & 3u;                       // the same for every lane: 4*cq keeps the alignment
    const uint32_t sel0 = 0x3210u + 0x1111u * al, sel1 = sel0 + 0x1111u;
    const uint32_t *jp = reinterpret_cast<const uint32_t *>(patch + (oy + rowbase) * JP + ((ox + 4 * cq) & ~3));
    const uint4 *tp = reinterpret_cast<const uint4 *>(tmpl + rowbase * TC + 4 * cq);
    uint32_t p0, p1;                                             // byte windows (b0..b3), (b1..b4) of the previous row
    {
        const uint32_t w0 = jp[0], w1 = jp[1];
        p0 = __byte_perm(w0, w1, sel0); p1 = __byte_perm(w0, w1, sel1);
    }
    S1 = 0; S2 = 0;
    for (int r0 = 0; r0 < RG; r0 += 16) {
        const int r1 = (WW && WH) ? ((RG < r0 + 16) ? RG : r0 + 16) : min(RG, r0 + 16);
        uint32_t b1lo = 0, b1hi = 0, b2lo = 0, b2hi = 0;
#pragma unroll((WW && WH) ? 16 : 2)
        for (int r = r0; r < r1; r++) {
            jp += JP >> 2;
            const uint32_t w0 = jp[0], w1 = jp[1];
            const uint32_t c0 = __byte_perm(w0, w1, sel0), c1 = __byte_perm(w0, w1, sel1);
            const uint4 t = tp[r * (TC >> 2)];
            const uint32_t j0 = dp2a_lo(wbot, c0, dp2a_lo(wtop, p0, 256u)) >> 9;
            const uint32_t j1 = dp2a_lo(wbot, c1, dp2a_lo(wtop, p1, 256u)) >> 9;
            const uint32_t j2 = dp2a_hi(wbot, c0, dp2a_hi(wtop, p0, 256u)) >> 9;
            const uint32_t j3 = dp2a_hi(wbot, c1, dp2a_hi(wtop, p1, 256u)) >> 9;
            const uint32_t jb01 = __byte_perm(j0, j1, 0x5140u), jb23 = __byte_perm(j2, j3, 0x5140u);
            b1lo = dp2a_lo(t.y, jb23, dp2a_lo(t.x, jb01, b1lo));
            b1hi = dp2a_hi(t.y, jb23, dp2a_hi(t.x, jb01, b1hi));
            b2lo = dp2a_lo(t.w, jb23, dp2a_lo(t.z, jb01, b2lo));
            b2hi = dp2a_hi(t.w, jb23, dp2a_hi(t.z, jb01, b2hi));
            p0 = c0; p1 = c1;
        }
        if (!lane_on) { b1lo = b1hi = b2lo = b2hi = 0; }        // lanes beyond the last row group
        S1 += (long long)__reduce_add_sync(0xffffffffu, (int)b1lo) + ((long long)__reduce_add_sync(0xffffffffu, (int)b1hi) << 8);
        S2 += (long long)__reduce_add_sync(0xffffffffu, (int)b2lo) + ((long long)__reduce_add_sync(0xffffffffu, (int)b2hi) << 8);
    }
}

// OpenCV's residual (A.5 step 9): sum |Jw - Iw| over the window, Iw recomputed from the still staged I patch.
// Same lane mapping as newton_sums; pixels outside the window are masked explicitly.  Runs once per point at most.
template <int WW, int WH>
__device__ __noinline__ long long window_err(const LKArgs &a, const uint8_t *jpatch, int ox, int oy, uint32_t wtop, uint32_t wbot,
                                             const uint8_t *ipatch, int iox, uint32_t iwtop, uint32_t iwbot, int rowbase, int cq,
                                             bool lane_on)
{
    const int winW = WW ? WW : a.winW, winH = WH ? WH : a.winH;
    const int RG = (WW && WH) ? lk_rg(WW, WH) : a.rg;
    const int JP = WW ? lk_jpitch(WW) : a.jpitch, IP = WW ? lk_ipitch(WW) : a.ipitch;
    const uint32_t jsel0 = 0x3210u + 0x1111u * ((uint32_t)ox & 3u), jsel1 = jsel0 + 0x1111u;
    const uint32_t isel0 = 0x3210u + 0x1111u * ((uint32_t)iox & 3u), isel1 = isel0 + 0x1111u;
    const uint32_t *jp = reinterpret_cast<const uint32_t *>(jpatch + (oy + rowbase) * JP + ((ox + 4 * cq) & ~3));
    const uint32_t *ip = reinterpret_cast<const uint32_t *>(ipatch + rowbase * IP + ((iox + 4 * cq) & ~3));
    uint32_t jp0 = __byte_perm(jp[0], jp[1], jsel0), jp1 = __byte_perm(jp[0], jp[1], jsel1);
    uint32_t ip0 = __byte_perm(ip[0], ip[1], isel0), ip1 = __byte_perm(ip[0], ip[1], isel1);
    long long S = 0;
    for (int r0 = 0; r0 < RG; r0 += 16) {
        int s = 0;
        for (int r = r0; r < min(RG, r0 + 16); r++) {
            jp += JP >> 2; ip += IP >> 2;
            const uint32_t jc0 = __byte_perm(jp[0], jp[1], jsel0), jc1 = __byte_perm(jp[0], jp[1], jsel1);
            const uint32_t ic0 = __byte_perm(ip[0], ip[1], isel0), ic1 = __byte_perm(ip[0], ip[1], isel1);
            if (rowbase + r < winH) {
                const int d0 = (int)(dp2a_lo(wbot, jc0, dp2a_lo(wtop, jp0, 256u)) >> 9) - (int)(dp2a_lo(iwbot, ic0, dp2a_lo(iwtop, ip0, 256u)) >> 9);
                const int d1 = (int)(dp2a_lo(wbot, jc1, dp2a_lo(wtop, jp1, 256u)) >> 9) - (int)(dp2a_lo(iwbot, ic1, dp2a_lo(iwtop, ip1, 256u)) >> 9);
                const int d2 = (int)(dp2a_hi(wbot, jc0, dp2a_hi(wtop, jp0, 256u)) >> 9) - (int)(dp2a_hi(iwbot, ic0, dp2a_hi(iwtop, ip0, 256u)) >> 9);
                const int d3 = (int)(dp2a_hi(wbot, jc1, dp2a_hi(wtop, jp1, 256u)) >> 9) - (int)(dp2a_hi(iwbot, ic1, dp2a_hi(iwtop, ip1, 256u)) >> 9);
                const int c = 4 * cq;
                if (c < winW) s += abs(d0);
                if (c + 1 < winW) s += abs(d1);
                if (c + 2 < winW) s += abs(d2);
                if (c + 3 < winW) s += abs(d3);
            }
            jp0 = jc0; jp1 = jc1; ip0 = ic0; ip1 = ic1;
        }
        if (!lane_on) s = 0;
        S += warp_sum_wide(s);
    }
    return S;
}

// Channel c's copy of p, `stride` bytes per channel after channel 0's.  Channel c owns the slab bytes [c, c + 1) * warp_smem,
// and its pyramid levels lie in PI[c], PJ[c].
template <typename T>
__device__ __forceinline__ T *lk_chan(T *p, int c, int stride)
{
    using B = std::conditional_t<std::is_const<T>::value, const unsigned char, unsigned char>;
    return reinterpret_cast<T *>(reinterpret_cast<B *>(p) + (size_t)c * stride);
}

// One pyramidal pass for one point over cn channel planes (PI[c], PJ[c]: the pyramids of channel c); every window sum runs
// over the pixels and the channels.  CN is the channel count, or 0 for a runtime cn: CN = 1 folds the channel loops away.
// On entry (ox, oy) holds the initial flow if use_init.  On exit (ox, oy) = nextPts[k], status/err as cv2 (err = 0 where
// status == 0).
template <int WW, int WH, int CN>
__device__ __forceinline__ void lk_point(const LKPyr *PI, const LKPyr *PJ, int cn_rt, const LKArgs &a, float ptx, float pty,
                                         bool use_init, bool want_status, bool want_err, float &ox, float &oy, int &status,
                                         float &err, int &iters, unsigned char *slab, int rowbase, int cq, bool lane_on,
                                         int lane, const CUtensorMap *mapI, const CUtensorMap *mapJ, const CUtensorMap *mapD,
                                         uint64_t *bars, unsigned &phases)
{
    const float FLT_SCALE = 1.f / (1 << 20);
    const int cn = CN ? CN : cn_rt;
    const int winW = WW ? WW : a.winW, winH = WH ? WH : a.winH;
    const int IPITCH = WW ? lk_ipitch(WW) : a.ipitch, JPITCH = WW ? lk_jpitch(WW) : a.jpitch;
    const int DPITCH = WW ? lk_dpitch(WW) : a.dpitch;
    const int JROWS = winH + 1 + 2 * LK_MARGIN;
    const float halfx = (winW - 1) * 0.5f, halfy = (winH - 1) * 0.5f;
    uint32_t *tmpl = reinterpret_cast<uint32_t *>(slab);
    uint32_t *dpatch = reinterpret_cast<uint32_t *>(slab);
    uint8_t *ipatch = slab + a.off_ipatch;
    uint8_t *jpatch = slab + a.off_jpatch;
    auto ch = [&](auto *p, int c) { return lk_chan(p, c, a.warp_smem); };                      // of a slab buffer
    auto chl = [](const LKLevel &l, int c) -> const LKLevel & { return *lk_chan(&l, c, (int)sizeof(LKPyr)); };  // of a level
    status = 1; err = 0.f;
    const int L = PI[0].nlevels;
    for (int level = L - 1; level >= 0; --level) {
        // channel 0 decides geometry and staging: every channel has the same sizes, and multi-channel pyramids have no tensor maps
        const LKLevel &LI = PI[0].lv[level];
        const LKLevel &LJ = PJ[0].lv[level];
        const int rows = LI.rows, cols = LI.cols;
        const float sc = __int_as_float((127 - level) << 23);       // 2^-level
        float ppx = __fmul_rn(ptx, sc), ppy = __fmul_rn(pty, sc);
        float nx, ny;
        if (level == L - 1) {
            if (use_init) { nx = __fmul_rn(ox, sc); ny = __fmul_rn(oy, sc); }
            else { nx = ppx; ny = ppy; }
        } else { nx = __fmul_rn(ox, 2.f); ny = __fmul_rn(oy, 2.f); }
        ox = nx; oy = ny;

        ppx = __fsub_rn(ppx, halfx); ppy = __fsub_rn(ppy, halfy);
        const int ipx = cv_floor(no_nan(ppx)), ipy = cv_floor(no_nan(ppy));
        if (window_oob(ipx, ipy, winW, winH, rows, cols)) {
            if (level == 0) { status = 0; err = 0.f; }
            continue;
        }
        nx = no_nan(__fsub_rn(nx, halfx)); ny = no_nan(__fsub_rn(ny, halfy));      // (ox, oy) keep a NaN guess

        // ---- one burst of async copies: I window + its Scharr planes (barrier / group 0), J search patch (1) -------------
        // TMA where the level has tensor maps and the patch needs no reflection (bulk tensor copies zero-fill outside the
        // image: right for the Scharr planes, wrong for intensities); else 4-byte cp.async; else the REFLECT_101 gather.
        const bool i_in = ipx >= 0 && ipy >= 0 && ipx + winW < cols && ipy + winH < rows;
        const bool i_fix = !i_in && patch_reflectable(ipx, ipx + winW, ipy, winH + 1, rows, cols);
        const bool i_tma = LI.tma_img && (i_in || i_fix), d_tma = LI.tma_der != 0;
        const int ipxa = i_tma ? (ipx & ~15) : (ipx & ~3);     // bulk tensor copies start on 16-byte boundaries
        const int doff = d_tma ? (ipx & 3) : 0;
        int px0 = 0, py0 = 0, vx0 = 0;                        // staged origin (aligned) and logical patch origin
        bool staged = false, j_tma = false, j_fix = false;
        const int jnx = cv_floor(nx), jny = cv_floor(ny);
        const bool j_ok = !window_oob(jnx, jny, winW, winH, rows, cols);
        if (j_ok) {
            const int bx = jnx - LK_MARGIN, by = jny - LK_MARGIN;
            // the logical patch (window + margin) must lie inside the image (or be mirrorable inside shared memory);
            // the box may stick out further (zero fill, never read)
            const bool j_in = bx >= 0 && by >= 0 && bx + winW + 2 * LK_MARGIN < cols && by + JROWS <= rows;
            j_fix = !j_in && patch_reflectable(bx, bx + winW + 2 * LK_MARGIN, by, JROWS, rows, cols);
            j_tma = LJ.tma_img && (j_in || j_fix);
            px0 = j_tma ? (bx & ~15) : (bx & ~3); py0 = by; vx0 = bx;
            staged = true;
        }
        if (lane == 0 && (i_tma || d_tma || j_tma)) {
            fence_proxy_async();                              // this warp's earlier generic-proxy slab accesses come first
            if (i_tma || d_tma) {
                mbar_expect_tx(&bars[0], (i_tma ? (unsigned)(IPITCH * (winH + 1)) : 0u) + (d_tma ? (unsigned)(DPITCH * 4 * (winH + 1)) : 0u));
                if (i_tma) tma_load_2d(ipatch, &mapI[level], ipxa, ipy, &bars[0]);
                if (d_tma) tma_load_2d(dpatch, &mapD[level], ipx - doff, ipy, &bars[0]);
            }
            if (j_tma) {
                mbar_expect_tx(&bars[1], (unsigned)(JPITCH * JROWS));
                tma_load_2d(jpatch, &mapJ[level], px0, py0, &bars[1]);
            }
        }
        for (int c = 0; c < cn; c++) {
            if (!i_tma) stage_bytes(chl(LI, c), ipxa, ipy, winH + 1, IPITCH, lane, ch(ipatch, c));
            if (!d_tma) stage_deriv<WW, WH>(chl(LI, c), a, ipx, ipy, ch(dpatch, c), lane);
        }
        cp_async_commit();
        if (j_ok && !j_tma)
            for (int c = 0; c < cn; c++) stage_bytes(chl(LJ, c), px0, py0, JROWS, JPITCH, lane, ch(jpatch, c));
        cp_async_commit();
        cp_async_wait<1>();
        if (i_tma || d_tma) { mbar_wait(&bars[0], phases & 1u); phases ^= 1u; }
        __syncwarp();
        if (i_tma && i_fix) patch_reflect(ipatch, IPITCH, ipxa, ipx, ipx + winW, ipy, winH + 1, rows, cols, lane);

        uint32_t wtop, wbot;
        int iw00, iw01, iw10, iw11;
        bilinear_weights(__fsub_rn(ppx, (float)ipx), __fsub_rn(ppy, (float)ipy), wtop, wbot, iw00, iw01, iw10, iw11);
        const uint32_t iwtop = wtop, iwbot = wbot;            // the residual stage at level 0 samples I again

        // ---- template window: (Ix, Iy) per pixel; structure tensor; C1 = sum Iw*Ix, C2 = sum Iw*Iy -------------------------
        long long sA11, sA12, sA22, sC1, sC2;
        // channel 0 sets the sums and the other channels add theirs (a loop from channel 0 costs the 35 x 35 kernel spills)
        build_template<WW, WH>(a, ipatch + (ipx - ipxa), dpatch + doff, tmpl, wtop, wbot, iw00, iw01, iw10, iw11, lane,
                               sA11, sA12, sA22, sC1, sC2);
        for (int c = 1; c < cn; c++) {
            long long t11, t12, t22, tc1, tc2;
            build_template<WW, WH>(a, ch(ipatch, c) + (ipx - ipxa), ch(dpatch, c) + doff, ch(tmpl, c), wtop, wbot, iw00, iw01, iw10, iw11, lane,
                                   t11, t12, t22, tc1, tc2);
            sA11 += t11; sA12 += t12; sA22 += t22; sC1 += tc1; sC2 += tc2;
        }
        cp_async_wait<0>();
        if (j_tma) { mbar_wait(&bars[1], (phases >> 1) & 1u); phases ^= 2u; }
        __syncwarp();
        if (j_tma && j_fix) patch_reflect(jpatch, JPITCH, px0, vx0, vx0 + winW + 2 * LK_MARGIN, py0, JROWS, rows, cols, lane);
        const float A11 = __fmul_rn(__ll2float_rn(sA11), FLT_SCALE);
        const float A12 = __fmul_rn(__ll2float_rn(sA12), FLT_SCALE);
        const float A22 = __fmul_rn(__ll2float_rn(sA22), FLT_SCALE);
        float D = __fsub_rn(__fmul_rn(A11, A22), __fmul_rn(A12, A12));
        const float dA = __fsub_rn(A11, A22);
        const float disc = __fadd_rn(__fmul_rn(dA, dA), __fmul_rn(__fmul_rn(4.f, A12), A12));
        const float minEig = __fdiv_rn(__fsub_rn(__fadd_rn(A22, A11), __fsqrt_rn(disc)), (float)(2 * winW * winH));
        if (a.flags & IBT_LK_GET_MIN_EIGENVALS) err = minEig;
        if (minEig < a.minEigThr || D < 1.1920929e-07f) {
            if (level == 0) status = 0;
            continue;
        }
        D = __fdiv_rn(1.f, D);
        float pdx = 0.f, pdy = 0.f;
        for (int j = 0; j < a.maxCount; j++) {
            const int inx = cv_floor(nx), iny = cv_floor(ny);
            if (window_oob(inx, iny, winW, winH, rows, cols)) {
                if (level == 0) status = 0;
                break;
            }
            if (!staged || (unsigned)(inx - vx0) > 2u * LK_MARGIN || (unsigned)(iny - py0) > 2u * LK_MARGIN) {
                vx0 = inx - LK_MARGIN; px0 = vx0 & ~3; py0 = iny - LK_MARGIN;
                for (int c = 0; c < cn; c++) restage_sync(chl(LJ, c), px0, py0, JROWS, JPITCH, ch(jpatch, c), lane);
                staged = true;
            }
            bilinear_weights(__fsub_rn(nx, (float)inx), __fsub_rn(ny, (float)iny), wtop, wbot, iw00, iw01, iw10, iw11);
            long long sb1 = 0, sb2 = 0;
            for (int c = 0; c < cn; c++) {
                long long t1, t2;
                newton_sums<WW, WH>(a, ch(jpatch, c), inx - px0, iny - py0, wtop, wbot, ch(tmpl, c), rowbase, cq, lane_on, t1, t2);
                sb1 += t1; sb2 += t2;
            }
            ++iters;
            const float b1 = __fmul_rn(__ll2float_rn(sb1 - sC1), FLT_SCALE);
            const float b2 = __fmul_rn(__ll2float_rn(sb2 - sC2), FLT_SCALE);
            const float dx = __fmul_rn(__fsub_rn(__fmul_rn(A12, b2), __fmul_rn(A22, b1)), D);
            const float dy = __fmul_rn(__fsub_rn(__fmul_rn(A12, b1), __fmul_rn(A11, b2)), D);
            nx = __fadd_rn(nx, dx); ny = __fadd_rn(ny, dy);
            ox = __fadd_rn(nx, halfx); oy = __fadd_rn(ny, halfy);
            if (__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)) <= a.eps2) break;
            if (j > 0 && fabsf(__fadd_rn(dx, pdx)) < 0.01f && fabsf(__fadd_rn(dy, pdy)) < 0.01f) {
                ox = __fsub_rn(ox, __fmul_rn(dx, 0.5f)); oy = __fsub_rn(oy, __fmul_rn(dy, 0.5f));
                break;
            }
            pdx = dx; pdy = dy;
        }
        // OpenCV's final stage at level 0 (A.5 step 9): bounds test of the final window (-> status) and the residual err.
        // The reference never reads status or err (s1:323-333): callers that pass no status / err buffers skip the stage.
        if (status && level == 0 && !(a.flags & IBT_LK_GET_MIN_EIGENVALS) && (want_status || want_err)) {
            const float qx = __fsub_rn(ox, halfx), qy = __fsub_rn(oy, halfy);
            const int iqx = cv_floor(no_nan(qx)), iqy = cv_floor(no_nan(qy));
            if (window_oob(iqx, iqy, winW, winH, rows, cols)) { status = 0; err = 0.f; continue; }
            if (!want_err) continue;
            if (!staged || (unsigned)(iqx - vx0) > 2u * LK_MARGIN || (unsigned)(iqy - py0) > 2u * LK_MARGIN) {
                vx0 = iqx - LK_MARGIN; px0 = vx0 & ~3; py0 = iqy - LK_MARGIN;
                for (int c = 0; c < cn; c++) restage_sync(chl(LJ, c), px0, py0, JROWS, JPITCH, ch(jpatch, c), lane);
            }
            bilinear_weights(__fsub_rn(qx, (float)iqx), __fsub_rn(qy, (float)iqy), wtop, wbot, iw00, iw01, iw10, iw11);
            long long s = 0;
            for (int c = 0; c < cn; c++)
                s += window_err<WW, WH>(a, ch(jpatch, c), iqx - px0, iqy - py0, wtop, wbot, ch(ipatch, c), ipx - ipxa, iwtop, iwbot,
                                        rowbase, cq, lane_on);
            err = __fdiv_rn(__ll2float_rn(s), (float)(32 * winW * cn * winH));
        }
        __syncwarp();
    }
    cp_async_wait<0>();
    if (!status && !(a.flags & IBT_LK_GET_MIN_EIGENVALS)) err = 0.f;
}

// The kernel's second parameter: gray frames (CN = 1) bring the tensor maps of a.pyr, multi-channel frames (CN = 0, any cn)
// their channel pyramids (a.pyr unused).
template <int CN> using LKFrames = std::conditional_t<CN == 1, LKMaps, LKMcPyr>;

// Gray frames: 3 CTAs of 8 warps per SM (80 registers).  Multi-channel frames: no minimum (0), which keeps the runtime-cn
// solver out of local memory (128 registers: 16 warps per SM).
template <int WW, int WH, int CN>
__global__ void __launch_bounds__(256, CN == 1 ? 3 : 0)
lk_kernel(const __grid_constant__ LKArgs a, const __grid_constant__ LKFrames<CN> fr)
{
    extern __shared__ __align__(128) unsigned char lk_smem[];
    __shared__ __align__(8) uint64_t lk_bars[8][2];        // per warp: [0] I window + Scharr planes, [1] J patch
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    if (lane == 0) {
        mbar_init(&lk_bars[wib][0], 1); mbar_init(&lk_bars[wib][1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    unsigned phases = 0u;                                  // bit b = parity to wait for on lk_bars[wib][b]
    int cn = 1;
    if constexpr (CN != 1) cn = fr.cn;
    unsigned char *slab = lk_smem + (size_t)wib * a.warp_smem * cn;     // cn channel slabs per warp
    // Newton mapping of this lane: row group and column quad (lanes beyond the last group idle on group 0's rows)
    const int NL = WW ? lk_nl(WW) : a.nl, NG = (WW && WH) ? lk_ng(WW, WH) : a.ng, RG = (WW && WH) ? lk_rg(WW, WH) : a.rg;
    const int grp = lane / NL;
    const bool lane_on = grp < NG;
    const int rowbase = lane_on ? grp * RG : 0, cq = lane_on ? lane - grp * NL : 0;

  for (;;) {                                            // persistent warp: points are handed out dynamically
    int k = 0;
    if (lane == 0) k = (int)atomicAdd(a.work_counter, 1u);
    k = __shfl_sync(0xffffffffu, k, 0);
    if (k >= a.n) break;
    if (a.alive && !a.alive[k]) continue;
    const float p0x = a.p0[2 * k], p0y = a.p0[2 * k + 1];
    float ptx = p0x, pty = p0y;
    int it_f = 0, it_b = 0;
    const int npass = a.fb ? 2 : 1;
    for (int pass = 0; pass < npass; ++pass) {          // one copy of the solver body: pass 1 swaps the pyramids
        float ox = 0.f, oy = 0.f, err;
        int status, iters = 0;
        const bool use_init = pass == 0 && (a.flags & IBT_LK_USE_INITIAL_FLOW) != 0;
        if (use_init) { ox = a.p1[2 * k]; oy = a.p1[2 * k + 1]; }
        const bool want_status = pass == 0 ? a.st1 != nullptr : a.st0 != nullptr;
        const bool want_err = pass == 0 ? a.err1 != nullptr : a.err0 != nullptr;
        const LKPyr *PI = a.pyr + pass, *PJ = a.pyr + (pass ^ 1);
        const CUtensorMap *mapI = nullptr, *mapJ = nullptr, *mapD = nullptr;
        if constexpr (CN == 1) { mapI = fr.imgI[pass]; mapJ = fr.imgJ[pass ^ 1]; mapD = fr.der[pass]; }
        else { PI = pass ? fr.J : fr.I; PJ = pass ? fr.I : fr.J; }
        lk_point<WW, WH, CN>(PI, PJ, cn, a, ptx, pty, use_init, want_status, want_err, ox, oy, status, err, iters,
                             slab, rowbase, cq, lane_on, lane, mapI, mapJ, mapD, lk_bars[wib], phases);
        if (pass == 0) it_f = iters; else it_b = iters;
        if (lane == 0) {
            if (pass == 0) {
                a.p1[2 * k] = ox; a.p1[2 * k + 1] = oy;
                if (a.st1) a.st1[k] = (uint8_t)status;
                if (a.err1) a.err1[k] = err;
            } else {
                if (a.p0r) { a.p0r[2 * k] = ox; a.p0r[2 * k + 1] = oy; }
                if (a.st0) a.st0[k] = (uint8_t)status;
                if (a.err0) a.err0[k] = err;
                const float d = glibc_hypotf(fabsf(__fsub_rn(p0x, ox)), fabsf(__fsub_rn(p0y, oy)));
                if (a.fbdist) a.fbdist[k] = d;
                if (a.alive) a.alive[k] = (d < a.fb_thresh) ? 1 : 0;
            }
        }
        ptx = ox; pty = oy;                             // the backward pass starts from p1 (s1:326)
    }
    if (lane == 0) {
        if (a.iters) {
            if (a.fb) { a.iters[2 * k] = it_f; a.iters[2 * k + 1] = it_b; }
            else a.iters[k] = it_f;
        }
        if (a.iter_total) atomicAdd(a.iter_total, (unsigned long long)(it_f + it_b));
    }
    __syncwarp();
  }
    // the last warp to leave re-arms the work queue for the next launch on this stream (no memset node per launch)
    if (lane == 0) {
        __threadfence();
        if (atomicAdd(a.work_counter + 1, 1u) == a.total_warps - 1u) {
            a.work_counter[0] = 0u; a.work_counter[1] = 0u;
            __threadfence();
        }
    }
}

static int fill_pyr(const ibt_pyramid_t *p, LKPyr &o, bool need_deriv)
{
    if (!p || p->nlevels < 1 || p->nlevels > IBT_MAX_LEVELS) return IBT_E_INVALID;
    o.nlevels = p->nlevels;
    for (int l = 0; l < p->nlevels; l++) {
        if (!p->img[l] || p->rows[l] <= 0 || p->cols[l] <= 0 || p->img_pitch[l] < p->cols[l] ||
            p->img_pitch[l] > 0x7fffffff)
            return IBT_E_INVALID;
        if (need_deriv && (!p->deriv[l] || p->deriv_pitch[l] % 4 != 0 || p->deriv_pitch[l] < (int64_t)p->cols[l] * 4 ||
                           reinterpret_cast<uintptr_t>(p->deriv[l]) % 4 != 0))
            return IBT_E_INVALID;
        o.lv[l].img = p->img[l];
        o.lv[l].deriv = reinterpret_cast<const uint32_t *>(p->deriv[l]);
        o.lv[l].img_pitch = (int)p->img_pitch[l];
        o.lv[l].deriv_pitch = (int)(p->deriv_pitch[l] / 4);
        o.lv[l].rows = p->rows[l];
        o.lv[l].cols = p->cols[l];
        o.lv[l].word_ok = (reinterpret_cast<uintptr_t>(p->img[l]) % 4 == 0) && (p->img_pitch[l] % 4 == 0);
        o.lv[l].tma_img = o.lv[l].tma_der = 0;
    }
    return IBT_OK;
}

// Per-device launcher state, shared by every host thread: guarded by one mutex.  A work queue (two words: next point,
// warps that have left) belongs to one (device, stream): launches on a stream are ordered, and the kernel re-arms its
// queue when its last warp leaves, so queues of different streams never alias however many launches are in flight.
struct LKQueue { int dev; cudaStream_t stream; unsigned int *words; };
static std::mutex lk_mu;
static int lk_max_ctas_per_sm = 0;          // ibt_lk_set_max_ctas_per_sm: 0 = fill the SM
static std::vector<LKQueue> lk_queues;
static bool lk_attr_set[64] = {false};

static int lk_queue_for(int dev, cudaStream_t st, unsigned int **out)
{
    for (const LKQueue &q : lk_queues)
        if (q.dev == dev && q.stream == st) { *out = q.words; return IBT_OK; }
    unsigned int *w = nullptr;
    IBT_CUDA_TRY(cudaMalloc(&w, 2 * sizeof(unsigned int)));
    // zeroed on the queue's own stream: a plain cudaMemset goes to the legacy default stream, which a non-blocking stream does
    // not wait for -- the zeroing could land in the middle of the first launches and leave the queue un-armed
    IBT_CUDA_TRY(cudaMemsetAsync(w, 0, 2 * sizeof(unsigned int), st));
    lk_queues.push_back({dev, st, w});
    *out = w;
    return IBT_OK;
}

// The one launcher of every LK entry point.  A and B are host arrays of cn pyramids, one per channel plane.  planes == false
// (ibt_lk, ibt_lk_fb; cn == 1): gray frames in a.pyr, with tensor maps, on the window-specialised kernels.  planes == true
// (ibt_lk_multichannel, ibt_lk_fb_multichannel): the channel pyramids travel as LKMcPyr to the runtime-cn kernel.
static int launch_lk(LKArgs &a, const ibt_pyramid_t *const *A, const ibt_pyramid_t *const *B, int cn, bool planes, int winW,
                     int winH, int max_count, double epsilon, double min_eig, cudaStream_t st)
{
    if (a.n < 0 || winW < 3 || winH < 3 || winW > IBT_MAX_WIN || winH > IBT_MAX_WIN || cn < 1 || cn > LK_MC_MAX || !A || !B)
        return IBT_E_INVALID;
    if (a.n == 0) return IBT_OK;
    if (!a.p0 || !a.p1) return IBT_E_INVALID;
    static thread_local LKMcPyr mc;
    LKPyr *PI = planes ? mc.I : &a.pyr[0], *PJ = planes ? mc.J : &a.pyr[1];
    mc.cn = cn;
    for (int c = 0; c < cn; c++) {
        int rc = fill_pyr(A[c], PI[c], true);
        if (rc) return rc;
        rc = fill_pyr(B[c], PJ[c], a.fb != 0);
        if (rc) return rc;
        if (A[c]->nlevels != A[0]->nlevels || B[c]->nlevels != A[0]->nlevels) return IBT_E_INVALID;
        for (int l = 0; l < A[0]->nlevels; l++)
            if (A[c]->rows[l] != A[0]->rows[l] || A[c]->cols[l] != A[0]->cols[l] || B[c]->rows[l] != A[0]->rows[l] ||
                B[c]->cols[l] != A[0]->cols[l])
                return IBT_E_INVALID;
    }
    a.winW = winW; a.winH = winH;
    a.nl = lk_nl(winW); a.ng = lk_ng(winW, winH); a.rg = lk_rg(winW, winH);
    a.trows = lk_trows(winW, winH); a.tcols = lk_tcols(winW);
    a.nstrips = lk_nstrips(winW);
    a.strip_cols = lk_strip_cols(winW);
    a.dpitch = lk_dpitch(winW);
    a.ipitch = lk_ipitch(winW);
    a.jpitch = lk_jpitch(winW);
    a.jrows = winH + 1 + 2 * LK_MARGIN;
    // The Scharr patch is consumed row by row while the template rows are produced, so the template OVERLAYS it: template
    // row r (4 * tcols bytes at 4 * tcols * r) is written only after patch row r+1 (at 4 * dpitch * (r+1)) has been read
    // into registers, and tcols <= dpitch keeps every later patch row intact.
    size_t off = (size_t)a.trows * a.tcols * 4;
    const size_t dbytes = (size_t)(winH + 1) * a.dpitch * 4;
    if (off < dbytes) off = dbytes;
    off = (off + 127) & ~(size_t)127;                     // TMA destinations are 128-byte aligned
    a.off_ipatch = (int)off; off += (size_t)(winH + 1) * a.ipitch; off = (off + 127) & ~(size_t)127;
    // Newton lanes of the last row group read (never use) J rows down to trows + 2 * MARGIN
    a.off_jpatch = (int)off; off += (size_t)(a.trows + 1 + 2 * LK_MARGIN) * a.jpitch;
    a.warp_smem = (int)((off + 127) & ~(size_t)127);      // one slab per channel
    // tensor maps (boxes: I window ipitch x (winH+1), J patch jpitch x jrows, Scharr window dpitch words x (winH+1))
    static thread_local LKMaps maps;
    static const bool no_tma = getenv("IBT_NO_TMA") != nullptr;
    for (int pi = 0; pi < 2 && !planes && !no_tma; pi++) {
        const ibt_pyramid_t *P = pi ? B[0] : A[0];
        for (int l = 0; l < P->nlevels; l++) {
            LKLevel &lv = a.pyr[pi].lv[l];
            lv.tma_img = make_map_2d(&maps.imgI[pi][l], CU_TENSOR_MAP_DATA_TYPE_UINT8, P->img[l], P->cols[l], P->rows[l],
                                     P->img_pitch[l], a.ipitch, winH + 1) &&
                         make_map_2d(&maps.imgJ[pi][l], CU_TENSOR_MAP_DATA_TYPE_UINT8, P->img[l], P->cols[l], P->rows[l],
                                     P->img_pitch[l], a.jpitch, a.jrows);
            lv.tma_der = P->deriv[l] != nullptr &&
                         make_map_2d(&maps.der[pi][l], CU_TENSOR_MAP_DATA_TYPE_UINT32, P->deriv[l], P->cols[l], P->rows[l],
                                     P->deriv_pitch[l], a.dpitch, winH + 1);
        }
    }
    a.maxCount = max_count < 0 ? 0 : (max_count > 100 ? 100 : max_count);
    if (epsilon < 0) epsilon = 0;
    if (epsilon > 10) epsilon = 10;
    a.eps2 = (float)(epsilon * epsilon);
    a.minEigThr = (float)min_eig;
    // warps per CTA: the choice that keeps the most warps resident in 227 KB of shared memory per SM, at most as many as the
    // registers allow (gray kernels: compiled for 3 CTAs of 8 warps per SM, 80 registers; runtime-cn kernel: 128 registers)
    const size_t per_warp = (size_t)a.warp_smem * cn;
    const int max_warps = planes ? 16 : 24;
    int wpc = 1, best = 0, best_ctas = 1;
    for (int w = 1; w <= 8; w++) {
        const size_t per_cta = per_warp * w + 1024;
        if (per_cta > 200 * 1024) break;
        int ctas = (int)((227 * 1024) / per_cta);
        if (ctas > 32) ctas = 32;
        if (ctas * w > max_warps) ctas = max_warps / w;
        const int warps = ctas * w;
        if (warps >= best) { best = warps; wpc = w; best_ctas = ctas; }
    }
    if (best == 0) return IBT_E_INVALID;
    {
        std::lock_guard<std::mutex> lock(lk_mu);
        if (lk_max_ctas_per_sm > 0 && best_ctas > lk_max_ctas_per_sm) best_ctas = lk_max_ctas_per_sm;
    }
    const size_t smem = per_warp * wpc;
    void (*kern)(const LKArgs, const LKMaps) = lk_kernel<0, 0, 1>;      // generic window; the sizes the configs use are specialised
    if (winW == 21 && winH == 21) kern = lk_kernel<21, 21, 1>;
    else if (winW == 31 && winH == 31) kern = lk_kernel<31, 31, 1>;
    else if (winW == 35 && winH == 35) kern = lk_kernel<35, 35, 1>;
    int dev_id = 0;
    IBT_CUDA_TRY(cudaGetDevice(&dev_id));
    if (dev_id < 0 || dev_id >= 64) return IBT_E_INVALID;
    {
        std::lock_guard<std::mutex> lock(lk_mu);
        if (!lk_attr_set[dev_id]) {
            const int lim = 200 * 1024;
            IBT_CUDA_TRY(cudaFuncSetAttribute(lk_kernel<0, 0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
            IBT_CUDA_TRY(cudaFuncSetAttribute(lk_kernel<21, 21, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
            IBT_CUDA_TRY(cudaFuncSetAttribute(lk_kernel<31, 31, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
            IBT_CUDA_TRY(cudaFuncSetAttribute(lk_kernel<35, 35, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
            IBT_CUDA_TRY(cudaFuncSetAttribute(lk_kernel<0, 0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
            lk_attr_set[dev_id] = true;
        }
        const int rc = lk_queue_for(dev_id, st, &a.work_counter);
        if (rc) return rc;
    }
    int blocks = kNumSMs * best_ctas;                   // persistent: one wave, warps pull points until none are left
    const int need = (a.n + wpc - 1) / wpc;
    if (blocks > need) blocks = need;
    a.total_warps = (unsigned)(blocks * wpc);
    // the tensor maps or the channel pyramids travel as a __grid_constant__ parameter
    if (planes) lk_kernel<0, 0, 0><<<blocks, wpc * 32, smem, st>>>(a, mc);
    else kern<<<blocks, wpc * 32, smem, st>>>(a, maps);
    return check_launch(planes ? "ibt_lk_multichannel" : "ibt_lk");
}

} // namespace ibt

IBT_API int ibt_lk_set_max_ctas_per_sm(int ctas)
{
    if (ctas < 0) return IBT_E_INVALID;
    std::lock_guard<std::mutex> lock(ibt::lk_mu);
    ibt::lk_max_ctas_per_sm = ctas;
    return IBT_OK;
}

IBT_API int ibt_lk(const ibt_pyramid_t *pyrI, const ibt_pyramid_t *pyrJ, const float *pts, float *next_pts, int N,
                   int winW, int winH, int max_count, double epsilon, double min_eig_threshold, int flags,
                   uint8_t *status, float *err, int32_t *iters, void *stream)
{
    ibt::LKArgs a;
    memset(&a, 0, sizeof(a));
    a.p0 = pts; a.n = N; a.flags = flags; a.fb = 0;
    a.p1 = next_pts; a.st1 = status; a.err1 = err; a.iters = iters;
    return ibt::launch_lk(a, &pyrI, &pyrJ, 1, false, winW, winH, max_count, epsilon, min_eig_threshold,
                          static_cast<cudaStream_t>(stream));
}

IBT_API int ibt_lk_fb(const ibt_pyramid_t *prev, const ibt_pyramid_t *next, const float *p0, int N, int winW, int winH,
                      int max_count, double epsilon, double min_eig_threshold, float fb_threshold, float *p1,
                      uint8_t *st1, float *err1, float *p0r, uint8_t *st0, float *err0, float *fbdist, uint8_t *alive,
                      int32_t *iters, unsigned long long *iter_total, void *stream)
{
    ibt::LKArgs a;
    memset(&a, 0, sizeof(a));
    a.p0 = p0; a.n = N; a.flags = 0; a.fb = 1; a.fb_thresh = fb_threshold;
    a.p1 = p1; a.st1 = st1; a.err1 = err1; a.p0r = p0r; a.st0 = st0; a.err0 = err0;
    a.fbdist = fbdist; a.alive = alive; a.iters = iters; a.iter_total = iter_total;
    return ibt::launch_lk(a, &prev, &next, 1, false, winW, winH, max_count, epsilon, min_eig_threshold,
                          static_cast<cudaStream_t>(stream));
}

IBT_API int ibt_lk_multichannel(const ibt_pyramid_t *const *pyrI, const ibt_pyramid_t *const *pyrJ, int cn, const float *pts,
                                float *next_pts, int N, int winW, int winH, int max_count, double epsilon,
                                double min_eig_threshold, int flags, uint8_t *status, float *err, int32_t *iters, void *stream)
{
    ibt::LKArgs a;
    memset(&a, 0, sizeof(a));
    a.p0 = pts; a.n = N; a.flags = flags; a.fb = 0;
    a.p1 = next_pts; a.st1 = status; a.err1 = err; a.iters = iters;
    return ibt::launch_lk(a, pyrI, pyrJ, cn, true, winW, winH, max_count, epsilon, min_eig_threshold,
                          static_cast<cudaStream_t>(stream));
}

IBT_API int ibt_lk_fb_multichannel(const ibt_pyramid_t *const *prev, const ibt_pyramid_t *const *next, int cn, const float *p0,
                                   int N, int winW, int winH, int max_count, double epsilon, double min_eig_threshold,
                                   float fb_threshold, float *p1, uint8_t *st1, float *err1, float *p0r, uint8_t *st0,
                                   float *err0, float *fbdist, uint8_t *alive, int32_t *iters, unsigned long long *iter_total,
                                   void *stream)
{
    if (cn < 2 || cn > ibt::LK_MC_MAX) return IBT_E_INVALID;
    ibt::LKArgs a;
    memset(&a, 0, sizeof(a));
    a.p0 = p0; a.n = N; a.flags = 0; a.fb = 1; a.fb_thresh = fb_threshold;
    a.p1 = p1; a.st1 = st1; a.err1 = err1; a.p0r = p0r; a.st0 = st0; a.err0 = err0;
    a.fbdist = fbdist; a.alive = alive; a.iters = iters; a.iter_total = iter_total;
    return ibt::launch_lk(a, prev, next, cn, true, winW, winH, max_count, epsilon, min_eig_threshold,
                          static_cast<cudaStream_t>(stream));
}
