// K2: Shi-Tomasi corner seeding (SURVEY.md A.6).  Replaces
// cv2.goodFeaturesToTrack(frame_gray, mask=mask, **feature_params), s1_lucaskanade_tracking.py:437
// (s0_1_test_lucaskanade_tracking.py:167).  Two launches, no host round trip in between:
//
//   K2a  eig_nms_kernel  one warp per (112-column strip, row chunk), 4 adjacent columns per lane, rows top to bottom:
//                        Sobel3 by dp4a on funnel-shifted byte windows -> (sx^2, sx*sy, sy^2) as exact int32 -> vertical
//                        sliding sum through a per-warp shared-memory ring (16-byte accesses) -> horizontal window sum
//                        by lane shuffles -> lambda_min (OpenCV's float formula) -> running masked maximum and 3x3
//                        non-maximum test on a three-row register ring.  The response map is never written: a pixel
//                        above the final threshold is a candidate iff it is a RAW 3x3 maximum (every neighbour above it
//                        would be above the threshold too), so raw maxima are appended as 64-bit keys
//                        (response bits << 32 | linear address) and thresholded afterwards; a running lower bound of
//                        the threshold (quality * maximum seen so far) drops most weak maxima on the spot.
//                        OpenCV rounds every product to float before its double box sum; the exact integer sums sit in
//                        the middle of that rounding noise (~1e-7 relative, the size of the wheel's own
//                        irreproducibility, SURVEY A.6).  REFLECT_101 acts on the product image, as in OpenCV's boxFilter.
//   K2b  gftt_select_kernel  ONE persistent launch (148 CTAs, software grid barrier) that runs the whole selection with
//                        device-side control flow: threshold + response histogram -> top-k prefilter (the strongest
//                        ~4*maxCorners candidates; all of them if culling leaves too few) -> stable LSD radix sort on the
//                        response bytes (ties by address) -> OpenCV's cell grid as CSR lists -> OpenCV's sequential greedy
//                        min-distance culling restated as a monotone fixed point over ranks (a candidate is REJECTED once
//                        a stronger candidate within minDistance in its 3x3 cell neighbourhood is ACCEPTED, ACCEPTED once
//                        all such candidates are REJECTED; rounds repeat until none is undecided) -> ordered compaction
//                        -> (x, y) float32 of the first maxCorners, count left in device memory.
//   ibt_min_eigen_f32    (cornerMinEigenVal test hook) keeps the map-writing eig_kernel.
//   cv2's other Sobel apertures (gradientSize / ksize = -1, 1, 5, 7) take eig_nms_ap_kernel / eig_ap_kernel in place of K2a /
//   eig_kernel (table and int64 bound at eig_ap_kernel); K2b is the same.
//   float32 images take eig_f32_kernel (every aperture; the fused K2a and the map hooks); K2b is the same.
#include "common.cuh"
#include <atomic>
#include <float.h>
#include <stddef.h>
#include <string.h>

namespace ibt {

// ---------------------------------------------------------------------------------------------
// K2a
constexpr int EW = 256;                 // threads per CTA = support columns per CTA row
constexpr int ERS = 64;                 // output rows per CTA
constexpr int MAX_BLOCK = 31;

__device__ __forceinline__ uint32_t enc_f32(float f)           // order-preserving float -> uint
{
    const uint32_t b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float dec_f32(uint32_t e)
{
    return __uint_as_float((e & 0x80000000u) ? (e & 0x7fffffffu) : ~e);
}

__global__ void __launch_bounds__(EW)
eig_kernel(const uint8_t *__restrict__ img, int H, int W, int64_t pitch, int bs, double s2, int harris, float harris_k,
           float *__restrict__ eig, int64_t eig_pitch_f,
           const uint8_t *__restrict__ mask, int64_t mask_pitch, uint32_t *__restrict__ maxbits)
{
    extern __shared__ int eig_smem[];
    int *prod = eig_smem;                      // [2][3][EW]   products of the current support row (double-buffered)
    int *ring = eig_smem + 2 * 3 * EW;         // [bs][3][EW]  horizontal window sums of the last bs support rows
    const int t = threadIdx.x;
    const int nout = EW - bs + 1;              // output columns per CTA
    const int a0 = -(bs / 2);
    const int X0 = blockIdx.x * nout, Y0 = blockIdx.y * ERS;
    const int x = X0 + t;                      // output column of this thread (t < nout)
    const bool xout = t < nout && x < W;
    // REFLECT_101 acts on the product image: support column -> image column
    const int px = r101(X0 + a0 + t, W);
    const int xm = r101(px - 1, W), xp = r101(px + 1, W);
    int vs0 = 0, vs1 = 0, vs2 = 0;
    uint32_t lmax = 0;
    const int nrows = min(ERS, H - Y0) + bs - 1;
    int slot = 0;
    // the 3x3 bytes of support row k+1 are fetched before the barrier of row k: the loads fly during the window sums
    int b00, b01, b02, b10, b12, b20, b21, b22;
    {
        const int py = r101(Y0 + a0, H);
        const uint8_t *r0 = img + (int64_t)r101(py - 1, H) * pitch, *r1 = img + (int64_t)py * pitch;
        const uint8_t *r2 = img + (int64_t)r101(py + 1, H) * pitch;
        b00 = r0[xm]; b01 = r0[px]; b02 = r0[xp]; b10 = r1[xm]; b12 = r1[xp]; b20 = r2[xm]; b21 = r2[px]; b22 = r2[xp];
    }
    for (int k = 0; k < nrows; k++) {
        const int sx = (b02 + 2 * b12 + b22) - (b00 + 2 * b10 + b20);
        const int sy = (b20 + 2 * b21 + b22) - (b00 + 2 * b01 + b02);
        int *pb = prod + (k & 1) * 3 * EW;
        pb[t] = sx * sx; pb[EW + t] = sx * sy; pb[2 * EW + t] = sy * sy;
        if (k + 1 < nrows) {
            const int py = r101(Y0 + a0 + k + 1, H);
            const uint8_t *r0 = img + (int64_t)r101(py - 1, H) * pitch, *r1 = img + (int64_t)py * pitch;
            const uint8_t *r2 = img + (int64_t)r101(py + 1, H) * pitch;
            b00 = r0[xm]; b01 = r0[px]; b02 = r0[xp]; b10 = r1[xm]; b12 = r1[xp]; b20 = r2[xm]; b21 = r2[px]; b22 = r2[xp];
        }
        __syncthreads();
        if (t < nout) {
            int h0 = 0, h1 = 0, h2 = 0;
            for (int j = 0; j < bs; j++) { h0 += pb[t + j]; h1 += pb[EW + t + j]; h2 += pb[2 * EW + t + j]; }
            int *rg = ring + slot * 3 * EW;
            if (k >= bs) { vs0 -= rg[t]; vs1 -= rg[EW + t]; vs2 -= rg[2 * EW + t]; }
            vs0 += h0; vs1 += h1; vs2 += h2;
            rg[t] = h0; rg[EW + t] = h1; rg[2 * EW + t] = h2;
            if (k >= bs - 1 && xout) {
                const int y = Y0 + k - (bs - 1);
                float e;
                if (harris) {                                   // cv2.cornerHarris: (a*c - b*b) - k*((a + c)*(a + c)), float, unfused
                    const float a = (float)((double)vs0 * s2), b = (float)((double)vs1 * s2), c = (float)((double)vs2 * s2);
                    const float tr = __fadd_rn(a, c);
                    e = __fsub_rn(__fsub_rn(__fmul_rn(a, c), __fmul_rn(b, b)), __fmul_rn(harris_k, __fmul_rn(tr, tr)));
                } else {
                    const float a = __fmul_rn((float)((double)vs0 * s2), 0.5f), b = (float)((double)vs1 * s2);
                    const float c = __fmul_rn((float)((double)vs2 * s2), 0.5f);
                    const float d = __fsub_rn(a, c);
                    e = __fsub_rn(__fadd_rn(a, c), __fsqrt_rn(__fadd_rn(__fmul_rn(d, d), __fmul_rn(b, b))));
                }
                eig[(int64_t)y * eig_pitch_f + x] = e;
                if (maxbits && (!mask || mask[(int64_t)y * mask_pitch + x])) lmax = max(lmax, enc_f32(e));
            }
        }
        slot = slot + 1 == bs ? 0 : slot + 1;
    }
    if (maxbits) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) lmax = max(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
        if ((t & 31) == 0 && lmax) atomicMax(maxbits, lmax);
    }
}

static size_t eig_smem_bytes(int bs) { return (size_t)(2 + bs) * 3 * EW * sizeof(int); }

static int launch_eig(const uint8_t *gray, int H, int W, int64_t pitch, int bs, int harris, double k, float *eig,
                      int64_t eig_pitch_bytes, const uint8_t *mask, int64_t mask_pitch, uint32_t *maxbits, cudaStream_t st)
{
    if (!gray || !eig || H <= 0 || W <= 0 || bs < 1 || bs > MAX_BLOCK || pitch < W || eig_pitch_bytes % 4 != 0 ||
        eig_pitch_bytes < (int64_t)W * 4)
        return IBT_E_INVALID;
    if (eig_smem_bytes(bs) > 48 * 1024)                 // large blockSize: opt in to > 48 KB dynamic shared memory (per device)
        IBT_CUDA_TRY(cudaFuncSetAttribute(eig_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)eig_smem_bytes(MAX_BLOCK)));
    const float scale = (float)(1.0 / (4.0 * bs * 255.0));       // OpenCV's Sobel scale for ksize 3 (SURVEY A.6 step 1)
    const double s2 = (double)scale * (double)scale;
    const int nout = EW - bs + 1;
    dim3 grid((W + nout - 1) / nout, (H + ERS - 1) / ERS);
    eig_kernel<<<grid, EW, eig_smem_bytes(bs), st>>>(gray, H, W, pitch, bs, s2, harris ? 1 : 0, (float)k, eig, eig_pitch_bytes / 4, mask, mask_pitch, maxbits);
    return check_launch("eig_kernel");
}

// ---------------------------------------------------------------------------------------------
// The other Sobel apertures of cv2's cornerEigenValsVecs (ksize / gradientSize = -1 (Scharr), 1, 5, 7).  dx correlates the
// derivative taps d along x and the smoothing taps s along y, dy the transpose; every aperture is written as KT = 3, 5 or 7
// taps (ksize 1: s = 0 1 0), so the Sobel radius is KT / 2.  OpenCV scales the derivatives by 1 / (sden * blockSize * 255):
//     g    d                   s                   sden   max |sx| on u8
//     1    -1 0 1              (0) 1 (0)             1      255
//     3    -1 0 1              1 2 1                 4      1 020        (eig_kernel / eig_nms_kernel above)
//    -1    -1 0 1              3 10 3                8      4 080
//     5    -1 -2 0 2 1         1 4 6 4 1            16      12 240
//     7    -1 -4 -5 0 5 4 1    1 6 15 20 15 6 1     64      163 200
// Aperture 3's exact int32 sums do not carry over: a blockSize-31 window sum of sx^2 reaches 1.6e10 (Scharr), 1.4e11 (5) and
// 2.6e13 (7) (6.2e7 for 1).  These kernels sum the products in int64; every sum stays below 2^53, so the conversion to double
// before the scaling is exact as well.
__host__ __device__ constexpr int ap_taps(int g) { return g == 5 ? 5 : g == 7 ? 7 : 3; }
__host__ __device__ constexpr int ap_d(int g, int j)
{
    return g == 5 ? (j == 0 ? -1 : j == 1 ? -2 : j == 2 ? 0 : j == 3 ? 2 : 1)
         : g == 7 ? (j == 0 ? -1 : j == 1 ? -4 : j == 2 ? -5 : j == 3 ? 0 : j == 4 ? 5 : j == 5 ? 4 : 1)
         : j - 1;
}
__host__ __device__ constexpr int ap_s(int g, int j)
{
    return g == 5 ? (j == 0 || j == 4 ? 1 : j == 2 ? 6 : 4)
         : g == 7 ? (j == 0 || j == 6 ? 1 : j == 1 || j == 5 ? 6 : j == 2 || j == 4 ? 15 : 20)
         : g == 1 ? (j == 1 ? 1 : 0)
         : g == -1 ? (j == 1 ? 10 : 3)
         : (j == 1 ? 2 : 1);
}
static bool ap_supported(int g) { return g == -1 || g == 1 || g == 3 || g == 5 || g == 7; }
static float ap_scale(int g, int bs)                  // OpenCV's Sobel / Scharr scale of cornerEigenValsVecs, rounded to float
{
    const double sden = g == -1 ? 8.0 : (double)(1 << (g - 1));
    return (float)(1.0 / (sden * bs * 255.0));
}

// eig_kernel for the apertures above: each thread gathers the KT x KT bytes of its support pixel; products, ring and sums in int64
template <int G>
__global__ void __launch_bounds__(EW)
eig_ap_kernel(const uint8_t *__restrict__ img, int H, int W, int64_t pitch, int bs, double s2, int harris, float harris_k,
              float *__restrict__ eig, int64_t eig_pitch_f)
{
    constexpr int KT = ap_taps(G), R = KT / 2;
    extern __shared__ long long eap_smem[];
    long long *prod = eap_smem;                      // [2][3][EW]   products of the current support row (double-buffered)
    long long *ring = eap_smem + 2 * 3 * EW;         // [bs][3][EW]  horizontal window sums of the last bs support rows
    const int t = threadIdx.x;
    const int nout = EW - bs + 1;
    const int a0 = -(bs / 2);
    const int X0 = blockIdx.x * nout, Y0 = blockIdx.y * ERS;
    const int x = X0 + t;
    const bool xout = t < nout && x < W;
    const int px = r101(X0 + a0 + t, W);             // REFLECT_101 on the product image, then again on the source
    int cx[KT];
#pragma unroll
    for (int j = 0; j < KT; j++) cx[j] = r101(px + j - R, W);
    long long vs0 = 0, vs1 = 0, vs2 = 0;
    const int nrows = min(ERS, H - Y0) + bs - 1;
    int slot = 0;
    for (int k = 0; k < nrows; k++) {
        const int py = r101(Y0 + a0 + k, H);
        int sx = 0, sy = 0;
#pragma unroll
        for (int i = 0; i < KT; i++) {
            const uint8_t *row = img + (int64_t)r101(py + i - R, H) * pitch;
            int hd = 0, hs = 0;
#pragma unroll
            for (int j = 0; j < KT; j++) { const int v = row[cx[j]]; hd += ap_d(G, j) * v; hs += ap_s(G, j) * v; }
            sx += ap_s(G, i) * hd; sy += ap_d(G, i) * hs;
        }
        long long *pb = prod + (k & 1) * 3 * EW;
        pb[t] = (long long)sx * sx; pb[EW + t] = (long long)sx * sy; pb[2 * EW + t] = (long long)sy * sy;
        __syncthreads();
        if (t < nout) {
            long long h0 = 0, h1 = 0, h2 = 0;
            for (int j = 0; j < bs; j++) { h0 += pb[t + j]; h1 += pb[EW + t + j]; h2 += pb[2 * EW + t + j]; }
            long long *rg = ring + slot * 3 * EW;
            if (k >= bs) { vs0 -= rg[t]; vs1 -= rg[EW + t]; vs2 -= rg[2 * EW + t]; }
            vs0 += h0; vs1 += h1; vs2 += h2;
            rg[t] = h0; rg[EW + t] = h1; rg[2 * EW + t] = h2;
            if (k >= bs - 1 && xout) {
                const int y = Y0 + k - (bs - 1);
                float e;
                if (harris) {                                   // cv2.cornerHarris: (a*c - b*b) - k*((a + c)*(a + c)), float, unfused
                    const float a = (float)((double)vs0 * s2), b = (float)((double)vs1 * s2), c = (float)((double)vs2 * s2);
                    const float tr = __fadd_rn(a, c);
                    e = __fsub_rn(__fsub_rn(__fmul_rn(a, c), __fmul_rn(b, b)), __fmul_rn(harris_k, __fmul_rn(tr, tr)));
                } else {
                    const float a = __fmul_rn((float)((double)vs0 * s2), 0.5f), b = (float)((double)vs1 * s2);
                    const float c = __fmul_rn((float)((double)vs2 * s2), 0.5f);
                    const float d = __fsub_rn(a, c);
                    e = __fsub_rn(__fadd_rn(a, c), __fsqrt_rn(__fadd_rn(__fmul_rn(d, d), __fmul_rn(b, b))));
                }
                eig[(int64_t)y * eig_pitch_f + x] = e;
            }
        }
        slot = slot + 1 == bs ? 0 : slot + 1;
    }
}

static size_t eig_ap_smem_bytes(int bs) { return (size_t)(2 + bs) * 3 * EW * sizeof(long long); }

template <int G>
static int launch_eig_ap_g(const uint8_t *gray, int H, int W, int64_t pitch, int bs, int harris, double k, float *eig,
                           int64_t eig_pitch_bytes, cudaStream_t st)
{
    if (eig_ap_smem_bytes(bs) > 48 * 1024)
        IBT_CUDA_TRY(cudaFuncSetAttribute(eig_ap_kernel<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)eig_ap_smem_bytes(MAX_BLOCK)));
    const float scale = ap_scale(G, bs);
    const double s2 = (double)scale * (double)scale;
    const int nout = EW - bs + 1;
    dim3 grid((W + nout - 1) / nout, (H + ERS - 1) / ERS);
    eig_ap_kernel<G><<<grid, EW, eig_ap_smem_bytes(bs), st>>>(gray, H, W, pitch, bs, s2, harris ? 1 : 0, (float)k, eig, eig_pitch_bytes / 4);
    return check_launch("eig_ap_kernel");
}

// the map hooks: aperture 3 keeps eig_kernel
static int launch_eig_ksize(const uint8_t *gray, int H, int W, int64_t pitch, int bs, int ksize, int harris, double k, float *eig,
                            int64_t eig_pitch_bytes, cudaStream_t st)
{
    if (!ap_supported(ksize)) return IBT_E_INVALID;
    if (ksize == 3) return launch_eig(gray, H, W, pitch, bs, harris, k, eig, eig_pitch_bytes, nullptr, 0, nullptr, st);
    if (!gray || !eig || H <= 0 || W <= 0 || bs < 1 || bs > MAX_BLOCK || pitch < W || eig_pitch_bytes % 4 != 0 ||
        eig_pitch_bytes < (int64_t)W * 4)
        return IBT_E_INVALID;
    switch (ksize) {
    case -1: return launch_eig_ap_g<-1>(gray, H, W, pitch, bs, harris, k, eig, eig_pitch_bytes, st);
    case 1: return launch_eig_ap_g<1>(gray, H, W, pitch, bs, harris, k, eig, eig_pitch_bytes, st);
    case 5: return launch_eig_ap_g<5>(gray, H, W, pitch, bs, harris, k, eig, eig_pitch_bytes, st);
    default: return launch_eig_ap_g<7>(gray, H, W, pitch, bs, harris, k, eig, eig_pitch_bytes, st);
    }
}

// ---------------------------------------------------------------------------------------------
// K2a/K2b fused: response + raw 3x3 maxima, one warp per (column strip, row chunk)
enum : uint8_t { ST_UNDECIDED = 0, ST_ACCEPTED = 1, ST_REJECTED = 2 };

struct GfttCounters {
    uint32_t maxbits;        // enc_f32 of the masked maximum, 0 = no allowed pixel
    uint32_t ncand;          // raw maxima appended by K2a (may exceed capacity)
    uint32_t nsel;           // candidates selected for ranking
    uint32_t nacc;           // accepted after culling
    uint32_t nout;           // corners written (min(nacc, limit))
    int32_t error;           // IBT_E_* raised on the device (capacity)
    uint32_t bar;            // grid barrier of K2b
    uint32_t pad;
    uint32_t remaining[64];  // undecided ranks left after culling round k (mod 64)
    uint32_t hist[4096];     // candidates above the threshold per top-12-bit bin of the ordered response
    unsigned long long tstamp[16];   // %globaltimer at the phase boundaries of K2b (CTA 0; tools/prof_gftt.py prints them)
};
__device__ __forceinline__ void stamp(GfttCounters *cnt, int i)
{
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        cnt->tstamp[i] = t;
    }
}

constexpr int EN_WARPS = 4;               // warps per CTA (independent of each other: no block-level barrier)
constexpr int EN_COLS = 128;              // support columns per warp (4 per lane)
constexpr int EN_CB = 192;                // per-warp candidate buffer (flushed every 8 rows once it holds >= 96 entries)
constexpr int EN_PAD = 32;                // generic blockSize: padding of the shared row buffer on both sides
constexpr int EN_MIN_CTAS = 5;            // CTAs of 4 warps per SM the register budget is compiled for
constexpr int EN_BORDER_SPLIT = 4;        // border strips (byte gathers, ~4x slower per row) get 4x shorter jobs
constexpr int EN_AP_MIN_CTAS = 3;         // eig_nms_ap_kernel: the tap rows and 64-bit sums need more registers

struct EigNmsArgs {
    const uint8_t *img; int H, W; int64_t pitch;
    const uint8_t *mask; int64_t mask_pitch;
    int bs;
    float harris_k;           // HARRIS instantiations only: k of cv2.cornerHarris, rounded to float as OpenCV's calcHarris does
    double s2, s2h, quality;
    GfttCounters *cnt; unsigned long long *keys; uint32_t cap;
    int outw, left, nstrips, word_ok;
    int first_right;          // strips >= first_right (and strip 0) reach outside the image: border variant
    int nborder, rows_border, chunks_border, rows_fast, njobs;
    int warp_smem_ints;      // per-warp shared memory (ring + candidate buffer + row buffer), in ints
};

__device__ __forceinline__ int dp4a_uu_(uint32_t a, uint32_t b) { return (int)__dp4a(a, b, 0u); }
__device__ __forceinline__ int dp4a_us_(uint32_t a, int b)
{
    int d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(0));
    return d;
}

// horizontal taps of one image row for the lane's 4 pixels: hx = I[x+1] - I[x-1], hs = I[x-1] + 2 I[x] + I[x+1]
__device__ __forceinline__ void taps_word(uint32_t w, int *hx, int *hs)
{
    const uint32_t L = __shfl_up_sync(0xffffffffu, w, 1), R = __shfl_down_sync(0xffffffffu, w, 1);
    // byte windows (x-1, x, x+1, .) of the four pixels
    const uint32_t w0 = __funnelshift_r(L, w, 24), w2 = __funnelshift_r(w, R, 8), w3 = __funnelshift_r(w, R, 16);
    hx[0] = dp4a_us_(w0, 0x000100FF); hx[1] = dp4a_us_(w, 0x000100FF);
    hx[2] = dp4a_us_(w2, 0x000100FF); hx[3] = dp4a_us_(w3, 0x000100FF);
    hs[0] = dp4a_uu_(w0, 0x00010201u); hs[1] = dp4a_uu_(w, 0x00010201u);
    hs[2] = dp4a_uu_(w2, 0x00010201u); hs[3] = dp4a_uu_(w3, 0x00010201u);
}
__device__ __forceinline__ void taps_bytes(const uint8_t *__restrict__ row, const int *pc, const int *pm, const int *pp, int *hx, int *hs)
{
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int m = __ldg(row + pm[k]), c = __ldg(row + pc[k]), p = __ldg(row + pp[k]);
        hx[k] = p - m;
        hs[k] = m + 2 * c + p;
    }
}

// window sum over columns [x + a0, x + a0 + BS) of a plane held as 4 values per lane (compile-time blockSize):
// the BS + 3 values the lane's four windows touch are gathered from the neighbouring lanes, then three slides.
template <int BS>
__device__ __forceinline__ void hbox_shfl(const int *v, int *out, int lane)
{
    constexpr int A0 = -(BS / 2);
    int g[BS + 3];
#pragma unroll
    for (int i = 0; i < BS + 3; i++) {
        const int rel = A0 + i;                              // column offset from the lane's first pixel
        const int dl = rel >= 0 ? rel / 4 : -((3 - rel) / 4);  // floor(rel / 4)
        const int comp = rel - 4 * dl;
        g[i] = dl == 0 ? v[comp] : __shfl_sync(0xffffffffu, v[comp], lane + dl);
    }
    int s = 0;
#pragma unroll
    for (int i = 0; i < BS; i++) s += g[i];
    out[0] = s;
#pragma unroll
    for (int k = 1; k < 4; k++) { s += g[k - 1 + BS] - g[k - 1]; out[k] = s; }
}

// runtime blockSize: the plane goes through a padded shared-memory row, one direct sum + three slides per lane
__device__ __forceinline__ void hbox_smem(const int *v, int *out, int *rowbuf, int bs, int lane)
{
    const int a0 = -(bs / 2);
    __syncwarp();
    *reinterpret_cast<int4 *>(rowbuf + EN_PAD + 4 * lane) = make_int4(v[0], v[1], v[2], v[3]);
    __syncwarp();
    const int *p = rowbuf + EN_PAD + 4 * lane + a0;
    int s = 0;
    for (int j = 0; j < bs; j++) s += p[j];
    out[0] = s;
#pragma unroll
    for (int k = 1; k < 4; k++) { s += p[k - 1 + bs] - p[k - 1]; out[k] = s; }
}

template <int BS, bool MASK, bool BORDER, bool HARRIS>
__device__ __forceinline__ void eig_nms_job(const EigNmsArgs &a, int strip, int Y0, int Y1, int *wsm, int lane)
{
    const int bs = BS ? BS : a.bs;
    const int a0 = -(bs / 2);
    const int H = a.H, W = a.W;
    const int ox0 = strip * a.outw;                       // first output column of the strip
    const int c0 = ox0 - a.left + 4 * lane;               // support column of this lane's pixel 0 (multiple of 4)
    const int ey0 = max(0, Y0 - 1), ey1 = min(H - 1, Y1);         // response rows needed (NMS halo rows included)
    uint32_t *ring = reinterpret_cast<uint32_t *>(wsm);           // [bs][128]: (sx & 0xffff) | (sy << 16) of the last bs product rows
    unsigned long long *cbuf = reinterpret_cast<unsigned long long *>(wsm + bs * EN_COLS);
    int *scount = reinterpret_cast<int *>(cbuf + EN_CB);          // entries in cbuf (may run past EN_CB: those went straight to global)
    int *rowbuf = scount + 4;                                     // generic blockSize only: [EN_PAD + 128 + EN_PAD]
    unsigned outmask = 0, candmask = 0;                           // pixels this lane owns / may emit
    int pc[4], pm[4], pp[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int c = c0 + k;
        const bool own = c >= ox0 && c < ox0 + a.outw && c < W;
        if (own) outmask |= 1u << k;
        if (own && c >= 1 && c <= W - 2) candmask |= 1u << k;
        pc[k] = r101(c, W);                                       // REFLECT_101 on the product image ...
        pm[k] = r101(pc[k] - 1, W); pp[k] = r101(pc[k] + 1, W);   // ... whose Sobel reflects the source again
    }
    if (lane == 0) *scount = 0;
    __syncwarp();
    int vxx[4] = {0, 0, 0, 0}, vxy[4] = {0, 0, 0, 0}, vyy[4] = {0, 0, 0, 0};
    float m3a[4], m3b[4], eprev[4];
#pragma unroll
    for (int k = 0; k < 4; k++) { m3a[k] = m3b[k] = -FLT_MAX; eprev[k] = 0.f; }
    unsigned mprev = 0;                                           // mask bits of the previous response row
    float lmax = -FLT_MAX;
    bool have_max = false;
    float thr_lb = 0.f;
    {
        const uint32_t mb = *reinterpret_cast<volatile const uint32_t *>(&a.cnt->maxbits);
        if (mb) thr_lb = fmaxf(0.f, (float)((double)dec_f32(mb) * a.quality));
    }
    auto flush = [&]() {
        __syncwarp();
        const int ncb = min(*reinterpret_cast<volatile int *>(scount), EN_CB);
        unsigned base = 0;
        if (lane == 0 && ncb) base = atomicAdd(&a.cnt->ncand, (unsigned)ncb);
        base = __shfl_sync(0xffffffffu, base, 0);
        for (int i = lane; i < ncb; i += 32)
            if (base + i < a.cap) a.keys[base + i] = cbuf[i];
        __syncwarp();
        if (lane == 0) *scount = 0;
        __syncwarp();
    };
    const int p_first = ey0 + a0, p_last = ey1 + a0 + bs - 1;
    int slot = 0;
    // taps of the image rows (rp-1, rp, rp+1) of product row p; rolled while the rows advance one by one
    int hxA[4], hsA[4], hxB[4], hsB[4], hxC[4], hsC[4];
    bool have = false;
    uint32_t wnext = 0;
    bool wnext_ok = false;
    for (int p = p_first; p <= p_last; p++) {
        // ---- taps of the three image rows under support row p ---------------------------------------------------------
        if (have && p >= 1 && p <= H - 2) {               // rows p-1, p are held: only row p+1 is new
#pragma unroll
            for (int k = 0; k < 4; k++) { hxA[k] = hxB[k]; hsA[k] = hsB[k]; hxB[k] = hxC[k]; hsB[k] = hsC[k]; }
            const uint8_t *rowC = a.img + (int64_t)(p + 1) * a.pitch;
            if (BORDER) taps_bytes(rowC, pc, pm, pp, hxC, hsC);
            else taps_word(wnext_ok ? wnext : __ldg(reinterpret_cast<const uint32_t *>(rowC + c0)), hxC, hsC);
        } else {
            const int rp = r101(p, H);
            const uint8_t *rowA = a.img + (int64_t)r101(rp - 1, H) * a.pitch;
            const uint8_t *rowB = a.img + (int64_t)rp * a.pitch;
            const uint8_t *rowC = a.img + (int64_t)r101(rp + 1, H) * a.pitch;
            if (BORDER) {
                taps_bytes(rowA, pc, pm, pp, hxA, hsA); taps_bytes(rowB, pc, pm, pp, hxB, hsB); taps_bytes(rowC, pc, pm, pp, hxC, hsC);
            } else {
                const uint32_t wa = __ldg(reinterpret_cast<const uint32_t *>(rowA + c0));
                const uint32_t wb = __ldg(reinterpret_cast<const uint32_t *>(rowB + c0));
                const uint32_t wc = __ldg(reinterpret_cast<const uint32_t *>(rowC + c0));
                taps_word(wa, hxA, hsA); taps_word(wb, hxB, hsB); taps_word(wc, hxC, hsC);
            }
        }
        have = p >= 0;                                    // (for p >= 0 the held rows B, C are the image rows p, p+1)
        wnext_ok = false;
        if (!BORDER && p >= 0 && p + 1 <= H - 2) {        // the next iteration rolls: fetch its new row (p + 2) now
            wnext = __ldg(reinterpret_cast<const uint32_t *>(a.img + (int64_t)(p + 2) * a.pitch + c0));
            wnext_ok = true;
        }
        // ---- vertical sliding sums of the products; the ring keeps (sx, sy) of the last bs rows -------------------------
        uint4 *rg = reinterpret_cast<uint4 *>(ring + slot * EN_COLS) + lane;
        if (p - p_first >= bs) {
            const uint4 o = *rg;
            const uint32_t ow[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int ox = (int)(short)(ow[k] & 0xffffu), oy = (int)ow[k] >> 16;
                vxx[k] -= ox * ox; vxy[k] -= ox * oy; vyy[k] -= oy * oy;
            }
        }
        uint32_t nw[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int sx = hxA[k] + 2 * hxB[k] + hxC[k], sy = hsC[k] - hsA[k];
            vxx[k] += sx * sx; vxy[k] += sx * sy; vyy[k] += sy * sy;
            nw[k] = ((uint32_t)sx & 0xffffu) | ((uint32_t)sy << 16);
        }
        *rg = make_uint4(nw[0], nw[1], nw[2], nw[3]);
        slot = slot + 1 == bs ? 0 : slot + 1;
        const int y = p - a0 - bs + 1;                    // response row completed by this product row
        if (y < ey0) continue;
        // ---- horizontal window sums, lambda_min --------------------------------------------------------------------------
        int bxx[4], bxy[4], byy[4];
        if (BS) {
            hbox_shfl<BS ? BS : 1>(vxx, bxx, lane); hbox_shfl<BS ? BS : 1>(vxy, bxy, lane); hbox_shfl<BS ? BS : 1>(vyy, byy, lane);
        } else {
            hbox_smem(vxx, bxx, rowbuf, bs, lane); hbox_smem(vxy, bxy, rowbuf, bs, lane); hbox_smem(vyy, byy, rowbuf, bs, lane);
        }
        float e[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (HARRIS) {                                 // cv2.cornerHarris: (a*c - b*b) - k*((a + c)*(a + c)), float, unfused
                const float fa = (float)((double)bxx[k] * a.s2), fb = (float)((double)bxy[k] * a.s2);
                const float fc = (float)((double)byy[k] * a.s2);
                const float tr = __fadd_rn(fa, fc);
                e[k] = __fsub_rn(__fsub_rn(__fmul_rn(fa, fc), __fmul_rn(fb, fb)), __fmul_rn(a.harris_k, __fmul_rn(tr, tr)));
            } else {
                const float fa = (float)((double)bxx[k] * a.s2h), fb = (float)((double)bxy[k] * a.s2);
                const float fc = (float)((double)byy[k] * a.s2h);
                const float d = __fsub_rn(fa, fc);
                e[k] = __fsub_rn(__fadd_rn(fa, fc), __fsqrt_rn(__fadd_rn(__fmul_rn(d, d), __fmul_rn(fb, fb))));
            }
        }
        // ---- masked maximum over the pixels this lane owns ------------------------------------------------------------------
        unsigned mcur = 0xfu;
        if (MASK) {
            mcur = 0;
#pragma unroll
            for (int k = 0; k < 4; k++)
                if ((outmask >> k) & 1u) mcur |= (a.mask[(int64_t)y * a.mask_pitch + c0 + k] ? 1u : 0u) << k;
        }
        if (y >= Y0 && y < Y1) {
#pragma unroll
            for (int k = 0; k < 4; k++)
                if (((outmask & mcur) >> k) & 1u) { lmax = fmaxf(lmax, e[k]); have_max = true; }
        }
        // ---- 3x3 raw maxima of the previous row -------------------------------------------------------------------------------
        const float el = __shfl_up_sync(0xffffffffu, e[3], 1), er = __shfl_down_sync(0xffffffffu, e[0], 1);
        float m3c[4];
        m3c[0] = fmaxf(fmaxf(el, e[0]), e[1]); m3c[1] = fmaxf(fmaxf(e[0], e[1]), e[2]);
        m3c[2] = fmaxf(fmaxf(e[1], e[2]), e[3]); m3c[3] = fmaxf(fmaxf(e[2], e[3]), er);
        const int yc = y - 1;
        if (yc >= max(Y0, 1) && yc < Y1 && yc <= H - 2) {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const float v = eprev[k];
                if ((((candmask & mprev) >> k) & 1u) && v > thr_lb && v == fmaxf(fmaxf(m3a[k], m3b[k]), m3c[k])) {
                    const unsigned long long key = ((unsigned long long)enc_f32(v) << 32) | (uint32_t)(yc * W + c0 + k);
                    const int pos = atomicAdd(scount, 1);
                    if (pos < EN_CB) cbuf[pos] = key;
                    else {                                              // buffer full (plateaus): straight to the global list
                        const unsigned g = atomicAdd(&a.cnt->ncand, 1u);
                        if (g < a.cap) a.keys[g] = key;
                    }
                }
            }
        }
#pragma unroll
        for (int k = 0; k < 4; k++) { m3a[k] = m3b[k]; m3b[k] = m3c[k]; eprev[k] = e[k]; }
        mprev = mcur;
        if ((y & 7) == 7) {
            __syncwarp();
            if (*reinterpret_cast<volatile int *>(scount) >= EN_CB / 2) flush();
            if ((y & 31) == 31) {                         // tighten the threshold bound with what this warp has seen
                float wm = lmax;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) wm = fmaxf(wm, __shfl_xor_sync(0xffffffffu, wm, o));
                if (wm > 0.f) thr_lb = fmaxf(thr_lb, (float)((double)wm * a.quality));
            }
        }
    }
    flush();
    uint32_t lbits = have_max ? enc_f32(lmax) : 0u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lbits = max(lbits, __shfl_xor_sync(0xffffffffu, lbits, o));
    if (lane == 0 && lbits) atomicMax(&a.cnt->maxbits, lbits);
}

template <int BS, bool MASK, bool HARRIS = false>
__global__ void __launch_bounds__(EN_WARPS * 32, EN_MIN_CTAS)
eig_nms_kernel(const __grid_constant__ EigNmsArgs a)
{
    extern __shared__ __align__(16) int en_smem[];
    pdl_launch_dependents();                              // (the selection kernel's CTAs may take their places while this grid drains)
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int job = blockIdx.x * EN_WARPS + wib;
    if (job >= a.njobs) return;
    int *wsm = en_smem + (size_t)wib * a.warp_smem_ints;
    // jobs [0, nborder * chunks_border): strips that reach outside the image (or every strip of an unaligned image), in
    // short row chunks: their byte gathers make a row ~4x slower, and the launch is one wave -- the longest job sets its time
    const int nbj = a.nborder * a.chunks_border;
    if (job < nbj) {
        const int sb = job % a.nborder, chunk = job / a.nborder;
        const int strip = a.nborder == a.nstrips ? sb : (sb == 0 ? 0 : a.first_right + sb - 1);
        const int Y0 = chunk * a.rows_border;
        eig_nms_job<BS, MASK, true, HARRIS>(a, strip, Y0, min(a.H, Y0 + a.rows_border), wsm, lane);
    } else {
        const int j = job - nbj, nfast = a.nstrips - a.nborder;
        const int strip = 1 + j % nfast, chunk = j / nfast;
        const int Y0 = chunk * a.rows_fast;
        eig_nms_job<BS, MASK, false, HARRIS>(a, strip, Y0, min(a.H, Y0 + a.rows_fast), wsm, lane);
    }
}

template <int BS, bool HARRIS = false>
static int launch_eig_nms_bs(const EigNmsArgs &a, cudaStream_t st)
{
    const size_t smem = (size_t)a.warp_smem_ints * 4 * EN_WARPS;
    const int blocks = (a.njobs + EN_WARPS - 1) / EN_WARPS;
    if (a.mask) {
        if (smem > 48 * 1024) IBT_CUDA_TRY(cudaFuncSetAttribute(eig_nms_kernel<BS, true, HARRIS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        eig_nms_kernel<BS, true, HARRIS><<<blocks, EN_WARPS * 32, smem, st>>>(a);
    } else {
        if (smem > 48 * 1024) IBT_CUDA_TRY(cudaFuncSetAttribute(eig_nms_kernel<BS, false, HARRIS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        eig_nms_kernel<BS, false, HARRIS><<<blocks, EN_WARPS * 32, smem, st>>>(a);
    }
    return check_launch("eig_nms_kernel");
}

// ---- K2a for the apertures other than 3 (table at eig_ap_kernel).  eig_nms_job's structure: one warp per (strip, row chunk),
// four adjacent columns per lane, rows top to bottom, word loads on the inner strips and byte gathers on the border strips;
// what changes is the front end.  The horizontal taps of an image row reach KT / 2 columns (bytes of the neighbour lanes'
// words, or gathers), the vertical taps combine the last KT rows of horizontal taps (held in registers), the ring keeps
// (sx, sy) as two int32 (|sx| reaches 163 200 at aperture 7) and the vertical and horizontal window sums are int64.
template <int G>
__device__ __forceinline__ void ap_taps_word(uint32_t w, int *hd, int *hs)
{
    constexpr int KT = ap_taps(G), R = KT / 2;
    const uint32_t L = __shfl_up_sync(0xffffffffu, w, 1), Rt = __shfl_down_sync(0xffffffffu, w, 1);
    int b[4 + 2 * R];                                             // bytes of columns c0 - R .. c0 + 3 + R
#pragma unroll
    for (int i = 0; i < 4 + 2 * R; i++) {
        const int rel = i - R;
        b[i] = (int)(((rel < 0 ? L : rel < 4 ? w : Rt) >> (((rel + 4) & 3) * 8)) & 0xffu);
    }
#pragma unroll
    for (int k = 0; k < 4; k++) {
        int d = 0, s = 0;
#pragma unroll
        for (int j = 0; j < KT; j++) { d += ap_d(G, j) * b[k + j]; s += ap_s(G, j) * b[k + j]; }
        hd[k] = d; hs[k] = s;
    }
}

// hbox_smem on int64 sums
__device__ __forceinline__ void hbox_smem64(const long long *v, long long *out, long long *rowbuf, int bs, int lane)
{
    const int a0 = -(bs / 2);
    __syncwarp();
    reinterpret_cast<longlong2 *>(rowbuf + EN_PAD + 4 * lane)[0] = make_longlong2(v[0], v[1]);
    reinterpret_cast<longlong2 *>(rowbuf + EN_PAD + 4 * lane)[1] = make_longlong2(v[2], v[3]);
    __syncwarp();
    const long long *p = rowbuf + EN_PAD + 4 * lane + a0;
    long long s = 0;
    for (int j = 0; j < bs; j++) s += p[j];
    out[0] = s;
#pragma unroll
    for (int k = 1; k < 4; k++) { s += p[k - 1 + bs] - p[k - 1]; out[k] = s; }
}

template <int G, bool MASK, bool BORDER, bool HARRIS>
__device__ __forceinline__ void eig_nms_ap_job(const EigNmsArgs &a, int strip, int Y0, int Y1, int *wsm, int lane)
{
    constexpr int KT = ap_taps(G), R = KT / 2;
    const int bs = a.bs;
    const int a0 = -(bs / 2);
    const int H = a.H, W = a.W;
    const int ox0 = strip * a.outw;                       // first output column of the strip
    const int c0 = ox0 - a.left + 4 * lane;               // support column of this lane's pixel 0 (multiple of 4)
    const int ey0 = max(0, Y0 - 1), ey1 = min(H - 1, Y1);         // response rows needed (NMS halo rows included)
    int *ring = wsm;                                              // [bs][128][2]: (sx, sy) of the last bs product rows
    unsigned long long *cbuf = reinterpret_cast<unsigned long long *>(wsm + bs * 2 * EN_COLS);
    int *scount = reinterpret_cast<int *>(cbuf + EN_CB);          // entries in cbuf (may run past EN_CB: those went straight to global)
    long long *rowbuf = reinterpret_cast<long long *>(scount + 4);  // [EN_PAD + 128 + EN_PAD]
    unsigned outmask = 0, candmask = 0;                           // pixels this lane owns / may emit
    int cx[4][KT];                                                // border strips: source columns of the lane's horizontal taps
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int c = c0 + k;
        const bool own = c >= ox0 && c < ox0 + a.outw && c < W;
        if (own) outmask |= 1u << k;
        if (own && c >= 1 && c <= W - 2) candmask |= 1u << k;
        const int pc = r101(c, W);                                // REFLECT_101 on the product image ...
#pragma unroll
        for (int j = 0; j < KT; j++) cx[k][j] = BORDER ? r101(pc + j - R, W) : 0;   // ... whose Sobel reflects the source again
    }
    if (lane == 0) *scount = 0;
    __syncwarp();
    long long vxx[4] = {0, 0, 0, 0}, vxy[4] = {0, 0, 0, 0}, vyy[4] = {0, 0, 0, 0};
    float m3a[4], m3b[4], eprev[4];
#pragma unroll
    for (int k = 0; k < 4; k++) { m3a[k] = m3b[k] = -FLT_MAX; eprev[k] = 0.f; }
    unsigned mprev = 0;                                           // mask bits of the previous response row
    float lmax = -FLT_MAX;
    bool have_max = false;
    float thr_lb = 0.f;
    {
        const uint32_t mb = *reinterpret_cast<volatile const uint32_t *>(&a.cnt->maxbits);
        if (mb) thr_lb = fmaxf(0.f, (float)((double)dec_f32(mb) * a.quality));
    }
    auto flush = [&]() {
        __syncwarp();
        const int ncb = min(*reinterpret_cast<volatile int *>(scount), EN_CB);
        unsigned base = 0;
        if (lane == 0 && ncb) base = atomicAdd(&a.cnt->ncand, (unsigned)ncb);
        base = __shfl_sync(0xffffffffu, base, 0);
        for (int i = lane; i < ncb; i += 32)
            if (base + i < a.cap) a.keys[base + i] = cbuf[i];
        __syncwarp();
        if (lane == 0) *scount = 0;
        __syncwarp();
    };
    auto row_taps = [&](const uint8_t *row, int *hd, int *hs) {
        if (BORDER) {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                int d = 0, s = 0;
#pragma unroll
                for (int j = 0; j < KT; j++) { const int v = __ldg(row + cx[k][j]); d += ap_d(G, j) * v; s += ap_s(G, j) * v; }
                hd[k] = d; hs[k] = s;
            }
        } else {
            ap_taps_word<G>(__ldg(reinterpret_cast<const uint32_t *>(row + c0)), hd, hs);
        }
    };
    const int p_first = ey0 + a0, p_last = ey1 + a0 + bs - 1;
    int slot = 0;
    int hd[KT][4], hs[KT][4];                             // horizontal taps of the KT image rows under product row p, top to bottom
    bool have = false;                                    // they hold the unreflected rows p-1-R .. p-1+R
    for (int p = p_first; p <= p_last; p++) {
        if (have && p + R <= H - 1) {                     // only row p+R is new
#pragma unroll
            for (int i = 0; i + 1 < KT; i++)
#pragma unroll
                for (int k = 0; k < 4; k++) { hd[i][k] = hd[i + 1][k]; hs[i][k] = hs[i + 1][k]; }
            row_taps(a.img + (int64_t)(p + R) * a.pitch, hd[KT - 1], hs[KT - 1]);
        } else {
            const int rp = r101(p, H);
#pragma unroll
            for (int i = 0; i < KT; i++) row_taps(a.img + (int64_t)r101(rp + i - R, H) * a.pitch, hd[i], hs[i]);
        }
        have = p - R >= 0 && p + R <= H - 1;
        // ---- vertical sliding sums of the products; the ring keeps (sx, sy) of the last bs rows -------------------------
        int4 *rg = reinterpret_cast<int4 *>(ring + slot * 2 * EN_COLS) + 2 * lane;
        if (p - p_first >= bs) {
            const int4 o0 = rg[0], o1 = rg[1];
            const int ox[4] = {o0.x, o0.z, o1.x, o1.z}, oy[4] = {o0.y, o0.w, o1.y, o1.w};
#pragma unroll
            for (int k = 0; k < 4; k++) {
                vxx[k] -= (long long)ox[k] * ox[k]; vxy[k] -= (long long)ox[k] * oy[k]; vyy[k] -= (long long)oy[k] * oy[k];
            }
        }
        int sx[4], sy[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            int x = 0, y = 0;
#pragma unroll
            for (int i = 0; i < KT; i++) { x += ap_s(G, i) * hd[i][k]; y += ap_d(G, i) * hs[i][k]; }
            sx[k] = x; sy[k] = y;
            vxx[k] += (long long)x * x; vxy[k] += (long long)x * y; vyy[k] += (long long)y * y;
        }
        rg[0] = make_int4(sx[0], sy[0], sx[1], sy[1]);
        rg[1] = make_int4(sx[2], sy[2], sx[3], sy[3]);
        slot = slot + 1 == bs ? 0 : slot + 1;
        const int y = p - a0 - bs + 1;                    // response row completed by this product row
        if (y < ey0) continue;
        // ---- horizontal window sums, response ----------------------------------------------------------------------------
        long long bxx[4], bxy[4], byy[4];
        hbox_smem64(vxx, bxx, rowbuf, bs, lane); hbox_smem64(vxy, bxy, rowbuf, bs, lane); hbox_smem64(vyy, byy, rowbuf, bs, lane);
        float e[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (HARRIS) {                                 // cv2.cornerHarris: (a*c - b*b) - k*((a + c)*(a + c)), float, unfused
                const float fa = (float)((double)bxx[k] * a.s2), fb = (float)((double)bxy[k] * a.s2);
                const float fc = (float)((double)byy[k] * a.s2);
                const float tr = __fadd_rn(fa, fc);
                e[k] = __fsub_rn(__fsub_rn(__fmul_rn(fa, fc), __fmul_rn(fb, fb)), __fmul_rn(a.harris_k, __fmul_rn(tr, tr)));
            } else {
                const float fa = (float)((double)bxx[k] * a.s2h), fb = (float)((double)bxy[k] * a.s2);
                const float fc = (float)((double)byy[k] * a.s2h);
                const float d = __fsub_rn(fa, fc);
                e[k] = __fsub_rn(__fadd_rn(fa, fc), __fsqrt_rn(__fadd_rn(__fmul_rn(d, d), __fmul_rn(fb, fb))));
            }
        }
        // ---- masked maximum, 3x3 raw maxima of the previous row, candidate buffer: as eig_nms_job ----------------------------
        unsigned mcur = 0xfu;
        if (MASK) {
            mcur = 0;
#pragma unroll
            for (int k = 0; k < 4; k++)
                if ((outmask >> k) & 1u) mcur |= (a.mask[(int64_t)y * a.mask_pitch + c0 + k] ? 1u : 0u) << k;
        }
        if (y >= Y0 && y < Y1) {
#pragma unroll
            for (int k = 0; k < 4; k++)
                if (((outmask & mcur) >> k) & 1u) { lmax = fmaxf(lmax, e[k]); have_max = true; }
        }
        const float el = __shfl_up_sync(0xffffffffu, e[3], 1), er = __shfl_down_sync(0xffffffffu, e[0], 1);
        float m3c[4];
        m3c[0] = fmaxf(fmaxf(el, e[0]), e[1]); m3c[1] = fmaxf(fmaxf(e[0], e[1]), e[2]);
        m3c[2] = fmaxf(fmaxf(e[1], e[2]), e[3]); m3c[3] = fmaxf(fmaxf(e[2], e[3]), er);
        const int yc = y - 1;
        if (yc >= max(Y0, 1) && yc < Y1 && yc <= H - 2) {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const float v = eprev[k];
                if ((((candmask & mprev) >> k) & 1u) && v > thr_lb && v == fmaxf(fmaxf(m3a[k], m3b[k]), m3c[k])) {
                    const unsigned long long key = ((unsigned long long)enc_f32(v) << 32) | (uint32_t)(yc * W + c0 + k);
                    const int pos = atomicAdd(scount, 1);
                    if (pos < EN_CB) cbuf[pos] = key;
                    else {
                        const unsigned g = atomicAdd(&a.cnt->ncand, 1u);
                        if (g < a.cap) a.keys[g] = key;
                    }
                }
            }
        }
#pragma unroll
        for (int k = 0; k < 4; k++) { m3a[k] = m3b[k]; m3b[k] = m3c[k]; eprev[k] = e[k]; }
        mprev = mcur;
        if ((y & 7) == 7) {
            __syncwarp();
            if (*reinterpret_cast<volatile int *>(scount) >= EN_CB / 2) flush();
            if ((y & 31) == 31) {
                float wm = lmax;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) wm = fmaxf(wm, __shfl_xor_sync(0xffffffffu, wm, o));
                if (wm > 0.f) thr_lb = fmaxf(thr_lb, (float)((double)wm * a.quality));
            }
        }
    }
    flush();
    uint32_t lbits = have_max ? enc_f32(lmax) : 0u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lbits = max(lbits, __shfl_xor_sync(0xffffffffu, lbits, o));
    if (lane == 0 && lbits) atomicMax(&a.cnt->maxbits, lbits);
}

template <int G, bool MASK, bool HARRIS>
__global__ void __launch_bounds__(EN_WARPS * 32, EN_AP_MIN_CTAS)
eig_nms_ap_kernel(const __grid_constant__ EigNmsArgs a)
{
    extern __shared__ __align__(16) int en_smem[];
    pdl_launch_dependents();
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int job = blockIdx.x * EN_WARPS + wib;
    if (job >= a.njobs) return;
    int *wsm = en_smem + (size_t)wib * a.warp_smem_ints;
    const int nbj = a.nborder * a.chunks_border;                  // job split of eig_nms_kernel
    if (job < nbj) {
        const int sb = job % a.nborder, chunk = job / a.nborder;
        const int strip = a.nborder == a.nstrips ? sb : (sb == 0 ? 0 : a.first_right + sb - 1);
        const int Y0 = chunk * a.rows_border;
        eig_nms_ap_job<G, MASK, true, HARRIS>(a, strip, Y0, min(a.H, Y0 + a.rows_border), wsm, lane);
    } else {
        const int j = job - nbj, nfast = a.nstrips - a.nborder;
        const int strip = 1 + j % nfast, chunk = j / nfast;
        const int Y0 = chunk * a.rows_fast;
        eig_nms_ap_job<G, MASK, false, HARRIS>(a, strip, Y0, min(a.H, Y0 + a.rows_fast), wsm, lane);
    }
}

template <int G, bool MASK, bool HARRIS>
static int launch_eig_nms_ap_kernel(const EigNmsArgs &a, size_t smem, int blocks, cudaStream_t st)
{
    if (smem > 48 * 1024) IBT_CUDA_TRY(cudaFuncSetAttribute(eig_nms_ap_kernel<G, MASK, HARRIS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    eig_nms_ap_kernel<G, MASK, HARRIS><<<blocks, EN_WARPS * 32, smem, st>>>(a);
    return check_launch("eig_nms_ap_kernel");
}

template <int G>
static int launch_eig_nms_ap(const EigNmsArgs &a, int harris, cudaStream_t st)
{
    const size_t smem = (size_t)a.warp_smem_ints * 4 * EN_WARPS;
    const int blocks = (a.njobs + EN_WARPS - 1) / EN_WARPS;
    if (a.mask) return harris ? launch_eig_nms_ap_kernel<G, true, true>(a, smem, blocks, st) : launch_eig_nms_ap_kernel<G, true, false>(a, smem, blocks, st);
    return harris ? launch_eig_nms_ap_kernel<G, false, true>(a, smem, blocks, st) : launch_eig_nms_ap_kernel<G, false, false>(a, smem, blocks, st);
}

static int launch_eig_nms(const uint8_t *gray, int H, int W, int64_t pitch, int bs, int ksize, int harris, double harris_k,
                          const uint8_t *mask, int64_t mask_pitch, double quality, GfttCounters *cnt, unsigned long long *keys, uint32_t cap, cudaStream_t st)
{
    if (bs < 1 || bs > MAX_BLOCK || !ap_supported(ksize)) return IBT_E_INVALID;
    EigNmsArgs a;
    a.img = gray; a.H = H; a.W = W; a.pitch = pitch; a.mask = mask; a.mask_pitch = mask_pitch; a.bs = bs;
    const float scale = ap_scale(ksize, bs);                      // OpenCV's Sobel scale (SURVEY A.6 step 1)
    a.s2 = (double)scale * (double)scale; a.s2h = a.s2 * 0.5;     // the halving of a and c folded in (exact: power of two)
    a.quality = quality; a.cnt = cnt; a.keys = keys; a.cap = cap;
    a.harris_k = (float)harris_k;
    // strip geometry: lane 0's first column is `left` columns before the strip (Sobel radius + window reach + NMS halo, rounded
    // to words); a warp owns `outw` of its 128 support columns
    const int half = bs / 2;                                      // window offsets [-half, bs - 1 - half]
    const int srad = ap_taps(ksize) / 2;                          // Sobel radius
    a.left = (srad + 1 + half + 3) & ~3;
    a.outw = (128 - srad - 1 - a.left - (bs - 1 - half)) & ~3;
    a.nstrips = (W + a.outw - 1) / a.outw;
    a.word_ok = (reinterpret_cast<uintptr_t>(gray) % 4 == 0) && (pitch % 4 == 0);
    // strips whose 128 support columns are all real pixels take the word-load path: 1 <= strip < first_right
    int first_right = a.nstrips;
    while (first_right > 1 && (first_right - 1) * a.outw - a.left + EN_COLS > W) first_right--;
    if (!a.word_ok || first_right <= 1) { a.nborder = a.nstrips; first_right = a.nstrips; }
    else a.nborder = 1 + (a.nstrips - first_right);
    a.first_right = first_right;
    // eig_nms_ap_kernel: (sx, sy) as two ints per ring entry, int64 row buffer
    a.warp_smem_ints = ksize == 3 ? bs * EN_COLS + EN_CB * 2 + 4 + (EN_PAD + EN_COLS + EN_PAD)
                                  : bs * 2 * EN_COLS + EN_CB * 2 + 4 + 2 * (EN_PAD + EN_COLS + EN_PAD);
    // rows per job: one wave of warps over the GPU (warm-up costs bs + 2 rows per job), at least 32 rows (8 for border strips)
    int wps = (int)((227 * 1024) / ((size_t)a.warp_smem_ints * 4 * EN_WARPS + 1024)) * EN_WARPS;       // resident warps per SM
    if (wps < 1) wps = 1;
    const int min_ctas = ksize == 3 ? EN_MIN_CTAS : EN_AP_MIN_CTAS;
    if (wps > min_ctas * EN_WARPS) wps = min_ctas * EN_WARPS;     // register budget (launch bounds)
    const int nfast = a.nstrips - a.nborder;
    const int weight = nfast + EN_BORDER_SPLIT * a.nborder;       // jobs per row chunk, border strips count EN_BORDER_SPLIT times
    int chunks = (kNumSMs * wps) / weight;
    if (chunks < 1) chunks = 1;
    int rows = (H + chunks - 1) / chunks;
    if (rows < 32) rows = 32;
    a.rows_fast = rows;
    a.rows_border = (rows + EN_BORDER_SPLIT - 1) / EN_BORDER_SPLIT;
    if (a.rows_border < 8) a.rows_border = 8;
    a.chunks_border = (H + a.rows_border - 1) / a.rows_border;
    a.njobs = a.nborder * a.chunks_border + nfast * ((H + rows - 1) / rows);
    // cv2's useHarrisDetector=True (never set by the reference): the response formula changes, nothing else; it takes the
    // runtime-blockSize instantiation whatever the block size
    switch (ksize) {
    case -1: return launch_eig_nms_ap<-1>(a, harris, st);
    case 1: return launch_eig_nms_ap<1>(a, harris, st);
    case 5: return launch_eig_nms_ap<5>(a, harris, st);
    case 7: return launch_eig_nms_ap<7>(a, harris, st);
    default: break;
    }
    if (harris) return launch_eig_nms_bs<0, true>(a, st);
    if (bs == 10) return launch_eig_nms_bs<10>(a, st);
    if (bs == 3) return launch_eig_nms_bs<3>(a, st);
    return launch_eig_nms_bs<0>(a, st);
}

// ---------------------------------------------------------------------------------------------
// float32 images (cv2 takes CV_8UC1 and CV_32FC1): eig_f32_kernel, one body for every aperture, both responses, the fused
// K2a (raw 3x3 maxima as keys for K2b) and the map hooks (MAP: the response map is written instead).  eig_nms_ap_job's warp /
// strip structure, with OpenCV's CV_32F front end: Sobel / Scharr in float with the scale 1 / (sden * blockSize) (no 255) on
// the smoothing taps (cv2's Sobel scales the smoothing kernel; taps rounded to float as its float kernels are), the
// derivative taps of a row first, then the column taps; float products; window sums in double; the float response.
//   - Inner strips load four floats per lane (16 bytes: image pointer and pitch multiples of 16), border strips (and every
//     strip of a less aligned image) gather.  Zero taps are skipped, so a NaN / inf pixel reaches the pixels cv2's does.
//   - The window sums are not cv2's running sums: each pixel adds its bs x bs products in a fixed order (rows of a column
//     first, then the columns), so its value depends on its window only -- the map hooks and goodFeaturesToTrack compute the
//     same bits, whatever the job split.  cv2's running double sums differ from these by rounding (bound in tests/f32_cases.py).
//   - A non-finite response (a NaN / inf pixel, or products beyond float range) sets GfttCounters.error to IBT_E_UNSUPPORTED:
//     goodFeaturesToTrack refuses the image rather than return corners derived from it.  The map hooks write NaN / inf.
struct EigF32Args {
    EigNmsArgs n;             // geometry, mask, counters and keys of the fused kernel (n.img unused)
    const float *img; int64_t pitch_f;
    float ss[7];              // smoothing taps * scale, rounded to float (the taps of the Sobel's smoothing direction)
    float *map; int64_t map_pitch_f;     // MAP instantiations
};

template <int G>
__device__ __forceinline__ void f32_taps_vec(float4 w4, const float *ss, float *hd, float *hs)
{
    constexpr int KT = ap_taps(G), R = KT / 2;
    const float w[4] = {w4.x, w4.y, w4.z, w4.w};
    float b[4 + 2 * R];                                            // columns c0 - R .. c0 + 3 + R (neighbour lanes' floats)
#pragma unroll
    for (int i = 0; i < 4 + 2 * R; i++) {
        const int rel = i - R;
        const float v = w[(rel + 4) & 3];
        b[i] = rel < 0 ? __shfl_up_sync(0xffffffffu, v, 1) : rel < 4 ? v : __shfl_down_sync(0xffffffffu, v, 1);
    }
#pragma unroll
    for (int k = 0; k < 4; k++) {
        float d = 0.f, s = 0.f;
#pragma unroll
        for (int j = 0; j < KT; j++) {
            if (ap_d(G, j) != 0) d = __fadd_rn(d, __fmul_rn((float)ap_d(G, j), b[k + j]));
            if (ap_s(G, j) != 0) s = __fadd_rn(s, __fmul_rn(ss[j], b[k + j]));
        }
        hd[k] = d; hs[k] = s;
    }
}

template <int G, bool MASK, bool BORDER, bool HARRIS, bool MAP>
__device__ __forceinline__ void eig_f32_job(const EigF32Args &f, int strip, int Y0, int Y1, int *wsm, int lane)
{
    constexpr int KT = ap_taps(G), R = KT / 2;
    const EigNmsArgs &a = f.n;
    const int bs = a.bs;
    const int a0 = -(bs / 2);
    const int H = a.H, W = a.W;
    const int ox0 = strip * a.outw;
    const int c0 = ox0 - a.left + 4 * lane;
    const int ey0 = max(0, Y0 - 1), ey1 = min(H - 1, Y1);
    float *ring = reinterpret_cast<float *>(wsm);                 // [bs][128][2]: (dx, dy) of the last bs product rows
    unsigned long long *cbuf = reinterpret_cast<unsigned long long *>(wsm + bs * 2 * EN_COLS);
    int *scount = reinterpret_cast<int *>(cbuf + EN_CB);
    double *rowbuf = reinterpret_cast<double *>(scount + 4);      // [EN_PAD + 128 + EN_PAD]
    float ss[KT];
#pragma unroll
    for (int j = 0; j < KT; j++) ss[j] = f.ss[j];
    unsigned outmask = 0, candmask = 0;
    int cx[4][KT];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int c = c0 + k;
        const bool own = c >= ox0 && c < ox0 + a.outw && c < W;
        if (own) outmask |= 1u << k;
        if (own && c >= 1 && c <= W - 2) candmask |= 1u << k;
        const int pc = r101(c, W);
#pragma unroll
        for (int j = 0; j < KT; j++) cx[k][j] = BORDER ? r101(pc + j - R, W) : 0;
    }
    if (!MAP && lane == 0) *scount = 0;
    __syncwarp();
    float m3a[4], m3b[4], eprev[4];
#pragma unroll
    for (int k = 0; k < 4; k++) { m3a[k] = m3b[k] = -FLT_MAX; eprev[k] = 0.f; }
    unsigned mprev = 0;
    float lmax = -FLT_MAX;
    bool have_max = false, finite = true;
    float thr_lb = 0.f;
    if (!MAP) {
        const uint32_t mb = *reinterpret_cast<volatile const uint32_t *>(&a.cnt->maxbits);
        if (mb) thr_lb = fmaxf(0.f, (float)((double)dec_f32(mb) * a.quality));
    }
    auto flush = [&]() {
        __syncwarp();
        const int ncb = min(*reinterpret_cast<volatile int *>(scount), EN_CB);
        unsigned base = 0;
        if (lane == 0 && ncb) base = atomicAdd(&a.cnt->ncand, (unsigned)ncb);
        base = __shfl_sync(0xffffffffu, base, 0);
        for (int i = lane; i < ncb; i += 32)
            if (base + i < a.cap) a.keys[base + i] = cbuf[i];
        __syncwarp();
        if (lane == 0) *scount = 0;
        __syncwarp();
    };
    auto row_taps = [&](const float *row, float *hd, float *hs) {
        if (BORDER) {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                float d = 0.f, s = 0.f;
#pragma unroll
                for (int j = 0; j < KT; j++) {
                    if (ap_d(G, j) == 0 && ap_s(G, j) == 0) continue;
                    const float v = __ldg(row + cx[k][j]);
                    if (ap_d(G, j) != 0) d = __fadd_rn(d, __fmul_rn((float)ap_d(G, j), v));
                    if (ap_s(G, j) != 0) s = __fadd_rn(s, __fmul_rn(ss[j], v));
                }
                hd[k] = d; hs[k] = s;
            }
        } else {
            f32_taps_vec<G>(__ldg(reinterpret_cast<const float4 *>(row + c0)), ss, hd, hs);
        }
    };
    // window sum over columns [x + a0, x + a0 + bs) of a double plane held as 4 values per lane, columns in order
    auto hbox = [&](const double *v, double *out) {
        __syncwarp();
        reinterpret_cast<double2 *>(rowbuf + EN_PAD + 4 * lane)[0] = make_double2(v[0], v[1]);
        reinterpret_cast<double2 *>(rowbuf + EN_PAD + 4 * lane)[1] = make_double2(v[2], v[3]);
        __syncwarp();
        const double *p = rowbuf + EN_PAD + 4 * lane + a0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            double s = 0.0;
            for (int j = 0; j < bs; j++) s = __dadd_rn(s, p[k + j]);
            out[k] = s;
        }
    };
    const int p_first = ey0 + a0, p_last = ey1 + a0 + bs - 1;
    int slot = 0;
    float hd[KT][4], hs[KT][4];
    bool have = false;
    for (int p = p_first; p <= p_last; p++) {
        if (have && p + R <= H - 1) {
#pragma unroll
            for (int i = 0; i + 1 < KT; i++)
#pragma unroll
                for (int k = 0; k < 4; k++) { hd[i][k] = hd[i + 1][k]; hs[i][k] = hs[i + 1][k]; }
            row_taps(f.img + (int64_t)(p + R) * f.pitch_f, hd[KT - 1], hs[KT - 1]);
        } else {
            const int rp = r101(p, H);
#pragma unroll
            for (int i = 0; i < KT; i++) row_taps(f.img + (int64_t)r101(rp + i - R, H) * f.pitch_f, hd[i], hs[i]);
        }
        have = p - R >= 0 && p + R <= H - 1;
        float dx[4], dy[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            float x = 0.f, y = 0.f;
#pragma unroll
            for (int i = 0; i < KT; i++) {
                if (ap_s(G, i) != 0) x = __fadd_rn(x, __fmul_rn(ss[i], hd[i][k]));
                if (ap_d(G, i) != 0) y = __fadd_rn(y, __fmul_rn((float)ap_d(G, i), hs[i][k]));
            }
            dx[k] = x; dy[k] = y;
        }
        float4 *rg = reinterpret_cast<float4 *>(ring + slot * 2 * EN_COLS) + 2 * lane;
        rg[0] = make_float4(dx[0], dy[0], dx[1], dy[1]);
        rg[1] = make_float4(dx[2], dy[2], dx[3], dy[3]);
        slot = slot + 1 == bs ? 0 : slot + 1;             // now the oldest row of the window
        const int y = p - a0 - bs + 1;
        if (y < ey0) continue;
        // ---- vertical window sums: the bs products of each column, top to bottom, in double ---------------------------
        double vxx[4] = {0.0, 0.0, 0.0, 0.0}, vxy[4] = {0.0, 0.0, 0.0, 0.0}, vyy[4] = {0.0, 0.0, 0.0, 0.0};
        int s = slot;
        for (int i = 0; i < bs; i++) {
            const float4 *q = reinterpret_cast<const float4 *>(ring + s * 2 * EN_COLS) + 2 * lane;
            const float4 o0 = q[0], o1 = q[1];
            const float ox[4] = {o0.x, o0.z, o1.x, o1.z}, oy[4] = {o0.y, o0.w, o1.y, o1.w};
#pragma unroll
            for (int k = 0; k < 4; k++) {
                vxx[k] = __dadd_rn(vxx[k], (double)__fmul_rn(ox[k], ox[k]));
                vxy[k] = __dadd_rn(vxy[k], (double)__fmul_rn(ox[k], oy[k]));
                vyy[k] = __dadd_rn(vyy[k], (double)__fmul_rn(oy[k], oy[k]));
            }
            s = s + 1 == bs ? 0 : s + 1;
        }
        double bxx[4], bxy[4], byy[4];
        hbox(vxx, bxx); hbox(vxy, bxy); hbox(vyy, byy);
        float e[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (HARRIS) {                                 // cv2.cornerHarris: (a*c - b*b) - k*((a + c)*(a + c)), float, unfused
                const float fa = (float)bxx[k], fb = (float)bxy[k], fc = (float)byy[k];
                const float tr = __fadd_rn(fa, fc);
                e[k] = __fsub_rn(__fsub_rn(__fmul_rn(fa, fc), __fmul_rn(fb, fb)), __fmul_rn(a.harris_k, __fmul_rn(tr, tr)));
            } else {
                const float fa = __fmul_rn((float)bxx[k], 0.5f), fb = (float)bxy[k], fc = __fmul_rn((float)byy[k], 0.5f);
                const float d = __fsub_rn(fa, fc);
                e[k] = __fsub_rn(__fadd_rn(fa, fc), __fsqrt_rn(__fadd_rn(__fmul_rn(d, d), __fmul_rn(fb, fb))));
            }
        }
        if (MAP) {
            if (y >= Y0 && y < Y1) {
#pragma unroll
                for (int k = 0; k < 4; k++)
                    if ((outmask >> k) & 1u) f.map[(int64_t)y * f.map_pitch_f + c0 + k] = e[k];
            }
            continue;
        }
        // ---- masked maximum, 3x3 raw maxima of the previous row, candidate buffer: as eig_nms_job ----------------------------
        unsigned mcur = 0xfu;
        if (MASK) {
            mcur = 0;
#pragma unroll
            for (int k = 0; k < 4; k++)
                if ((outmask >> k) & 1u) mcur |= (a.mask[(int64_t)y * a.mask_pitch + c0 + k] ? 1u : 0u) << k;
        }
        if (y >= Y0 && y < Y1) {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                if ((outmask >> k) & 1u) finite = finite && isfinite(e[k]);
                if (((outmask & mcur) >> k) & 1u) { lmax = fmaxf(lmax, e[k]); have_max = true; }
            }
        }
        const float el = __shfl_up_sync(0xffffffffu, e[3], 1), er = __shfl_down_sync(0xffffffffu, e[0], 1);
        float m3c[4];
        m3c[0] = fmaxf(fmaxf(el, e[0]), e[1]); m3c[1] = fmaxf(fmaxf(e[0], e[1]), e[2]);
        m3c[2] = fmaxf(fmaxf(e[1], e[2]), e[3]); m3c[3] = fmaxf(fmaxf(e[2], e[3]), er);
        const int yc = y - 1;
        if (yc >= max(Y0, 1) && yc < Y1 && yc <= H - 2) {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const float v = eprev[k];
                if ((((candmask & mprev) >> k) & 1u) && v > thr_lb && v == fmaxf(fmaxf(m3a[k], m3b[k]), m3c[k])) {
                    const unsigned long long key = ((unsigned long long)enc_f32(v) << 32) | (uint32_t)(yc * W + c0 + k);
                    const int pos = atomicAdd(scount, 1);
                    if (pos < EN_CB) cbuf[pos] = key;
                    else {
                        const unsigned g = atomicAdd(&a.cnt->ncand, 1u);
                        if (g < a.cap) a.keys[g] = key;
                    }
                }
            }
        }
#pragma unroll
        for (int k = 0; k < 4; k++) { m3a[k] = m3b[k]; m3b[k] = m3c[k]; eprev[k] = e[k]; }
        mprev = mcur;
        if ((y & 7) == 7) {
            __syncwarp();
            if (*reinterpret_cast<volatile int *>(scount) >= EN_CB / 2) flush();
            if ((y & 31) == 31) {
                float wm = lmax;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) wm = fmaxf(wm, __shfl_xor_sync(0xffffffffu, wm, o));
                if (wm > 0.f) thr_lb = fmaxf(thr_lb, (float)((double)wm * a.quality));
            }
        }
    }
    if (MAP) return;
    flush();
    uint32_t lbits = have_max ? enc_f32(lmax) : 0u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lbits = max(lbits, __shfl_xor_sync(0xffffffffu, lbits, o));
    if (lane == 0 && lbits) atomicMax(&a.cnt->maxbits, lbits);
    if (!__all_sync(0xffffffffu, finite) && lane == 0) atomicCAS(&a.cnt->error, 0, IBT_E_UNSUPPORTED);
}

template <int G, bool MASK, bool HARRIS, bool MAP>
__global__ void __launch_bounds__(EN_WARPS * 32, EN_AP_MIN_CTAS)
eig_f32_kernel(const __grid_constant__ EigF32Args f)
{
    extern __shared__ __align__(16) int en_smem[];
    if (!MAP) pdl_launch_dependents();
    const EigNmsArgs &a = f.n;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int job = blockIdx.x * EN_WARPS + wib;
    if (job >= a.njobs) return;
    int *wsm = en_smem + (size_t)wib * a.warp_smem_ints;
    const int nbj = a.nborder * a.chunks_border;                  // job split of eig_nms_kernel
    if (job < nbj) {
        const int sb = job % a.nborder, chunk = job / a.nborder;
        const int strip = a.nborder == a.nstrips ? sb : (sb == 0 ? 0 : a.first_right + sb - 1);
        const int Y0 = chunk * a.rows_border;
        eig_f32_job<G, MASK, true, HARRIS, MAP>(f, strip, Y0, min(a.H, Y0 + a.rows_border), wsm, lane);
    } else {
        const int j = job - nbj, nfast = a.nstrips - a.nborder;
        const int strip = 1 + j % nfast, chunk = j / nfast;
        const int Y0 = chunk * a.rows_fast;
        eig_f32_job<G, MASK, false, HARRIS, MAP>(f, strip, Y0, min(a.H, Y0 + a.rows_fast), wsm, lane);
    }
}

template <int G, bool MASK, bool HARRIS, bool MAP>
static int launch_eig_f32_kernel(const EigF32Args &f, cudaStream_t st)
{
    const size_t smem = (size_t)f.n.warp_smem_ints * 4 * EN_WARPS;
    const int blocks = (f.n.njobs + EN_WARPS - 1) / EN_WARPS;
    if (smem > 48 * 1024) IBT_CUDA_TRY(cudaFuncSetAttribute(eig_f32_kernel<G, MASK, HARRIS, MAP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    eig_f32_kernel<G, MASK, HARRIS, MAP><<<blocks, EN_WARPS * 32, smem, st>>>(f);
    return check_launch("eig_f32_kernel");
}

template <int G>
static int launch_eig_f32_g(const EigF32Args &f, int harris, int map, cudaStream_t st)
{
    if (map) return harris ? launch_eig_f32_kernel<G, false, true, true>(f, st) : launch_eig_f32_kernel<G, false, false, true>(f, st);
    if (f.n.mask) return harris ? launch_eig_f32_kernel<G, true, true, false>(f, st) : launch_eig_f32_kernel<G, true, false, false>(f, st);
    return harris ? launch_eig_f32_kernel<G, false, true, false>(f, st) : launch_eig_f32_kernel<G, false, false, false>(f, st);
}

static bool f32_image_ok(const float *img, int H, int W, int64_t pitch_bytes)
{
    return img && H > 0 && W > 0 && reinterpret_cast<uintptr_t>(img) % 4 == 0 && pitch_bytes % 4 == 0 &&
           pitch_bytes >= (int64_t)W * 4;
}

// map hooks (map != nullptr: mask / counters unused) and the fused K2a of goodFeaturesToTrack on a float32 image
static int launch_eig_f32(const float *img, int H, int W, int64_t pitch_bytes, int bs, int ksize, int harris, double harris_k,
                          float *map, int64_t map_pitch_bytes, const uint8_t *mask, int64_t mask_pitch, double quality,
                          GfttCounters *cnt, unsigned long long *keys, uint32_t cap, cudaStream_t st)
{
    if (bs < 1 || bs > MAX_BLOCK || !ap_supported(ksize) || !f32_image_ok(img, H, W, pitch_bytes) || !(harris_k == harris_k))
        return IBT_E_INVALID;
    if (map && (map_pitch_bytes % 4 != 0 || map_pitch_bytes < (int64_t)W * 4)) return IBT_E_INVALID;
    EigF32Args f;
    memset(&f, 0, sizeof(f));
    EigNmsArgs &a = f.n;
    a.H = H; a.W = W; a.mask = mask; a.mask_pitch = mask_pitch; a.bs = bs;
    a.quality = quality; a.cnt = cnt; a.keys = keys; a.cap = cap;
    a.harris_k = (float)harris_k;
    f.img = img; f.pitch_f = pitch_bytes / 4;
    f.map = map; f.map_pitch_f = map_pitch_bytes / 4;
    const double sden = ksize == -1 ? 8.0 : (double)(1 << ((ksize > 0 ? ksize : 3) - 1));
    const double scale = 1.0 / (sden * bs);                       // cv2's CV_32F scale: no factor 255
    for (int j = 0; j < ap_taps(ksize); j++) f.ss[j] = (float)(ap_s(ksize, j) * scale);
    // strip geometry of launch_eig_nms; 16-byte loads on the inner strips
    const int half = bs / 2;
    const int srad = ap_taps(ksize) / 2;
    a.left = (srad + 1 + half + 3) & ~3;
    a.outw = (128 - srad - 1 - a.left - (bs - 1 - half)) & ~3;
    a.nstrips = (W + a.outw - 1) / a.outw;
    a.word_ok = (reinterpret_cast<uintptr_t>(img) % 16 == 0) && (pitch_bytes % 16 == 0);
    int first_right = a.nstrips;
    while (first_right > 1 && (first_right - 1) * a.outw - a.left + EN_COLS > W) first_right--;
    if (!a.word_ok || first_right <= 1) { a.nborder = a.nstrips; first_right = a.nstrips; }
    else a.nborder = 1 + (a.nstrips - first_right);
    a.first_right = first_right;
    a.warp_smem_ints = bs * 2 * EN_COLS + EN_CB * 2 + 4 + 2 * (EN_PAD + EN_COLS + EN_PAD);
    int wps = (int)((227 * 1024) / ((size_t)a.warp_smem_ints * 4 * EN_WARPS + 1024)) * EN_WARPS;
    if (wps < 1) wps = 1;
    if (wps > EN_AP_MIN_CTAS * EN_WARPS) wps = EN_AP_MIN_CTAS * EN_WARPS;
    const int nfast = a.nstrips - a.nborder;
    const int weight = nfast + EN_BORDER_SPLIT * a.nborder;
    int chunks = (kNumSMs * wps) / weight;
    if (chunks < 1) chunks = 1;
    int rows = (H + chunks - 1) / chunks;
    if (rows < 32) rows = 32;
    a.rows_fast = rows;
    a.rows_border = (rows + EN_BORDER_SPLIT - 1) / EN_BORDER_SPLIT;
    if (a.rows_border < 8) a.rows_border = 8;
    a.chunks_border = (H + a.rows_border - 1) / a.rows_border;
    a.njobs = a.nborder * a.chunks_border + nfast * ((H + rows - 1) / rows);
    const int m = map ? 1 : 0;
    switch (ksize) {
    case -1: return launch_eig_f32_g<-1>(f, harris, m, st);
    case 1: return launch_eig_f32_g<1>(f, harris, m, st);
    case 3: return launch_eig_f32_g<3>(f, harris, m, st);
    case 5: return launch_eig_f32_g<5>(f, harris, m, st);
    default: return launch_eig_f32_g<7>(f, harris, m, st);
    }
}

// ---------------------------------------------------------------------------------------------
// K2b: the whole selection in ONE persistent launch.  sorted[r] = ~key of rank r (rank 0 = strongest).
constexpr int SEL_THREADS = 256;
constexpr int SEL_CTAS_PER_SM = 2;                   // 2 x 256 threads x 128 registers fill an SM: the grid is kNumSMs * 2, all resident
constexpr int SEL_WARPS = SEL_THREADS / 32;
constexpr int SEL_STEPS = 4, SEL_TILE = SEL_WARPS * SEL_STEPS * 32, SEL_TILE_SHIFT = 10;   // 1024 keys per sort tile: ~80 tiles for 81 k keys
constexpr uint32_t CELL_END = 0xffffffffu;

struct SelArgs {
    GfttCounters *cnt;
    unsigned long long *keys0, *keys1, *keys2;     // candidates (kept), ping-pong buffers of the sort
    uint32_t cap;
    uint32_t *hist3;                               // 3 x [256][ntu] digit counts per destination tile (sort passes, rotating)
    uint32_t *pos, *head, *next, *blockcnt;        // positions by rank; cell lists (head per cell, next per rank); accepted per 256 ranks
    uint8_t *state;
    int H, W, maxCorners, cull, cell, gw, gh;
    uint32_t ncells, limit;
    double quality;
    float md2;
    float *out_xy;
    int *out_count;                                // device
};

// all CTAs of the launch are resident (grid <= SM count): a monotone counter is a barrier
__device__ __forceinline__ void grid_barrier(uint32_t *bar, uint32_t &target)
{
    __syncthreads();
    if (threadIdx.x == 0) {
        target += gridDim.x;
        __threadfence();
        atomicAdd(bar, 1u);
        unsigned spins = 0;
        while (*reinterpret_cast<volatile uint32_t *>(bar) < target)
            if (++spins > (1u << 28)) __trap();                    // a lost CTA must fail loudly, not hang the GPU
        __threadfence();
    }
    __syncthreads();
}

// exclusive scan of v[0..len) (shared memory, len <= 4096) by the 256 threads of the CTA; returns the total
__device__ __forceinline__ uint32_t block_scan_excl(uint32_t *v, int len, uint32_t *wtot /* [9] shared */)
{
    const int per = (len + SEL_THREADS - 1) / SEL_THREADS;
    const int i0 = threadIdx.x * per;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t sum = 0;
    for (int i = i0; i < min(len, i0 + per); i++) sum += v[i];
    uint32_t inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
    __syncthreads();
    if (lane == 31) wtot[wid] = inc;
    __syncthreads();
    if (threadIdx.x == 0) { uint32_t run = 0; for (int w = 0; w < 8; w++) { const uint32_t c = wtot[w]; wtot[w] = run; run += c; } wtot[8] = run; }
    __syncthreads();
    uint32_t run = wtot[wid] + inc - sum;
    for (int i = i0; i < min(len, i0 + per); i++) { const uint32_t c = v[i]; v[i] = run; run += c; }
    __syncthreads();
    return wtot[8];
}

// sum of g[0..len) over the CTA (every thread gets it)
__device__ __forceinline__ uint32_t block_sum_global(const uint32_t *g, uint32_t len, uint32_t *wtot)
{
    uint32_t part = 0;
    for (uint32_t t = threadIdx.x; t < len; t += SEL_THREADS) part += __ldcg(&g[t]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) wtot[threadIdx.x >> 5] = part;
    __syncthreads();
    uint32_t tot = 0;
#pragma unroll
    for (int w = 0; w < 8; w++) tot += wtot[w];
    __syncthreads();
    return tot;
}

// digit tables of the sort: [tile / 4][digit][tile % 4] -- one 16-byte load brings four tiles of a digit, a warp's loads coalesce
__device__ __forceinline__ uint32_t hidx(uint32_t digit, uint32_t tile) { return (((tile >> 2) << 8) + digit) * 4 + (tile & 3u); }

// one evaluation of OpenCV's greedy rule for rank r by walking its 3x3 cell neighbourhood: 0 = still blocked, else the state.
// Breadth first: the nine list heads are fetched together, then all nine lists advance one element per step with their
// loads in flight together -- a warp pays one latency chain per list DEPTH, not one per (cell, element) of its 32 lanes.
__device__ __forceinline__ uint8_t cull_walk(const SelArgs &a, volatile const uint8_t *state, uint32_t r, int x, int y,
                                             uint32_t *nb, int &nnb, bool &over, bool gather)
{
    const int cx = x / a.cell, cy = y / a.cell;
    uint32_t q[9];
#pragma unroll
    for (int i = 0; i < 9; i++) {
        const int xx = cx + (i % 3) - 1, yy = cy + (i / 3) - 1;
        q[i] = (xx >= 0 && xx < a.gw && yy >= 0 && yy < a.gh) ? __ldcg(&a.head[yy * a.gw + xx]) : CELL_END;
    }
    bool blocked = false, killed = false;
    for (;;) {
        bool any = false;
        uint32_t qn[9], pq[9];
#pragma unroll
        for (int i = 0; i < 9; i++) {
            qn[i] = CELL_END; pq[i] = 0;
            if (q[i] != CELL_END) { any = true; qn[i] = __ldcg(&a.next[q[i]]); if (q[i] < r) pq[i] = __ldcg(&a.pos[q[i]]); }
        }
        if (!any) break;
        uint8_t sq[9];
        bool hit[9];
#pragma unroll
        for (int i = 0; i < 9; i++) {
            hit[i] = false; sq[i] = ST_REJECTED;
            if (q[i] != CELL_END && q[i] < r) {                               // only stronger candidates matter
                const float dx = (float)(x - (int)(pq[i] & 0xffffu)), dy = (float)(y - (int)(pq[i] >> 16));
                if (dx * dx + dy * dy < a.md2) { hit[i] = true; sq[i] = state[q[i]]; }
            }
        }
#pragma unroll
        for (int i = 0; i < 9; i++) {
            if (hit[i]) {
                if (gather) { if (nnb < 8) nb[nnb++] = q[i]; else over = true; }
                if (sq[i] == ST_ACCEPTED) killed = true;
                else if (sq[i] == ST_UNDECIDED) blocked = true;
            }
            q[i] = qn[i];
        }
    }
    return killed ? ST_REJECTED : (blocked ? ST_UNDECIDED : ST_ACCEPTED);
}

__global__ void __launch_bounds__(SEL_THREADS, SEL_CTAS_PER_SM)
gftt_select_kernel(const __grid_constant__ SelArgs a)
{
    __shared__ uint32_t sh[4096];
    __shared__ uint32_t wcount[SEL_WARPS][256];
    __shared__ uint32_t wtot[9];
    __shared__ uint32_t s_misc[8];
    GfttCounters *cnt = a.cnt;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const uint32_t gtid = blockIdx.x * SEL_THREADS + tid, gsize = gridDim.x * SEL_THREADS;
    uint32_t bar_target = 0;
    pdl_wait();                                           // candidates, maximum and counters are the previous launch's output
    stamp(cnt, 0);
    const uint32_t mb = __ldcg(&cnt->maxbits);
    const uint32_t ncand = __ldcg(&cnt->ncand);
    if (!mb || !ncand || ncand > a.cap) {                 // uniform over the grid: nothing to select (or overflow)
        if (gtid == 0) {
            if (ncand > a.cap) cnt->error = IBT_E_CAPACITY;
            cnt->nout = 0; *a.out_count = 0;
        }
        return;
    }
    const float thr = (float)((double)dec_f32(mb) * a.quality);
    const uint32_t thrbits = enc_f32(thr);                // enc is order preserving: v > thr  <=>  enc(v) > thrbits
    const uint32_t ntu = (((ncand + SEL_TILE - 1) / SEL_TILE) + 3) & ~3u; // tiles of the sort at most, in whole groups of four
    const uint32_t nchunk_u = (ncand + SEL_THREADS - 1) / SEL_THREADS;

    // ---- phase 1: response histogram of the candidates above the threshold; clear the tables of the later phases ---------
    for (int i = tid; i < 4096; i += SEL_THREADS) sh[i] = 0;
    __syncthreads();
    for (uint32_t i = gtid; i < ncand; i += gsize) {
        const uint32_t e = (uint32_t)(__ldcg(&a.keys0[i]) >> 32);
        if (e > thrbits) atomicAdd(&sh[e >> 20], 1u);
    }
    __syncthreads();
    for (int i = tid; i < 4096; i += SEL_THREADS) if (sh[i]) atomicAdd(&cnt->hist[i], sh[i]);
    for (uint32_t i = gtid; i < 3u * 256u * ntu; i += gsize) a.hist3[i] = 0;
    for (uint32_t i = gtid; i < nchunk_u + 1; i += gsize) a.blockcnt[i] = 0;
    if (a.cull) for (uint32_t i = gtid; i < a.ncells; i += gsize) a.head[i] = CELL_END;
    grid_barrier(&cnt->bar, bar_target);
    stamp(cnt, 1);

    // ---- phase 2 (every CTA, redundantly): the response bin that keeps the strongest ~4 * maxCorners candidates ------------
    for (int i = tid; i < 4096; i += SEL_THREADS) sh[i] = __ldcg(&cnt->hist[i]);
    __syncthreads();
    {
        uint32_t lo = 4096, hi = 0;
        for (int i = tid; i < 4096; i += SEL_THREADS) if (sh[i]) { lo = min(lo, (uint32_t)i); hi = max(hi, (uint32_t)i); }
        for (int o = 16; o > 0; o >>= 1) { lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o)); hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o)); }
        if (tid == 0) { s_misc[0] = 4096; s_misc[1] = 0; }
        __syncthreads();
        if (lane == 0) { atomicMin(&s_misc[0], lo); atomicMax(&s_misc[1], hi); }
        __syncthreads();
    }
    const uint32_t lo_bin_all = s_misc[0], hi_bin = s_misc[1];
    // bins in DESCENDING order, so that the exclusive scan gives "candidates in stronger bins"
    for (int i = tid; i < 2048; i += SEL_THREADS) { const uint32_t t = sh[i]; sh[i] = sh[4095 - i]; sh[4095 - i] = t; }
    __syncthreads();
    const uint32_t total = block_scan_excl(sh, 4096, wtot);       // sh[j] = candidates in bins > 4095 - j
    if (total == 0) {                                            // nothing above the threshold (cannot happen: the maximum is)
        if (gtid == 0) { cnt->nout = 0; *a.out_count = 0; }
        return;
    }
    const uint64_t want = a.maxCorners > 0 ? (uint64_t)a.maxCorners * 4 + 1024 : 0;
    uint32_t min_bin = 0;
    bool subset = false;
    if (a.maxCorners > 0 && a.cull && (uint64_t)total > 2 * want) {
        // smallest j with (candidates in bins >= 4095 - j) >= want
        if (tid == 0) s_misc[2] = 4095;
        __syncthreads();
        uint32_t jm = 4095;
        for (int j = tid; j < 4096; j += SEL_THREADS) {
            const uint32_t incl = j == 4095 ? total : sh[j + 1];
            if (incl >= want) jm = min(jm, (uint32_t)j);
        }
        for (int o = 16; o > 0; o >>= 1) jm = min(jm, __shfl_xor_sync(0xffffffffu, jm, o));
        if (lane == 0) atomicMin(&s_misc[2], jm);
        __syncthreads();
        const uint32_t j = s_misc[2];
        const uint32_t b = 4095 - j;
        const uint32_t cum = j == 4095 ? total : sh[j + 1];
        if (b > 0 && cum < total) { min_bin = b; subset = true; }
    }
    __syncthreads();

    uint32_t nacc = 0;
    stamp(cnt, 2);
    for (int attempt = 0; attempt < 2; attempt++) {
        // attempt 0 may rank the strongest candidates only; if culling leaves fewer than maxCorners of them, attempt 1 repeats
        // with every candidate.  The greedy order makes the prefix exact either way: whether a candidate is accepted depends
        // on stronger candidates only.
        const uint32_t lo_bin = max(lo_bin_all, min_bin);
        // sort key = (hi_bound - response bits) << 32 | ~address: ascending order = (response desc, address desc), and only the
        // bytes the selected response range can differ in are sorted
        const uint32_t hi_bound = (hi_bin << 20) | 0xfffffu;
        const uint32_t range = ((hi_bin - lo_bin + 1) << 20) - 1;            // largest possible hi_bound - e
        const int last_pass = range < (1u << 8) ? 4 : range < (1u << 16) ? 5 : range < (1u << 24) ? 6 : 7;
        // ---- select; every kept key also counts its first sort digit for the tile it lands in ------------------------------------
        for (uint32_t i0 = blockIdx.x * SEL_THREADS; i0 < ncand; i0 += gsize) {
            const uint32_t i = i0 + tid;
            unsigned long long k = 0;
            bool keep = false;
            if (i < ncand) { k = __ldcg(&a.keys0[i]); const uint32_t e = (uint32_t)(k >> 32); keep = e > thrbits && (e >> 20) >= min_bin; }
            const uint32_t ballot = __ballot_sync(0xffffffffu, keep);
            if (ballot) {
                uint32_t base = 0;
                if (lane == 0) base = atomicAdd(&cnt->nsel, (uint32_t)__popc(ballot));
                base = __shfl_sync(0xffffffffu, base, 0);
                if (keep) {
                    const uint32_t j = base + __popc(ballot & ((1u << lane) - 1u));
                    const unsigned long long ck = ((unsigned long long)(hi_bound - (uint32_t)(k >> 32)) << 32) | (uint32_t)(~(uint32_t)k);
                    a.keys1[j] = ck;
                    atomicAdd(&a.hist3[hidx((uint32_t)((ck >> 32) & 0xff), j >> SEL_TILE_SHIFT)], 1u);
                }
            }
        }
        grid_barrier(&cnt->bar, bar_target);
        stamp(cnt, 3);
        const uint32_t n = __ldcg(&cnt->nsel);
        const unsigned long long *src = a.keys1;
        unsigned long long *dst = a.keys2;

        // ---- stable LSD radix sort on the response bytes; each pass counts the next pass's digits while it scatters --------
        if (n > 1) {
            const uint32_t ntiles = (n + SEL_TILE - 1) / SEL_TILE;
            for (int p = 4; p <= last_pass; p++) {
                const int shift = 8 * p;
                const uint32_t *hcur = a.hist3 + (size_t)((p - 4) % 3) * 256 * ntu;
                uint32_t *hnext = a.hist3 + (size_t)((p - 3) % 3) * 256 * ntu;
                if (p + 2 <= last_pass) {                                       // the table of pass p+2 was used by pass p-1
                    uint32_t *hz = a.hist3 + (size_t)((p - 2) % 3) * 256 * ntu;
                    for (uint32_t i = gtid; i < 256u * ntu; i += gsize) hz[i] = 0;
                }
                for (uint32_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
                    // thread d: its digit summed over all tiles (-> digit base by an exclusive scan) and over the tiles before this one
                    uint32_t rs = 0, before = 0;
                    const uint4 *hq = reinterpret_cast<const uint4 *>(hcur) + tid;
#pragma unroll 4
                    for (uint32_t g = 0; g < (ntiles + 3) / 4; g++) {
                        const uint4 c = __ldcg(hq + (size_t)g * 256);
                        const uint32_t t0 = 4 * g;
                        rs += c.x + c.y + c.z + c.w;
                        before += (t0 < tile ? c.x : 0) + (t0 + 1 < tile ? c.y : 0) + (t0 + 2 < tile ? c.z : 0) + (t0 + 3 < tile ? c.w : 0);
                    }
                    __syncthreads();
                    sh[tid] = rs;
                    __syncthreads();
                    block_scan_excl(sh, 256, wtot);
                    const uint32_t digit_base = sh[tid];
                    __syncthreads();
                    for (int i = tid; i < SEL_WARPS * 256; i += SEL_THREADS) (&wcount[0][0])[i] = 0;
                    __syncthreads();
                    const uint32_t wbase = tile * SEL_TILE + wid * (SEL_STEPS * 32);
                    unsigned long long k[SEL_STEPS];
                    uint32_t rank[SEL_STEPS];
#pragma unroll
                    for (int s = 0; s < SEL_STEPS; s++) {                       // all loads of the tile in flight together
                        const uint32_t g = wbase + s * 32 + lane;
                        k[s] = g < n ? __ldcg(&src[g]) : 0ull;
                    }
#pragma unroll
                    for (int s = 0; s < SEL_STEPS; s++) {
                        const uint32_t g = wbase + s * 32 + lane;
                        const bool valid = g < n;
                        const uint32_t d = (uint32_t)((k[s] >> shift) & 0xff);
                        const uint32_t vmask = __ballot_sync(0xffffffffu, valid);
                        uint32_t peers = __match_any_sync(0xffffffffu, valid ? d : 0x100u + lane) & vmask;
                        if (!valid) peers = 0;
                        const uint32_t bef = __popc(peers & ((1u << lane) - 1u));
                        uint32_t prev = 0;
                        if (valid) prev = wcount[wid][d];          // all peers read the same value before the leader updates
                        __syncwarp();
                        if (valid && bef == 0) wcount[wid][d] = prev + __popc(peers);
                        __syncwarp();
                        rank[s] = prev + bef;                      // rank within this warp's chunk for digit d
                    }
                    __syncthreads();
                    {
                        uint32_t run = digit_base + before;        // thread d: exclusive prefix over warps + global offset of (digit, tile)
#pragma unroll
                        for (int w = 0; w < SEL_WARPS; w++) { const uint32_t c = wcount[w][tid]; wcount[w][tid] = run; run += c; }
                    }
                    __syncthreads();
#pragma unroll
                    for (int s = 0; s < SEL_STEPS; s++) {
                        const uint32_t g = wbase + s * 32 + lane;
                        if (g < n) {
                            const uint32_t d = (uint32_t)((k[s] >> shift) & 0xff);
                            const uint32_t j = wcount[wid][d] + rank[s];
                            dst[j] = k[s];
                            if (p < last_pass) atomicAdd(&hnext[hidx((uint32_t)((k[s] >> (shift + 8)) & 0xff), j >> SEL_TILE_SHIFT)], 1u);
                        }
                    }
                    __syncthreads();
                }
                grid_barrier(&cnt->bar, bar_target);
                stamp(cnt, p);
                const unsigned long long *t = src; src = dst; dst = const_cast<unsigned long long *>(t);
            }
        }
        // ---- positions by rank, cell lists.  Equal responses kept their arrival order: the first element of a run of equal
        // responses orders the run by address (complemented keys ascending = address descending, OpenCV's tie-break) ------
        {
            unsigned long long *srt = const_cast<unsigned long long *>(src);
            for (uint32_t i = gtid; i < n; i += gsize) {
                const uint32_t v = (uint32_t)(__ldcg(&srt[i]) >> 32);
                if (i > 0 && (uint32_t)(__ldcg(&srt[i - 1]) >> 32) == v) continue;
                uint32_t e = i + 1;
                while (e < n && (uint32_t)(__ldcg(&srt[e]) >> 32) == v) e++;
                for (uint32_t x = i + 1; x < e; x++) {                          // insertion sort of srt[i..e): runs are rare and short
                    const unsigned long long kk = srt[x];
                    uint32_t b = x;
                    while (b > i && srt[b - 1] > kk) { srt[b] = srt[b - 1]; b--; }
                    srt[b] = kk;
                }
                for (uint32_t x = i; x < e; x++) {
                    const uint32_t idx = ~(uint32_t)srt[x];
                    const uint32_t y = idx / a.W, xc = idx - y * a.W;
                    a.pos[x] = xc | (y << 16);
                    a.state[x] = ST_UNDECIDED;
                    if (a.cull) a.next[x] = atomicExch(&a.head[(y / a.cell) * a.gw + xc / a.cell], x);
                }
            }
        }
        grid_barrier(&cnt->bar, bar_target);
        stamp(cnt, 8);
        // ---- culling: decisions are final and monotone, so a thread may read fresh or stale states.  Every thread first collects
        // the stronger conflicting candidates of its ranks (walk of the 3x3 cell lists, once), then polls their states a few
        // times per grid barrier until no rank of the grid is undecided.  Ranks are handed out in rank-ordered batches of two per
        // thread: dependencies point to stronger ranks only, so a batch never waits for a later one -----------------------------
        if (a.cull) {
            volatile uint8_t *state = a.state;
            uint32_t round_no = 0;
            for (uint32_t b0 = 0; b0 < n; b0 += 2 * gsize) {
                uint32_t r[2], nb[2][8];
                int xs[2], ys[2], nnb[2];
                bool over[2], open[2];
#pragma unroll
                for (int j = 0; j < 2; j++) {
                    r[j] = b0 + j * gsize + gtid;
                    open[j] = r[j] < n;
                    nnb[j] = 0; over[j] = false; xs[j] = ys[j] = 0;
                    if (open[j]) {
                        const uint32_t p = __ldcg(&a.pos[r[j]]);
                        xs[j] = (int)(p & 0xffffu); ys[j] = (int)(p >> 16);
                        const uint8_t s = cull_walk(a, state, r[j], xs[j], ys[j], nb[j], nnb[j], over[j], true);
                        if (s != ST_UNDECIDED) {
                            state[r[j]] = s; open[j] = false;
                            if (s == ST_ACCEPTED) atomicAdd(&a.blockcnt[r[j] >> 8], 1u);
                        }
                    }
                }
                for (;;) {
                    for (int it = 0; it < 4 && (open[0] || open[1]); it++) {
#pragma unroll
                        for (int j = 0; j < 2; j++) {
                            if (!open[j]) continue;
                            uint8_t s = ST_ACCEPTED;
                            if (over[j]) {
                                int dummy = 8; bool od = false;
                                s = cull_walk(a, state, r[j], xs[j], ys[j], nb[j], dummy, od, false);
                            } else {
#pragma unroll
                                for (int i = 0; i < 8; i++) {
                                    if (i < nnb[j]) {
                                        const uint8_t sq = state[nb[j][i]];
                                        if (sq == ST_ACCEPTED) s = ST_REJECTED;
                                        else if (sq == ST_UNDECIDED && s != ST_REJECTED) s = ST_UNDECIDED;
                                    }
                                }
                            }
                            if (s != ST_UNDECIDED) {
                                state[r[j]] = s; open[j] = false;
                                if (s == ST_ACCEPTED) atomicAdd(&a.blockcnt[r[j] >> 8], 1u);
                            }
                        }
                    }
                    // anyone still undecided in this batch?  (one counter per round, recycled after 32 rounds)
                    const int left = __syncthreads_count(open[0] || open[1]);
                    if (tid == 0) {
                        if (left) atomicAdd(&cnt->remaining[round_no & 63], (uint32_t)left);
                        if (blockIdx.x == 0) cnt->remaining[(round_no + 32) & 63] = 0;
                    }
                    grid_barrier(&cnt->bar, bar_target);
                    const uint32_t rem = __ldcg(&cnt->remaining[round_no & 63]);
                    round_no++;
                    if (rem == 0) break;
                }
            }
        }
        stamp(cnt, 9);
        // ---- accepted candidates in rank order -> (x, y), first `limit` -------------------------------------------------------
        const uint32_t nchunk = (n + SEL_THREADS - 1) / SEL_THREADS;
        nacc = a.cull ? block_sum_global(a.blockcnt, nchunk, wtot) : n;
        for (uint32_t c = blockIdx.x; c < nchunk; c += gridDim.x) {
            const uint32_t off = a.cull ? block_sum_global(a.blockcnt, c, wtot) : c * SEL_THREADS;
            if (off >= a.limit) continue;                                   // block-uniform
            const uint32_t r = c * SEL_THREADS + tid;
            const bool acc = r < n && (!a.cull || __ldcg(&a.state[r]) == ST_ACCEPTED);
            const uint32_t ballot = __ballot_sync(0xffffffffu, acc);
            __syncthreads();
            if (lane == 0) wtot[wid] = __popc(ballot);
            __syncthreads();
            uint32_t wb = off;
            for (int w = 0; w < wid; w++) wb += wtot[w];
            if (acc) {
                const uint32_t m = wb + __popc(ballot & ((1u << lane) - 1u));
                if (m < a.limit) {
                    const uint32_t p = __ldcg(&a.pos[r]);
                    a.out_xy[2 * m] = (float)(p & 0xffffu);
                    a.out_xy[2 * m + 1] = (float)(p >> 16);
                }
            }
            __syncthreads();
        }
        if (!subset || nacc >= (uint32_t)a.maxCorners) break;          // done (the subset produced a full prefix)
        // ---- too few survivors among the strongest: once more with every candidate above the threshold ---------------------------
        grid_barrier(&cnt->bar, bar_target);                            // everyone has read blockcnt / state
        min_bin = 0; subset = false;
        if (gtid == 0) cnt->nsel = 0;
        for (uint32_t i = gtid; i < 3u * 256u * ntu; i += gsize) a.hist3[i] = 0;
        for (uint32_t i = gtid; i < nchunk_u + 1; i += gsize) a.blockcnt[i] = 0;
        for (uint32_t i = gtid; i < a.ncells; i += gsize) a.head[i] = CELL_END;
        grid_barrier(&cnt->bar, bar_target);
    }
    stamp(cnt, 10);
    if (gtid == 0) {
        uint32_t nout = nacc;
        if (a.maxCorners > 0 && nout > (uint32_t)a.maxCorners) nout = (uint32_t)a.maxCorners;
        if (nout > a.limit) { cnt->error = IBT_E_CAPACITY; }
        cnt->nacc = nacc;
        cnt->nout = nout;
        *a.out_count = (int)nout;
    }
}

// workspace layout
struct GfttLayout {
    size_t off_cnt, off_keys0, off_keys1, off_keys2, off_hist3, off_pos, off_state, off_head, off_next, off_blockcnt, total;
    uint32_t cap, max_sort_blocks, max_cells;
};
static GfttLayout gftt_layout(int H, int W)
{
    GfttLayout L;
    const size_t np = (size_t)H * W;
    auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
    L.cap = (uint32_t)(np / 4 + 4096);                 // isolated 3x3 maxima cannot be denser than 1 in 4 pixels (plateaus can: IBT_E_CAPACITY)
    L.max_sort_blocks = (L.cap + 1024 - 1) / 1024;          // SEL_TILE
    L.max_cells = (uint32_t)np + 1;                    // cell >= 1 pixel
    size_t o = 0;
    L.off_cnt = o; o = up(o + sizeof(GfttCounters));
    L.off_keys0 = o; o = up(o + (size_t)L.cap * 8);
    L.off_keys1 = o; o = up(o + (size_t)L.cap * 8);
    L.off_keys2 = o; o = up(o + (size_t)L.cap * 8);
    L.off_hist3 = o; o = up(o + (size_t)3 * 256 * (L.max_sort_blocks + 4) * 4);
    L.off_pos = o; o = up(o + (size_t)L.cap * 4);
    L.off_state = o; o = up(o + (size_t)L.cap);
    L.off_head = o; o = up(o + (size_t)L.max_cells * 4);
    L.off_next = o; o = up(o + (size_t)L.cap * 4);
    L.off_blockcnt = o; o = up(o + ((size_t)L.cap / 256 + 4) * 4);
    L.total = o;
    return L;
}

// Both launches of goodFeaturesToTrack on `st`; nothing is read back.  count_dev (device int) receives the corner count.
// f32src: `gray` is a float32 image and `pitch` its byte pitch (eig_f32_kernel produces the candidates).
static int gftt_enqueue(const void *gray, int64_t pitch, const uint8_t *mask, int64_t mask_pitch, int H, int W,
                        int maxCorners, double qualityLevel, double minDistance, int blockSize, int ksize, int useHarris, double harris_k,
                        void *workspace, size_t workspace_bytes, float *out_xy, int cap, int *count_dev, cudaStream_t st,
                        bool f32src = false)
{
    if (!gray || !workspace || H < 3 || W < 3 || H > 65535 || W > 65535 || (int64_t)H * W > 0x7fffffffLL ||
        cap < 0 || (cap > 0 && !out_xy) || (mask && mask_pitch < W) || qualityLevel < 0 || minDistance < 0 || minDistance > 1024 ||
        pitch < W || !(harris_k == harris_k) || !ap_supported(ksize) || blockSize < 1 || blockSize > MAX_BLOCK ||
        (f32src && !f32_image_ok(static_cast<const float *>(gray), H, W, pitch)))
        return IBT_E_INVALID;
    const GfttLayout L = gftt_layout(H, W);
    if (workspace_bytes < L.total) return IBT_E_WORKSPACE;
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    GfttCounters *cnt = reinterpret_cast<GfttCounters *>(ws + L.off_cnt);
    IBT_CUDA_TRY(cudaMemsetAsync(cnt, 0, sizeof(GfttCounters), st));
    unsigned long long *keys0 = reinterpret_cast<unsigned long long *>(ws + L.off_keys0);
    int rc = f32src ? launch_eig_f32(static_cast<const float *>(gray), H, W, pitch, blockSize, ksize, useHarris, harris_k, nullptr, 0,
                                     mask, mask_pitch, qualityLevel, cnt, keys0, L.cap, st)
                    : launch_eig_nms(static_cast<const uint8_t *>(gray), H, W, pitch, blockSize, ksize, useHarris, harris_k, mask,
                                     mask_pitch, qualityLevel, cnt, keys0, L.cap, st);
    if (rc) return rc;
    SelArgs a;
    a.cnt = cnt; a.keys0 = keys0;
    a.keys1 = reinterpret_cast<unsigned long long *>(ws + L.off_keys1);
    a.keys2 = reinterpret_cast<unsigned long long *>(ws + L.off_keys2);
    a.cap = L.cap;
    a.hist3 = reinterpret_cast<uint32_t *>(ws + L.off_hist3);
    a.pos = reinterpret_cast<uint32_t *>(ws + L.off_pos);
    a.state = ws + L.off_state;
    a.head = reinterpret_cast<uint32_t *>(ws + L.off_head);
    a.next = reinterpret_cast<uint32_t *>(ws + L.off_next);
    a.blockcnt = reinterpret_cast<uint32_t *>(ws + L.off_blockcnt);
    a.H = H; a.W = W; a.maxCorners = maxCorners;
    a.cull = minDistance >= 1.0 ? 1 : 0;
    a.cell = a.cull ? (int)lrint(minDistance) : 65536;        // no culling: only positions are needed
    a.gw = (W + a.cell - 1) / a.cell; a.gh = (H + a.cell - 1) / a.cell;
    a.ncells = (uint32_t)a.gw * a.gh;
    uint32_t limit = (maxCorners > 0) ? (uint32_t)maxCorners : 0xffffffffu;
    if (limit > (uint32_t)cap) limit = (uint32_t)cap;
    a.limit = limit;
    a.quality = qualityLevel;
    a.md2 = (float)(minDistance * minDistance);
    a.out_xy = out_xy;
    a.out_count = count_dev ? count_dev : reinterpret_cast<int *>(&cnt->pad);
    // every CTA must be resident (the kernel synchronises its grid itself): size the grid from what THIS device can hold
    static std::atomic<int> sel_grid[64];                          // (host threads may race here: they compute the same value)
    int dev_id = 0;
    IBT_CUDA_TRY(cudaGetDevice(&dev_id));
    if (dev_id < 0 || dev_id >= 64) return IBT_E_INVALID;
    int grid = sel_grid[dev_id].load(std::memory_order_relaxed);
    if (!grid) {
        int sms = 0, per_sm = 0;
        IBT_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev_id));
        IBT_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, gftt_select_kernel, SEL_THREADS, 0));
        if (per_sm > SEL_CTAS_PER_SM) per_sm = SEL_CTAS_PER_SM;
        if (sms < 1 || per_sm < 1) return IBT_E_CUDA;
        grid = sms * per_sm;
        sel_grid[dev_id].store(grid, std::memory_order_relaxed);
    }
    IBT_CUDA_TRY(launch_pdl(gftt_select_kernel, dim3(grid), dim3(SEL_THREADS), 0, st, a));
    return check_launch("gftt_select_kernel");
}

} // namespace ibt

IBT_API int ibt_min_eigen_f32(const uint8_t *gray, int H, int W, int64_t pitch, int blockSize, float *eig,
                              int64_t eig_pitch, void *stream)
{
    return ibt::launch_eig(gray, H, W, pitch, blockSize, 0, 0.0, eig, eig_pitch, nullptr, 0, nullptr, static_cast<cudaStream_t>(stream));
}

IBT_API int ibt_min_eigen_ksize_f32(const uint8_t *gray, int H, int W, int64_t pitch, int blockSize, int ksize, float *eig,
                                    int64_t eig_pitch, void *stream)
{
    return ibt::launch_eig_ksize(gray, H, W, pitch, blockSize, ksize, 0, 0.0, eig, eig_pitch, static_cast<cudaStream_t>(stream));
}

IBT_API int ibt_corner_harris_f32(const uint8_t *gray, int H, int W, int64_t pitch, int blockSize, double k, float *dst,
                                  int64_t dst_pitch, void *stream)
{
    if (!(k == k)) return IBT_E_INVALID;
    return ibt::launch_eig(gray, H, W, pitch, blockSize, 1, k, dst, dst_pitch, nullptr, 0, nullptr, static_cast<cudaStream_t>(stream));
}

IBT_API int ibt_corner_harris_ksize_f32(const uint8_t *gray, int H, int W, int64_t pitch, int blockSize, int ksize, double k,
                                        float *dst, int64_t dst_pitch, void *stream)
{
    if (!(k == k)) return IBT_E_INVALID;
    return ibt::launch_eig_ksize(gray, H, W, pitch, blockSize, ksize, 1, k, dst, dst_pitch, static_cast<cudaStream_t>(stream));
}

IBT_API size_t ibt_gftt_workspace_bytes(int H, int W)
{
    if (H <= 0 || W <= 0) return 0;
    return ibt::gftt_layout(H, W).total;
}

IBT_API int ibt_gftt_async_ksize(const uint8_t *gray, int64_t pitch, const uint8_t *mask, int64_t mask_pitch, int H, int W,
                                 int maxCorners, double qualityLevel, double minDistance, int blockSize, int gradientSize,
                                 int useHarrisDetector, double k, void *workspace, size_t workspace_bytes, float *out_xy, int cap,
                                 int *count_dev, void *stream)
{
    if (!count_dev) return IBT_E_INVALID;
    return ibt::gftt_enqueue(gray, pitch, mask, mask_pitch, H, W, maxCorners, qualityLevel, minDistance, blockSize, gradientSize,
                             useHarrisDetector, k, workspace, workspace_bytes, out_xy, cap, count_dev,
                             static_cast<cudaStream_t>(stream));
}

IBT_API int ibt_gftt_async(const uint8_t *gray, int64_t pitch, const uint8_t *mask, int64_t mask_pitch, int H, int W,
                           int maxCorners, double qualityLevel, double minDistance, int blockSize, int useHarrisDetector,
                           double k, void *workspace, size_t workspace_bytes, float *out_xy, int cap, int *count_dev,
                           void *stream)
{
    return ibt_gftt_async_ksize(gray, pitch, mask, mask_pitch, H, W, maxCorners, qualityLevel, minDistance, blockSize, 3,
                                useHarrisDetector, k, workspace, workspace_bytes, out_xy, cap, count_dev, stream);
}

// the synchronous form: both launches, then the one host round trip -- the corner count decides the shapes the caller
// allocates next
static int gftt_sync(const void *img, int64_t pitch, const uint8_t *mask, int64_t mask_pitch, int H, int W, int maxCorners,
                     double qualityLevel, double minDistance, int blockSize, int gradientSize, int useHarrisDetector, double k,
                     void *workspace, size_t workspace_bytes, float *out_xy, int cap, int *out_count, void *stream, bool f32src)
{
    using namespace ibt;
    if (!out_count) return IBT_E_INVALID;
    *out_count = 0;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int rc = gftt_enqueue(img, pitch, mask, mask_pitch, H, W, maxCorners, qualityLevel, minDistance, blockSize, gradientSize,
                          useHarrisDetector, k, workspace, workspace_bytes, out_xy, cap, nullptr, st, f32src);
    if (rc) return rc;
    struct Head { uint32_t maxbits, ncand, nsel, nacc, nout; int32_t error; };
    static thread_local Head *hc = nullptr;                        // page-locked: the copy is a real asynchronous DMA
    if (!hc) IBT_CUDA_TRY(cudaHostAlloc(reinterpret_cast<void **>(&hc), sizeof(Head), cudaHostAllocDefault));
    IBT_CUDA_TRY(cudaMemcpyAsync(hc, workspace, sizeof(Head), cudaMemcpyDeviceToHost, st));
    IBT_CUDA_TRY(cudaStreamSynchronize(st));
    *out_count = (int)hc->nout;
    return hc->error ? hc->error : IBT_OK;
}

IBT_API int ibt_gftt_ksize(const uint8_t *gray, int64_t pitch, const uint8_t *mask, int64_t mask_pitch, int H, int W,
                           int maxCorners, double qualityLevel, double minDistance, int blockSize, int gradientSize,
                           int useHarrisDetector, double k, void *workspace, size_t workspace_bytes, float *out_xy, int cap,
                           int *out_count, void *stream)
{
    return gftt_sync(gray, pitch, mask, mask_pitch, H, W, maxCorners, qualityLevel, minDistance, blockSize, gradientSize,
                     useHarrisDetector, k, workspace, workspace_bytes, out_xy, cap, out_count, stream, false);
}

IBT_API int ibt_gftt_f32src(const float *img, int64_t pitch, const uint8_t *mask, int64_t mask_pitch, int H, int W,
                            int maxCorners, double qualityLevel, double minDistance, int blockSize, int gradientSize,
                            int useHarrisDetector, double k, void *workspace, size_t workspace_bytes, float *out_xy, int cap,
                            int *out_count, void *stream)
{
    return gftt_sync(img, pitch, mask, mask_pitch, H, W, maxCorners, qualityLevel, minDistance, blockSize, gradientSize,
                     useHarrisDetector, k, workspace, workspace_bytes, out_xy, cap, out_count, stream, true);
}

IBT_API int ibt_min_eigen_f32src(const float *img, int H, int W, int64_t pitch, int blockSize, int ksize, float *eig,
                                 int64_t eig_pitch, void *stream)
{
    if (!eig) return IBT_E_INVALID;
    return ibt::launch_eig_f32(img, H, W, pitch, blockSize, ksize, 0, 0.0, eig, eig_pitch, nullptr, 0, 0.0, nullptr, nullptr, 0,
                               static_cast<cudaStream_t>(stream));
}

IBT_API int ibt_corner_harris_f32src(const float *img, int H, int W, int64_t pitch, int blockSize, int ksize, double k,
                                     float *dst, int64_t dst_pitch, void *stream)
{
    if (!dst) return IBT_E_INVALID;
    return ibt::launch_eig_f32(img, H, W, pitch, blockSize, ksize, 1, k, dst, dst_pitch, nullptr, 0, 0.0, nullptr, nullptr, 0,
                               static_cast<cudaStream_t>(stream));
}

IBT_API int ibt_gftt(const uint8_t *gray, int64_t pitch, const uint8_t *mask, int64_t mask_pitch, int H, int W,
                     int maxCorners, double qualityLevel, double minDistance, int blockSize, int useHarrisDetector, double k,
                     void *workspace, size_t workspace_bytes, float *out_xy, int cap, int *out_count, void *stream)
{
    return ibt_gftt_ksize(gray, pitch, mask, mask_pitch, H, W, maxCorners, qualityLevel, minDistance, blockSize, 3,
                          useHarrisDetector, k, workspace, workspace_bytes, out_xy, cap, out_count, stream);
}
