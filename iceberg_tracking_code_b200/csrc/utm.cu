// K4: photo -> UTM ray/plane projection of track vertices (SURVEY.md A.9).  Replaces the per-vertex
// Python calls cam.photocords_cropped_to_uncropped + cam.photo_to_utm at s2_cam_to_utm.py:247-254
// (imports/camtools.py:414-421, 286-332).  fp64 throughout: northing ~6.5e6 m needs it.
// The nine direction cosines are evaluated once on the host (libm, like numpy) and passed by value;
// the reference recomputes them per vertex with identical inputs, so results do not change.
#include "common.cuh"
#include <math.h>

namespace ibt {

struct UtmCam {
    double cl, ct, halfW, halfH, Hc, E0, N0;
    double sX0, sX1, sX2;                  // sigma * X
    double U0, U1, U2, V0, V1, V2;
};

__global__ void __launch_bounds__(256)
photo_to_utm_kernel(const float2 *__restrict__ xy, int64_t n, const __grid_constant__ UtmCam c, double2 *__restrict__ EN)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float2 p = xy[i];
        // same operation order as camtools.py:300-301, 326-330; no FMA contraction (-fmad=false)
        const double xi = ((double)p.x + c.cl) - c.halfW;
        const double yi = ((double)p.y + c.ct) - c.halfH;
        const double den = c.sX2 + xi * c.U2 + yi * c.V2;
        const double tx = c.Hc * (c.sX0 + xi * c.U0 + yi * c.V0) / den + c.E0;
        const double ty = c.Hc * (c.sX1 + xi * c.U1 + yi * c.V1) / den + c.N0;
        EN[i] = make_double2(tx, ty);
    }
}

// s2_cam_to_utm.py:243-343 for one track per thread: project every vertex (fp64), segment velocities u, v (m/s) and speed,
// then the three plausibility criteria.  Python's max() over a list is restated literally (m = first; if x > m: m = x),
// which also reproduces its NaN behaviour (0/0 speeds ratios of motionless tracks).  One divergence, documented: for T == 1
// with max speed above speed_threshold the reference raises (max() of the empty ratio list, s2:337); here the track is kept.
struct VelArgs {
    UtmCam cam;
    const float2 *tracks; int M, T;
    double interval, min_speed, max_speed, max_speedfactor, max_angle, speed_threshold;
    double2 *EN; double2 *uv; double *speed; uint8_t *keep;
};

__device__ __forceinline__ double2 project(const UtmCam &c, float2 p)
{
    const double xi = ((double)p.x + c.cl) - c.halfW;
    const double yi = ((double)p.y + c.ct) - c.halfH;
    const double den = c.sX2 + xi * c.U2 + yi * c.V2;
    return make_double2(c.Hc * (c.sX0 + xi * c.U0 + yi * c.V0) / den + c.E0,
                        c.Hc * (c.sX1 + xi * c.U1 + yi * c.V1) / den + c.N0);
}

// numpy's float64 hypot (s2:286, 328) as glibc >= 2.35 computes it without FMA: Borges, "An Improved Algorithm for
// hypot(a, b)" (arXiv:1904.09481), restated operation for operation (tests/test_libm_restatements.py pins it on the host's
// libm).  It is not correctly rounded, and CUDA's hypot rounds differently, so the speeds written to the hourly files and
// compared with min_speed, max_speed and speed_threshold would differ from numpy's in the last bit.
__device__ __forceinline__ double glibc_hypot_kernel(double ax, double ay)         // ax >= ay >= 0, squares in range
{
    double h = __dsqrt_rn(__dadd_rn(__dmul_rn(ax, ax), __dmul_rn(ay, ay)));
    double t1, t2;
    if (h <= __dmul_rn(2.0, ay)) {
        const double d = __dsub_rn(h, ay);
        t1 = __dmul_rn(ax, __dsub_rn(__dmul_rn(2.0, d), ax));
        t2 = __dmul_rn(__dsub_rn(d, __dmul_rn(2.0, __dsub_rn(ax, ay))), d);
    } else {
        const double d = __dsub_rn(h, ax);
        t1 = __dmul_rn(__dmul_rn(2.0, d), __dsub_rn(ax, __dmul_rn(2.0, ay)));
        t2 = __dadd_rn(__dmul_rn(__dsub_rn(__dmul_rn(4.0, d), ay), ay), __dmul_rn(d, d));
    }
    return __dsub_rn(h, __ddiv_rn(__dadd_rn(t1, t2), __dmul_rn(2.0, h)));
}

__device__ double glibc_hypot(double x, double y)
{
    constexpr double kScale = 0x1p-600, kLarge = 0x1p+511, kTiny = 0x1p-459, kEps = 0x1p-54;
    if (isinf(x) || isinf(y)) return __longlong_as_double(0x7ff0000000000000ll);
    if (isnan(x) || isnan(y)) return __dadd_rn(x, y);
    x = fabs(x); y = fabs(y);
    const double ax = x < y ? y : x, ay = x < y ? x : y;
    if (ax > kLarge) {                                   // scale down: the squares would overflow
        if (ay <= __dmul_rn(ax, kEps)) return __dadd_rn(ax, ay);
        return __ddiv_rn(glibc_hypot_kernel(__dmul_rn(ax, kScale), __dmul_rn(ay, kScale)), kScale);
    }
    if (ay < kTiny) {                                    // scale up: the correction terms would underflow
        if (ax >= __ddiv_rn(ay, kEps)) return __dadd_rn(ax, ay);
        return __dmul_rn(glibc_hypot_kernel(__ddiv_rn(ax, kScale), __ddiv_rn(ay, kScale)), kScale);
    }
    if (ay <= __dmul_rn(ax, kEps)) return __dadd_rn(ax, ay);
    return glibc_hypot_kernel(ax, ay);
}

// np.mean(speedsublist) (s2:310) sums with numpy's pairwise scheme (loops_utils.h.src @TYPE@_pairwise_sum): sequential below 8
// elements, 8 accumulators up to 128, recursive halving above.  A borderline mean < min_speed decision follows numpy's bits.
__device__ double np_sum_block(const double *v, int n)
{
    if (n < 8) {
        double res = 0.0;
        for (int i = 0; i < n; i++) res = res + v[i];
        return res;
    }
    double r[8];
#pragma unroll
    for (int j = 0; j < 8; j++) r[j] = v[j];
    int i = 8;
    for (; i < n - (n % 8); i += 8) {
#pragma unroll
        for (int j = 0; j < 8; j++) r[j] = r[j] + v[i + j];
    }
    double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; i++) res = res + v[i];
    return res;
}
__device__ double np_sum(const double *v, int n)
{
    if (n <= 128) return np_sum_block(v, n);
    int n2 = n / 2;
    n2 -= n2 % 8;
    return np_sum(v, n2) + np_sum(v + n2, n - n2);      // depth log2(n / 128): a track has at most a few hundred vertices
}

__global__ void __launch_bounds__(128)
track_velocities_kernel(const __grid_constant__ VelArgs a)
{
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= a.M) return;
    const int T = a.T;
    const float2 *tr = a.tracks + (int64_t)m * (T + 1);
    double2 *en = a.EN + (int64_t)m * (T + 1);
    double2 *uv = a.uv + (int64_t)m * T;
    double *sp = a.speed + (int64_t)m * T;
    double2 prev = project(a.cam, tr[0]);
    en[0] = prev;
    double smax = 0.0;
    for (int i = 1; i <= T; i++) {
        const double2 cur = project(a.cam, tr[i]);
        en[i] = cur;
        const double u = (cur.x - prev.x) / a.interval, v = (cur.y - prev.y) / a.interval;     // s2:284-285
        const double s = glibc_hypot(u, v);                                                     // s2:286
        uv[i - 1] = make_double2(u, v);
        sp[i - 1] = s;
        if (i == 1 || s > smax) smax = s;
        prev = cur;
    }
    bool keep = true;
    if ((np_sum(sp, T) / (double)T < a.min_speed) || (smax > a.max_speed)) keep = false;       // criterion 1, s2:310
    if (keep && smax > a.speed_threshold && T >= 2) {                                           // s2:314
        double rmax = 0.0, amax = 0.0;
        for (int c1 = 0; c1 + 1 < T; c1++) {
            const double2 a1 = uv[c1], a2 = uv[c1 + 1];
            const double dot = a1.x * a2.x + a1.y * a2.y;
            const double mag1 = glibc_hypot(a1.x, a1.y), mag2 = glibc_hypot(a2.x, a2.y);
            const double ang = fabs(acos(dot / (mag1 * mag2)) * (180.0 / 3.14159265358979323846));   // s2:327-329
            const double s1 = sp[c1], s2 = sp[c1 + 1];
            const double hi = (s2 > s1) ? s2 : s1;                    // max([s1, s2])
            const double lo = (s2 < s1) ? s2 : s1;                    // min([s1, s2])
            const double ratio = hi / lo;
            if (c1 == 0 || ratio > rmax) rmax = ratio;
            if (c1 == 0 || ang > amax) amax = ang;
        }
        if (rmax > a.max_speedfactor) keep = false;                                             // criterion 2, s2:337
        else if (amax > a.max_angle) keep = false;                                              // criterion 3, s2:342
    }
    a.keep[m] = keep ? 1 : 0;
}

} // namespace ibt

static void fill_cam(const double *cam, ibt::UtmCam &c)
{
    const double sg = cam[4], th = cam[6], ph = cam[7], ps = cam[8];
    c.cl = cam[0]; c.ct = cam[1]; c.halfW = cam[2] / 2; c.halfH = cam[3] / 2; c.Hc = cam[5]; c.E0 = cam[9]; c.N0 = cam[10];
    c.sX0 = sg * (cos(th) * cos(ph)); c.sX1 = sg * (sin(th) * cos(ph)); c.sX2 = sg * sin(ph);
    c.U0 = sin(th) * cos(ps) - cos(th) * sin(ph) * sin(ps);
    c.U1 = -cos(th) * cos(ps) - sin(th) * sin(ph) * sin(ps);
    c.U2 = cos(ph) * sin(ps);
    c.V0 = -sin(th) * sin(ps) - cos(th) * sin(ph) * cos(ps);
    c.V1 = cos(th) * sin(ps) - sin(th) * sin(ph) * cos(ps);
    c.V2 = cos(ph) * cos(ps);
}

IBT_API int ibt_photo_to_utm(const float *xy, int64_t n, const double *cam, double *EN, void *stream)
{
    using namespace ibt;
    if (n < 0 || !cam) return IBT_E_INVALID;
    if (n == 0) return IBT_OK;
    if (!xy || !EN || reinterpret_cast<uintptr_t>(xy) % 8 != 0 || reinterpret_cast<uintptr_t>(EN) % 16 != 0) return IBT_E_INVALID;
    UtmCam c;
    fill_cam(cam, c);
    int64_t blocks = (n + 255) / 256;
    if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
    photo_to_utm_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<const float2 *>(xy), n, c, reinterpret_cast<double2 *>(EN));
    return check_launch("ibt_photo_to_utm");
}

IBT_API int ibt_track_velocities(const float *tracks, int M, int T, const double *cam, double interval_s, double min_speed,
                                 double max_speed, double max_speedfactor, double max_angle_deg, double speed_threshold,
                                 double *EN, double *uv, double *speed, uint8_t *keep, void *stream)
{
    using namespace ibt;
    if (M < 0 || T < 1 || !cam || !(interval_s > 0)) return IBT_E_INVALID;
    if (M == 0) return IBT_OK;
    if (!tracks || !EN || !uv || !speed || !keep || reinterpret_cast<uintptr_t>(tracks) % 8 != 0 ||
        reinterpret_cast<uintptr_t>(EN) % 16 != 0 || reinterpret_cast<uintptr_t>(uv) % 16 != 0)
        return IBT_E_INVALID;
    VelArgs a;
    fill_cam(cam, a.cam);
    a.tracks = reinterpret_cast<const float2 *>(tracks); a.M = M; a.T = T; a.interval = interval_s;
    a.min_speed = min_speed; a.max_speed = max_speed; a.max_speedfactor = max_speedfactor; a.max_angle = max_angle_deg;
    a.speed_threshold = speed_threshold;
    a.EN = reinterpret_cast<double2 *>(EN); a.uv = reinterpret_cast<double2 *>(uv); a.speed = speed; a.keep = keep;
    track_velocities_kernel<<<(M + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(a);
    return check_launch("ibt_track_velocities");
}
