/*
 * ibt.h -- C ABI of libibt.so, the B200 (sm_100a) implementation of the tracking hot path of
 * glacierbliss/iceberg_tracking_code.
 *
 * The reference has no FFI layer on this path: its seam is the Python call boundary of three
 * OpenCV functions plus the numpy forward-backward arithmetic around them.  Every entry point
 * below names the reference call site (file:line under /root/reference) it replaces; the
 * Python host (iceberg_tracking_code_b200/cv.py, tracking.py) binds them with ctypes and keeps
 * cv2's signatures.  INTEGRATION.md shows the binding a maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the parameter comment says HOST;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*) unless stated;
 *   - no hidden device allocation: scratch comes from the caller (`*_workspace_bytes`);
 *   - return value 0 = ok, negative = IBT_E_* (ibt_error_string gives text);
 *   - pitches are in BYTES.
 */
#ifndef IBT_H_
#define IBT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IBT_MAX_LEVELS 8          /* maxLevel <= 7 */
#define IBT_MAX_WIN 63            /* winSize components 3..63 */

#define IBT_OK 0
#define IBT_E_INVALID (-1)        /* bad argument (shape, range, null pointer) */
#define IBT_E_CUDA (-2)           /* a CUDA runtime call / kernel launch failed */
#define IBT_E_WORKSPACE (-3)      /* workspace too small */
#define IBT_E_CAPACITY (-4)       /* output capacity too small (count is still reported) */
#define IBT_E_UNSUPPORTED (-5)    /* valid input this library does not handle (e.g. progressive JPEG) */

/* flags of ibt_lk / ibt_lk_fb: same values as cv2.OPTFLOW_* */
#define IBT_LK_USE_INITIAL_FLOW 4
#define IBT_LK_GET_MIN_EIGENVALS 8

/* coefficient sets of ibt_gray_u8 */
#define IBT_GRAY_CV4_15BIT 0      /* OpenCV 4.x: (c0*3735 + c1*19235 + c2*9798 + 2^14) >> 15 */
#define IBT_GRAY_CV3_14BIT 1      /* OpenCV 3.x: (c0*1868 + c1*9617 + c2*4899 + 2^13) >> 14  */

int ibt_version(void);
const char *ibt_error_string(int code);
/* text of the last CUDA error seen by this library on the calling thread (HOST string) */
const char *ibt_last_cuda_error(void);

/* ---- K0: cv2.cvtColor(frame, cv2.COLOR_BGR2GRAY)  s1_lucaskanade_tracking.py:283,311;
 *      s0_1_test_lucaskanade_tracking.py:71,80.  src (H,W,cn) u8, cn = 3 or 4; channel 0
 *      takes the "B" weight whatever it holds (the reference feeds PIL RGB). */
int ibt_gray_u8(const uint8_t *src, int H, int W, int cn, int64_t src_pitch,
                uint8_t *dst, int64_t dst_pitch, int coeffset, void *stream);

/* ---- K1: Gaussian pyramid + Scharr derivative, built inside cv2.calcOpticalFlowPyrLK
 *      (s1:323,326; s0_1:92,95) == cv2.buildOpticalFlowPyramid / cv2.pyrDown.
 * ibt_pyramid_levels: HOST helper.  sizes_hw (HOST, 2*(maxLevel+1) ints) receives (h,w) of
 *      each level kept; returns the effective maxLevel (level l+1 kept only while both dims
 *      exceed the window, strictly). */
int ibt_pyramid_levels(int H, int W, int winW, int winH, int maxLevel, int *sizes_hw);

/* One fused level step: reads level l (h x w, u8) once; writes its Scharr planes
 * (h x w, interleaved int16 dx,dy; pass NULL to skip) and level l+1 (((h+1)/2) x ((w+1)/2), u8;
 * pass NULL to skip).  Borders REFLECT_101.  deriv_pitch % 16 == 0 and deriv % 16 == 0 enable
 * the vector store path (any pitch works). */
int ibt_pyr_level_u8(const uint8_t *src, int h, int w, int64_t src_pitch,
                     int16_t *deriv, int64_t deriv_pitch,
                     uint8_t *down, int64_t down_pitch, void *stream);

/* A pyramid as the LK solver consumes it.  HOST struct, passed by pointer, copied at launch. */
typedef struct ibt_pyramid {
    int32_t nlevels;                              /* effective maxLevel + 1 */
    int32_t rows[IBT_MAX_LEVELS], cols[IBT_MAX_LEVELS];
    const uint8_t *img[IBT_MAX_LEVELS];           /* level images, u8 */
    int64_t img_pitch[IBT_MAX_LEVELS];
    const int16_t *deriv[IBT_MAX_LEVELS];         /* Scharr planes (may be NULL for a J-only pyramid) */
    int64_t deriv_pitch[IBT_MAX_LEVELS];          /* bytes, multiple of 4 */
} ibt_pyramid_t;

/* Whole pyramid of one frame: pyr->img[0] is the caller's gray frame (not copied);
 * pyr->img[1..] and pyr->deriv[0..] are caller-allocated outputs.  with_derivs = 0 skips
 * the Scharr planes. */
int ibt_pyramid_build(const ibt_pyramid_t *pyr, int with_derivs, void *stream);

/* Whole pyramids of one multi-channel frame (cv2.buildOpticalFlowPyramid / calcOpticalFlowPyrLK on an (H,W,cn) u8 frame):
 * frame (H,W,cn) u8 interleaved, row pitch frame_pitch >= W*cn bytes, any pitch and any alignment; cn 2..4.  pyr is a HOST
 * array of cn pyramid pointers, one per channel plane, all with the same nlevels, rows and cols.  Unlike ibt_pyramid_build,
 * pyr[c]->img[0] is an OUTPUT: channel c's level-0 plane, de-interleaved from the frame; pyr[c]->img[1..] and
 * pyr[c]->deriv[0..] are caller-allocated outputs as there.  For every channel the result is ibt_pyramid_build of that
 * channel's plane, which is what OpenCV builds for a multi-channel frame (level l of channel c = the gray pyramid of plane c;
 * OpenCV's derivative channels 2c, 2c+1 = its Scharr (dx, dy)).  One launch reads the frame once and writes every channel's
 * level 0, Scharr planes and level 1; each further level of all channels is one launch.  16-byte aligned frames (base and
 * pitch) are staged by 16-byte copies, any other frame (e.g. a crop view) by a byte gather; the planes take the vector paths
 * of ibt_pyramid_build with 16-byte aligned rows (the LK solver's staging wants 128-byte pitches).  Invalid arguments (cn,
 * null pointers, geometry that differs between channels or levels, a bad pitch) return IBT_E_INVALID before any CUDA call. */
int ibt_pyramid_build_multichannel(const uint8_t *frame, int64_t frame_pitch, int cn, const ibt_pyramid_t *const *pyr,
                                   int with_derivs, void *stream);

/* ---- K3: cv2.calcOpticalFlowPyrLK(img0, img1, p0, None, **lk_params)  s1:323 (forward),
 *      s1:326 (backward); s0_1:92,95.  One pass, I = pyrI (needs deriv), J = pyrJ.
 *      pts (N,2) f32; next_pts (N,2) f32 out (in/out with IBT_LK_USE_INITIAL_FLOW);
 *      status (N) u8; err (N) f32 (0 where status == 0; cv2 leaves garbage there);
 *      iters (N) i32 or NULL: inner Newton iterations executed, summed over levels.
 *      max_count/epsilon are the TERM_CRITERIA values after cv2's defaults were applied
 *      (clamped here to [0,100] / [0,10] like cv2).
 *      Non-finite points (NaN or +-inf in x or y) and points beyond +-2^31 px put the window out of bounds at every
 *      level, as cv2 does on x86: status 0, err 0, no iterations, and next_pts = the input (or the initial flow)
 *      scaled to the top level and back.  A NaN initial flow gives status 0 with no iterations (err = the level-0
 *      minimum eigenvalue with IBT_LK_GET_MIN_EIGENVALS, else 0).  ibt_lk_fb reports such points as not valid. */
int ibt_lk(const ibt_pyramid_t *pyrI, const ibt_pyramid_t *pyrJ,
           const float *pts, float *next_pts, int N,
           int winW, int winH, int max_count, double epsilon, double min_eig_threshold, int flags,
           uint8_t *status, float *err, int32_t *iters, void *stream);

/* Forward + backward pass and the forward-backward check in ONE launch:
 *   p1,st1,err1   = LK(prev -> next, p0)             s1:323
 *   p0r,st0,err0  = LK(next -> prev, p1)             s1:326
 *   fbdist        = hypot(|p0 - p0r|)                s1:329-330 (status is NOT consulted, as in the reference)
 *   alive[k]     &= fbdist < fb_threshold            s1:333, 340-359 (track kept or dropped)
 * alive (N) u8 in/out or NULL (all alive; no write).  Points with alive == 0 are skipped and
 * their outputs left untouched.  iters (N,2) i32 or NULL (fwd, bwd).  iter_total: one u64 or
 * NULL, atomically incremented by the iterations executed (the BASELINE.md unit).
 * Any of st1, err1, st0, err0 may be NULL. */
int ibt_lk_fb(const ibt_pyramid_t *prev, const ibt_pyramid_t *next,
              const float *p0, int N,
              int winW, int winH, int max_count, double epsilon, double min_eig_threshold,
              float fb_threshold,
              float *p1, uint8_t *st1, float *err1,
              float *p0r, uint8_t *st0, float *err0,
              float *fbdist, uint8_t *alive, int32_t *iters, unsigned long long *iter_total,
              void *stream);
/* cv2.calcOpticalFlowPyrLK on multi-channel 8-bit images (cv2 takes 3-channel frames as well, SURVEY 8b; the reference converts
 * to gray first, s1:311, so this is the plain form of the solver): pyrI / pyrJ are HOST arrays of cn (1..4) pointers to
 * single-channel pyramids, one per channel plane (pyrI with Scharr planes).  OpenCV sums the structure tensor, the mismatch
 * vector and the residual over the window pixels and the channels; err is divided by 32 * winW * cn * winH.  Same arguments
 * and outputs as ibt_lk otherwise. */
int ibt_lk_multichannel(const ibt_pyramid_t *const *pyrI, const ibt_pyramid_t *const *pyrJ, int cn,
                        const float *pts, float *next_pts, int N,
                        int winW, int winH, int max_count, double epsilon, double min_eig_threshold, int flags,
                        uint8_t *status, float *err, int32_t *iters, void *stream);
/* ibt_lk_fb on multi-channel frames: prev / next are HOST arrays of cn (2..4) channel pyramids as in ibt_lk_multichannel, and
 * BOTH need Scharr planes (the backward pass tracks next -> prev).  Forward, backward and the forward-backward check run in one
 * launch with ibt_lk_fb's arguments and outputs; each pass equals ibt_lk_multichannel in that direction. */
int ibt_lk_fb_multichannel(const ibt_pyramid_t *const *prev, const ibt_pyramid_t *const *next, int cn,
                           const float *p0, int N,
                           int winW, int winH, int max_count, double epsilon, double min_eig_threshold,
                           float fb_threshold,
                           float *p1, uint8_t *st1, float *err1,
                           float *p0r, uint8_t *st0, float *err0,
                           float *fbdist, uint8_t *alive, int32_t *iters, unsigned long long *iter_total,
                           void *stream);
/* Process-wide occupancy cap of the persistent LK launches: at most `ctas` resident CTAs (of 8 warps) per SM, 0 = fill the SM
 * (default, 3 for the usual window sizes).  With 2 the launch leaves a third of every SM's shared memory and registers to
 * kernels of other streams -- e.g. the JPEG decode of the next frame (measured: LK 7 % slower, decode fully overlapped). */
int ibt_lk_set_max_ctas_per_sm(int ctas);

/* ---- K2: cv2.goodFeaturesToTrack(frame_gray, mask=mask, **feature_params)  s1:437; s0_1:167.
 * cornerMinEigenVal / cornerHarris test hooks (Sobel3 -> products -> blockSize^2 box sum -> lambda_min, or OpenCV's Harris
 * response (a*c - b*b) - k*(a + c)^2 in float). */
int ibt_min_eigen_f32(const uint8_t *gray, int H, int W, int64_t pitch, int blockSize,
                      float *eig, int64_t eig_pitch, void *stream);
int ibt_corner_harris_f32(const uint8_t *gray, int H, int W, int64_t pitch, int blockSize, double k,
                          float *dst, int64_t dst_pitch, void *stream);
/* The same maps for cv2's other Sobel apertures: ksize (cv2's ksize / gradientSize) is -1 (Scharr), 1, 3, 5 or 7; anything else
 * returns IBT_E_INVALID before any CUDA call.  ksize 3 is exactly ibt_min_eigen_f32 / ibt_corner_harris_f32.  As in OpenCV's
 * cornerEigenValsVecs, dx correlates the derivative taps d along x and the smoothing taps s along y (dy the transpose), and
 * the derivatives are scaled by 1 / (sden * blockSize * 255):
 *     ksize   d                   s                   sden   max |dx| before scaling, u8 input
 *       1     -1 0 1              1                     1      255
 *       3     -1 0 1              1 2 1                 4      1 020
 *      -1     -1 0 1              3 10 3 (Scharr)       8      4 080
 *       5     -1 -2 0 2 1         1 4 6 4 1            16      12 240
 *       7     -1 -4 -5 0 5 4 1    1 6 15 20 15 6 1     64      163 200
 * The window sums of the exact integer products reach 1.6e10 (Scharr), 1.4e11 (5) and 2.6e13 (7) at blockSize 31, beyond
 * int32: apertures other than 3 sum them in int64, exact (every sum is below 2^53). */
int ibt_min_eigen_ksize_f32(const uint8_t *gray, int H, int W, int64_t pitch, int blockSize, int ksize,
                            float *eig, int64_t eig_pitch, void *stream);
int ibt_corner_harris_ksize_f32(const uint8_t *gray, int H, int W, int64_t pitch, int blockSize, int ksize, double k,
                                float *dst, int64_t dst_pitch, void *stream);

size_t ibt_gftt_workspace_bytes(int H, int W);
/* mask may be NULL (all allowed).  out_xy (cap,2) f32 receives integer-valued x,y ordered by
 * response (ties: higher linear address first), culled by minDistance on cv2's cell grid and
 * truncated to maxCorners (<= 0: unlimited).  useHarrisDetector / k: cv2's arguments of the same name (the reference leaves
 * them at False / 0.04, s1:240-243): non-zero ranks the Harris response instead of lambda_min.  out_count: HOST int*.
 * SYNCHRONISES `stream` (the corner count decides the shapes the caller allocates next, like cv2's return value).
 * Returns IBT_E_CAPACITY (and the full count) if cap was too small.  It also returns IBT_E_CAPACITY when the raw 3x3 maxima
 * above the threshold exceed the workspace's candidate capacity, H*W/4 + 4096: isolated maxima never do, only plateaus of
 * exactly equal responses (e.g. blockSize 31 on a periodic 0/255 checkerboard). */
int ibt_gftt(const uint8_t *gray, int64_t pitch, const uint8_t *mask, int64_t mask_pitch,
             int H, int W, int maxCorners, double qualityLevel, double minDistance, int blockSize,
             int useHarrisDetector, double k,
             void *workspace, size_t workspace_bytes,
             float *out_xy, int cap, int *out_count, void *stream);
/* Same two launches, nothing read back: count_dev (DEVICE int*) receives the corner count when the stream reaches it, out_xy
 * the corners.  The frame loop (s1:437-448) seeds the next group with it while earlier work is still in flight; the count
 * travels to ibt_lk_fb as n_dev.  A capacity overflow is reported by the next synchronous call on the workspace. */
int ibt_gftt_async(const uint8_t *gray, int64_t pitch, const uint8_t *mask, int64_t mask_pitch,
                   int H, int W, int maxCorners, double qualityLevel, double minDistance, int blockSize,
                   int useHarrisDetector, double k,
                   void *workspace, size_t workspace_bytes,
                   float *out_xy, int cap, int *count_dev, void *stream);
/* ibt_gftt / ibt_gftt_async with cv2's gradientSize: the Sobel aperture of the response (-1, 1, 3, 5 or 7, as
 * ibt_min_eigen_ksize_f32; anything else returns IBT_E_INVALID before any CUDA call).  The plain forms are gradientSize 3. */
int ibt_gftt_ksize(const uint8_t *gray, int64_t pitch, const uint8_t *mask, int64_t mask_pitch,
                   int H, int W, int maxCorners, double qualityLevel, double minDistance, int blockSize, int gradientSize,
                   int useHarrisDetector, double k,
                   void *workspace, size_t workspace_bytes,
                   float *out_xy, int cap, int *out_count, void *stream);
int ibt_gftt_async_ksize(const uint8_t *gray, int64_t pitch, const uint8_t *mask, int64_t mask_pitch,
                         int H, int W, int maxCorners, double qualityLevel, double minDistance, int blockSize, int gradientSize,
                         int useHarrisDetector, double k,
                         void *workspace, size_t workspace_bytes,
                         float *out_xy, int cap, int *count_dev, void *stream);

/* ---- track bookkeeping at a group boundary (s1:362-395): stable compaction of the live
 * tracks.  tracks_tm (T+1, N, 2) f32 time-major, quality_tm (T, N) f32, alive (N) u8 ->
 * out_tracks (M, T+1, 2) f32, out_quality (M, T) f32 in seed order.  scratch: (N+1) int32.
 * out_count: HOST int*; SYNCHRONISES `stream`. */
int ibt_tracks_compact(const float *tracks_tm, const float *quality_tm, const uint8_t *alive,
                       int N, int T, int32_t *scratch, float *out_tracks, float *out_quality,
                       int *out_count, void *stream);
/* Same launches, nothing read back: the survivor count stays in scratch[N] (device) -- the frame loop copies it to pinned host
 * memory together with the arrays and finalises the group one group later, while the next group's kernels run. */
int ibt_tracks_compact_async(const float *tracks_tm, const float *quality_tm, const uint8_t *alive,
                             int N, int T, int32_t *scratch, float *out_tracks, float *out_quality, void *stream);

/* ---- K4: Camera.photocords_cropped_to_uncropped + Camera.photo_to_utm
 *      imports/camtools.py:414-421, 286-332, called per vertex at s2_cam_to_utm.py:247-254.
 * xy (n,2) f32 track vertices in cropped-image pixels; cam: HOST, 12 doubles
 * { crop_left, crop_top, image_width, image_height, sigma_px, H_cam, theta, phi, psi (radians),
 *   easting, northing, reserved }.  EN (n,2) f64.  All arithmetic in fp64. */
int ibt_photo_to_utm(const float *xy, int64_t n, const double *cam, double *EN, void *stream);

/* ---- s2 consumer: the per-track body of cam_to_utm, s2_cam_to_utm.py:243-343, for all tracks of one .npz file:
 *      project every vertex (as ibt_photo_to_utm), u = dE/dt, v = dN/dt, speed = hypot(u, v) per segment (s2:279-290),
 *      then the plausibility criteria (s2:309-343): mean speed < min_speed or max speed > max_speed; and, only when
 *      max speed > speed_threshold, consecutive speed ratio > max_speedfactor or direction change > max_angle_deg.
 *      tracks (M, T+1, 2) f32; cam HOST 12 doubles; EN (M, T+1, 2) f64; uv (M, T, 2) f64; speed (M, T) f64; keep (M) u8. */
int ibt_track_velocities(const float *tracks, int M, int T, const double *cam, double interval_s, double min_speed,
                         double max_speed, double max_speedfactor, double max_angle_deg, double speed_threshold,
                         double *EN, double *uv, double *speed, uint8_t *keep, void *stream);

/* ---- mask: Camera.mask_meshgrid (imports/camtools.py:184-211) as used at s1:285-294: rasterise the (already
 *      crop-shifted) water polygon over the H x W pixel centres.  poly_xy: DEVICE (E,2) f64, 3 <= E <= 2048,
 *      implicitly closed; crossing-number rule of matplotlib.path.Path.contains_points (radius 0).
 *      out[y*pitch + x] = inside ? inside_value : 0. */
int ibt_polygon_mask(const double *poly_xy, int E, int H, int W, uint8_t *out, int64_t pitch, int inside_value,
                     void *stream);

/* ---- K5: frame = np.array(Image.open(image))  s1_lucaskanade_tracking.py:310; s0_1_test_lucaskanade_tracking.py:79
 *      (+ the cv2.cvtColor of s1:311 / s0_1:80 fused): baseline JPEG decoding on the GPU, bit-exact with Pillow's
 *      libjpeg-turbo defaults (islow IDCT, fancy upsampling, fixed-point YCbCr->RGB).
 *      Handled: baseline / extended sequential 8-bit Huffman (SOF0, SOF1), one interleaved scan, grey-scale or YCbCr with
 *      4:4:4, 4:2:2 (2x1) or 4:2:0 (2x2) sampling, with or without restart markers.  Anything else -> IBT_E_UNSUPPORTED
 *      (callers fall back to their own decoder and upload the pixels). */
typedef struct ibt_jpeg_info {
    int32_t width, height, ncomp;                 /* ncomp 1 (grey) or 3 (YCbCr) */
    int32_t hsamp[3], vsamp[3];                   /* sampling factors per component */
    int32_t qsel[3], dcsel[3], acsel[3];          /* table selectors per component */
    int32_t restart_interval;                     /* DRI value (0 = none) */
    int32_t reserved;
    int64_t scan_offset, scan_bytes;              /* entropy-coded segment inside the file */
    uint16_t quant[4][64];                        /* quantisation tables, natural (row-major) order */
    uint8_t dc_bits[4][16], dc_vals[4][16];       /* Huffman tables as in DHT: counts per length 1..16, symbols */
    uint8_t ac_bits[4][16], ac_vals[4][256];
} ibt_jpeg_info_t;

/* HOST only (no GPU work): parse the markers of a JPEG file held in host memory. */
int ibt_jpeg_parse(const uint8_t *host_file, int64_t nbytes, ibt_jpeg_info_t *info);
/* bytes of device scratch ibt_jpeg_decode needs for this file (0 if the info is not decodable) */
int64_t ibt_jpeg_workspace_bytes(const ibt_jpeg_info_t *info);
/* d_file: the whole file in DEVICE memory (4-byte aligned).  info: HOST.  workspace: 256-byte aligned.
 * rgb (H,W,3) u8 = what np.array(Image.open(f)) holds (NULL to skip; must be NULL for grey-scale files);
 * gray (H,W) u8 = cv2.cvtColor(that, COLOR_BGR2GRAY) with the reference's channel order (NULL to skip; for a
 * grey-scale file: the decoded plane).  coeffset as ibt_gray_u8.  out_rounds: HOST int* or NULL, in/out: on entry a hint
 * (> 0: rounds a similar file needed; sizes the first batch of rounds), on return the number of Huffman synchronisation
 * rounds this file needed.  SYNCHRONISES `stream` (convergence of the speculative Huffman decode). */
int ibt_jpeg_decode(const uint8_t *d_file, const ibt_jpeg_info_t *info, void *workspace, int64_t workspace_bytes,
                    uint8_t *rgb, int64_t rgb_pitch, uint8_t *gray, int64_t gray_pitch, int coeffset,
                    int *out_rounds, void *stream);
/* ibt_jpeg_decode without the host round trip: exactly `rounds` synchronisation rounds are enqueued (1..64; a round after the
 * fixed point changes nothing and costs a few microseconds), their change counters are copied to h_pinned[0 .. rounds) (uint32,
 * PINNED host memory of at least ibt_jpeg_async_host_bytes(), owned by this call until the stream has passed it) and the
 * rest of the decode is enqueued right away.  Once the stream has reached that point: the output is valid iff one of the
 * counters is 0; otherwise call ibt_jpeg_decode (and use more rounds next time). */
int64_t ibt_jpeg_async_host_bytes(void);
int ibt_jpeg_decode_async(const uint8_t *d_file, const ibt_jpeg_info_t *info, void *workspace, int64_t workspace_bytes,
                          uint8_t *rgb, int64_t rgb_pitch, uint8_t *gray, int64_t gray_pitch, int coeffset, int rounds,
                          void *h_pinned, int64_t h_pinned_bytes, void *stream);
/* Process-wide switch of the entry-state probe of the Huffman pass (default on).  The probe decodes every subsequence once per
 * block position of the MCU to guess its entry state: fewer synchronisation rounds, i.e. a shorter decode LATENCY (7 instead of
 * 9 rounds on a dense 24 MP file), at the price of a full-grid kernel.  A frame loop that keeps several decodes in flight beside
 * the tracker (ibt_jpeg_decode_async) hides the latency anyway and runs ~4 % faster without it (the rounds occupy few SMs). */
int ibt_jpeg_set_probe(int enabled);

/* ---- the save-and-reopen round trip of the reference's cropping pre-pass, without the files:
 *      `img_crop.save(outpath)` (imports/camtools.py:80,102,232 via crop_image_parallel, s1_lucaskanade_tracking.py:272)
 *      followed by `np.array(Image.open(image))` (s1:310; + the cv2.cvtColor of s1:311 fused).  Pillow's save re-encodes the
 *      crop with libjpeg-turbo (defaults: quality 75, 4:2:0, islow DCT); entropy coding is lossless, so the pixels the
 *      reference tracks are decode(quantise(FDCT(downsample(RGB->YCbCr(crop))))) -- computed here bit-exactly as pure integer
 *      work on the GPU, which removes the ~0.3 s per 24 MP frame host pre-pass without changing a pixel.
 *      rgb_in: DEVICE (height, width, 3) u8 with row pitch in_pitch bytes, any alignment (a crop VIEW of a decoded frame).
 *      quality 1..100 as Image.save(quality=); hsamp x vsamp = luma sampling 2x2 (4:2:0, Pillow's default), 2x1, 1x1.
 *      workspace: 256-byte aligned, ibt_jpeg_recompress_workspace_bytes().  rgb / gray / coeffset as ibt_jpeg_decode.
 *      Asynchronous on `stream`. */
int64_t ibt_jpeg_recompress_workspace_bytes(int width, int height, int hsamp, int vsamp);
int ibt_jpeg_recompress(const uint8_t *rgb_in, int64_t in_pitch, int width, int height, int quality, int hsamp, int vsamp,
                        void *workspace, int64_t workspace_bytes, uint8_t *rgb, int64_t rgb_pitch, uint8_t *gray,
                        int64_t gray_pitch, int coeffset, void *stream);

/* ---- s3 consumer: the cell-binning loop of s3_utm_to_gridded_utm.py:391-421 over the square grid of
 *      imports/tracking_misc.py:25-58.  Cell (i, j), i < cols, j < rows, is the square with top-left corner
 *      (topleft_x + i*spacing, topleft_y - j*spacing); membership is matplotlib.path.Path(poly).contains_points (radius 0).
 *      x, y, u, v: (n) f64 each.  Outputs indexed i*rows + j: count (observations in the cell), sum_u, sum_v =
 *      np.sum of the selected displacements in point order (numpy's pairwise summation, bit-exact). */
int64_t ibt_grid_bin_workspace_bytes(int64_t n, int cols, int rows);
int ibt_grid_bin(const double *x, const double *y, const double *u, const double *v, int64_t n,
                 double topleft_x, double topleft_y, double spacing, int cols, int rows,
                 void *workspace, int64_t workspace_bytes,
                 int32_t *count, double *sum_u, double *sum_v, void *stream);
/* matplotlib.path.Path(poly).contains_points(pts) (radius 0; polygon implicitly closed; 3 <= E <= 4096), e.g. the
 * cell centres inside the fjord outline, imports/tracking_misc.py:34-52.  poly_xy (E,2) f64, pts_xy (n,2) f64, out (n) u8. */
int ibt_points_in_polygon(const double *poly_xy, int E, const double *pts_xy, int64_t n, uint8_t *out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* IBT_H_ */
