// s3 consumer (SURVEY.md 8f rank 4): the binning loop of s3_utm_to_gridded_utm.py:391-421 -- for every square cell of the
// fjord grid (imports/tracking_misc.py:25-58), matplotlib.path.Path(poly).contains_points(points) selects the velocities
// inside it and np.sum / count gives the cell mean.  The reference tests every point against every cell polygon.
// Here: each point tests the 3x3 cells around its own position with matplotlib's crossing rule (same fp64 expressions,
// same half-open edges), the (cell, point) pairs are ordered by a stable radix sort, and one thread per cell adds its
// velocities IN POINT ORDER with numpy's pairwise summation (8 accumulators up to 128 elements, recursive halving above):
// count and sums are bit-identical to the reference's np.sum over the boolean-indexed array.
// Also here: Path.contains_point(s) for arbitrary points (cell centres inside the fjord outline, tracking_misc.py:52).
#include <atomic>
#include "common.cuh"

namespace ibt {

// matplotlib _path.h point_in_path_impl (the "crossings" test, polygon implicitly closed), fp64
__device__ __forceinline__ bool crossing_step(double v0x, double v0y, double v1x, double v1y, double tx, double ty, bool &yflag0,
                                              bool inside)
{
    const bool yflag1 = v1y >= ty;
    if (yflag0 != yflag1) {
        if (((v1y - ty) * (v0x - v1x) >= (v1x - tx) * (v0y - v1y)) == yflag1) inside = !inside;
    }
    yflag0 = yflag1;
    return inside;
}

constexpr int GRID_MAX_POLY = 4096;

__global__ void __launch_bounds__(256)
points_in_polygon_kernel(const double2 *__restrict__ poly, int E, const double2 *__restrict__ pts, int64_t n, uint8_t *__restrict__ out)
{
    extern __shared__ double2 sp[];
    for (int i = threadIdx.x; i < E; i += blockDim.x) sp[i] = poly[i];
    __syncthreads();
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const double2 t = pts[p];
    double2 v0 = sp[E - 1];
    bool yflag0 = v0.y >= t.y, inside = false;
    for (int i = 0; i < E; i++) {
        const double2 v1 = sp[i];
        inside = crossing_step(v0.x, v0.y, v1.x, v1.y, t.x, t.y, yflag0, inside);
        v0 = v1;
    }
    out[p] = inside ? 1 : 0;
}

// square cell (i, j): create_squares(origin, spacing, spacing) with origin = [topleft[0] + i*spacing, topleft[1] - j*spacing]
// (tracking_misc.py:15-23, 44-46): vertices (x,y), (x+w,y), (x+w,y-w), (x,y-w)
__device__ __forceinline__ bool in_cell(double tx, double ty, double x0, double y0, double s, int i, int j)
{
    const double x = x0 + (double)i * s, y = y0 - (double)j * s;
    const double xr = x + s, yb = y - s;
    bool yflag0 = yb >= ty, inside = false;                   // previous vertex of the first one: (x, y-w)
    inside = crossing_step(x, yb, x, y, tx, ty, yflag0, inside);
    inside = crossing_step(x, y, xr, y, tx, ty, yflag0, inside);
    inside = crossing_step(xr, y, xr, yb, tx, ty, yflag0, inside);
    inside = crossing_step(xr, yb, x, yb, tx, ty, yflag0, inside);
    return inside;
}

constexpr int GRID_SLOTS = 4;                                 // cells one point can belong to (1 except on 1-ulp seams)
constexpr unsigned long long GRID_NONE = ~0ull;

__global__ void __launch_bounds__(256)
grid_assign_kernel(const double *__restrict__ px, const double *__restrict__ py, uint32_t n, double x0, double y0, double s, int cols,
                   int rows, unsigned long long *__restrict__ keys)
{
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const double tx = px[p], ty = py[p];
    unsigned long long k[GRID_SLOTS] = {GRID_NONE, GRID_NONE, GRID_NONE, GRID_NONE};
    const double fi = floor((tx - x0) / s), fj = floor((y0 - ty) / s);
    // NaN / far-away points fail this test and land in no cell.  (Deliberate difference: the crossing rule itself puts a
    // point with x = NaN into EVERY cell of its row -- all its comparisons are false -- which is a quirk, not a result.)
    if (fi >= -1.0 && fi <= (double)cols && fj >= -1.0 && fj <= (double)rows) {
        const int i0 = (int)fi, j0 = (int)fj;
        int m = 0;
        for (int i = max(i0 - 1, 0); i <= min(i0 + 1, cols - 1); i++)
            for (int j = max(j0 - 1, 0); j <= min(j0 + 1, rows - 1); j++)
                if (m < GRID_SLOTS && in_cell(tx, ty, x0, y0, s, i, j))
                    k[m++] = (unsigned long long)((uint32_t)i * (uint32_t)rows + (uint32_t)j) << 32 | p;
    }
#pragma unroll
    for (int q = 0; q < GRID_SLOTS; q++) keys[(size_t)p * GRID_SLOTS + q] = k[q];
}

__global__ void __launch_bounds__(256)
grid_segments_kernel(const unsigned long long *__restrict__ keys, uint32_t nk, uint32_t *__restrict__ seg_start, uint32_t *__restrict__ seg_end)
{
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nk) return;
    const unsigned long long k = keys[t];
    if (k == GRID_NONE) return;
    const uint32_t c = (uint32_t)(k >> 32);
    if (t == 0 || (uint32_t)(keys[t - 1] >> 32) != c) seg_start[c] = t;
    if (t + 1 == nk || keys[t + 1] == GRID_NONE || (uint32_t)(keys[t + 1] >> 32) != c) seg_end[c] = t + 1;
}

// numpy's pairwise summation (loops_utils.h.src, @TYPE@_pairwise_sum) of val[idx[k] & 0xffffffff], k in [lo, lo + n)
__device__ double np_block_sum(const double *__restrict__ val, const unsigned long long *__restrict__ keys, uint32_t lo, uint32_t n)
{
    auto at = [&](uint32_t k) { return val[(uint32_t)keys[lo + k]]; };
    if (n < 8) {
        double res = 0.0;
        for (uint32_t i = 0; i < n; i++) res = res + at(i);
        return res;
    }
    double r[8];
#pragma unroll
    for (int j = 0; j < 8; j++) r[j] = at(j);
    uint32_t i = 8;
    for (; i < n - (n % 8); i += 8) {
#pragma unroll
        for (int j = 0; j < 8; j++) r[j] = r[j] + at(i + j);
    }
    double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; i++) res = res + at(i);
    return res;
}
__device__ double np_pairwise_sum(const double *__restrict__ val, const unsigned long long *__restrict__ keys, uint32_t lo, uint32_t n)
{
    if (n <= 128) return np_block_sum(val, keys, lo, n);
    // iterative form of: n2 = n/2 - (n/2)%8; return sum(a, n2) + sum(a + n2, n - n2)   (post-order, explicit stack)
    struct Frame { uint32_t lo, n; int state; double left; };
    Frame st[40];
    int sp = 0;
    st[0] = {lo, n, 0, 0.0};
    double ret = 0.0;
    while (sp >= 0) {
        Frame &f = st[sp];
        if (f.n <= 128) { ret = np_block_sum(val, keys, f.lo, f.n); sp--; continue; }
        uint32_t n2 = f.n / 2; n2 -= n2 % 8;
        if (f.state == 0) { f.state = 1; st[sp + 1] = {f.lo, n2, 0, 0.0}; sp++; }
        else if (f.state == 1) { f.left = ret; f.state = 2; st[sp + 1] = {f.lo + n2, f.n - n2, 0, 0.0}; sp++; }
        else { ret = f.left + ret; sp--; }
    }
    return ret;
}

__global__ void __launch_bounds__(128)
grid_reduce_kernel(const double *__restrict__ u, const double *__restrict__ v, const unsigned long long *__restrict__ keys,
                   const uint32_t *__restrict__ seg_start, const uint32_t *__restrict__ seg_end, int ncell, int32_t *__restrict__ count,
                   double *__restrict__ sum_u, double *__restrict__ sum_v)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncell) return;
    const uint32_t lo = seg_start[c], n = seg_end[c] - lo;
    count[c] = (int32_t)n;
    // np.sum = add.reduce: the accumulator starts at the identity 0.0
    sum_u[c] = 0.0 + np_pairwise_sum(u, keys, lo, n);
    sum_v[c] = 0.0 + np_pairwise_sum(v, keys, lo, n);
}

// radix sort (ascending, 64-bit keys, stable LSD, 8-bit digits)
constexpr int RS_WARPS = 8, RS_STEPS = 16, RS_TILE = RS_WARPS * RS_STEPS * 32;   // 4096 keys per block

__global__ void __launch_bounds__(256)
rs_count_kernel(const unsigned long long *__restrict__ keys, uint32_t n, int shift, uint32_t nblocks,
                uint32_t *__restrict__ blockhist /*[256][nblocks]*/)
{
    __shared__ uint32_t sh[256];
    sh[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t base = blockIdx.x * RS_TILE;
    for (uint32_t i = threadIdx.x; i < RS_TILE; i += 256) {
        const uint32_t g = base + i;
        if (g < n) atomicAdd(&sh[(uint32_t)((keys[g] >> shift) & 0xff)], 1u);
    }
    __syncthreads();
    blockhist[threadIdx.x * nblocks + blockIdx.x] = sh[threadIdx.x];
}

__global__ void __launch_bounds__(256)
rs_scatter_kernel(const unsigned long long *__restrict__ src, unsigned long long *__restrict__ dst, uint32_t n,
                  int shift, uint32_t nblocks, const uint32_t *__restrict__ blockoff /*[256][nblocks] scanned*/)
{
    __shared__ uint32_t wcount[RS_WARPS][256];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < RS_WARPS * 256; i += 256) (&wcount[0][0])[i] = 0;
    __syncthreads();
    const uint32_t wbase = blockIdx.x * RS_TILE + wid * (RS_STEPS * 32);
    unsigned long long k[RS_STEPS];
    uint32_t rank[RS_STEPS];
#pragma unroll
    for (int s = 0; s < RS_STEPS; s++) {
        const uint32_t g = wbase + s * 32 + lane;
        const bool valid = g < n;
        k[s] = valid ? src[g] : 0ull;
        const uint32_t d = (uint32_t)((k[s] >> shift) & 0xff);
        const uint32_t vmask = __ballot_sync(0xffffffffu, valid);
        uint32_t peers = __match_any_sync(0xffffffffu, valid ? d : 0x100u + lane) & vmask;
        if (!valid) peers = 0;
        const uint32_t before = __popc(peers & ((1u << lane) - 1));
        uint32_t prev = 0;
        if (valid) prev = wcount[wid][d];          // all peers read the same value before the leader updates
        __syncwarp();
        if (valid && before == 0) wcount[wid][d] = prev + __popc(peers);
        __syncwarp();
        rank[s] = prev + before;                  // rank within this warp's chunk for digit d
    }
    __syncthreads();
    // exclusive prefix over warps per digit, plus the global offset of (digit, block)
    {
        const int d = threadIdx.x;
        uint32_t run = blockoff[d * nblocks + blockIdx.x];
#pragma unroll
        for (int w = 0; w < RS_WARPS; w++) { const uint32_t c = wcount[w][d]; wcount[w][d] = run; run += c; }
    }
    __syncthreads();
#pragma unroll
    for (int s = 0; s < RS_STEPS; s++) {
        const uint32_t g = wbase + s * 32 + lane;
        if (g < n) {
            const uint32_t d = (uint32_t)((k[s] >> shift) & 0xff);
            dst[wcount[wid][d] + rank[s]] = k[s];
        }
    }
}

// Stable LSD radix sort of n 64-bit keys on bytes [first_byte, last_byte].  keys0 holds the input, keys1 is the ping-pong
// buffer; returns the buffer that holds the result.  scratch: radix_sort_scratch_words(n) uint32, n <= 2^30.
static size_t radix_sort_scratch_words(uint32_t n)
{
    const size_t nblocks = ((size_t)n + RS_TILE - 1) / RS_TILE;
    return 256 * nblocks + scan_partial_words((int)(256 * nblocks), 1);
}
static unsigned long long *radix_sort_u64_bytes(unsigned long long *keys0, unsigned long long *keys1, uint32_t n, int first_byte,
                                                int last_byte, uint32_t *scratch, cudaStream_t st)
{
    if (n <= 1) return keys0;
    const uint32_t nblocks = (n + RS_TILE - 1) / RS_TILE;
    uint32_t *blockhist = scratch, *partial = scratch + 256 * (size_t)nblocks;
    unsigned long long *src = keys0, *dst = keys1;
    for (int p = first_byte; p <= last_byte; p++) {
        rs_count_kernel<<<nblocks, 256, 0, st>>>(src, n, 8 * p, nblocks, blockhist);
        launch_scan(blockhist, blockhist, partial, (int)(256 * nblocks), 1, 0, nullptr, st);
        rs_scatter_kernel<<<nblocks, 256, 0, st>>>(src, dst, n, 8 * p, nblocks, blockhist);
        unsigned long long *t = src; src = dst; dst = t;
    }
    return src;
}

struct GridLayout { size_t off_keys0, off_keys1, off_scratch, off_start, off_end, total; };
static void grid_layout(int64_t n, int ncell, GridLayout &L)
{
    size_t o = 0;
    auto take = [&](size_t b) { const size_t r = o; o += (b + 255) & ~(size_t)255; return r; };
    const size_t nk = (size_t)n * GRID_SLOTS;
    L.off_keys0 = take(nk * 8);
    L.off_keys1 = take(nk * 8);
    L.off_scratch = take(radix_sort_scratch_words((uint32_t)nk) * 4);
    L.off_start = take((size_t)ncell * 4);
    L.off_end = take((size_t)ncell * 4);
    L.total = o;
}

} // namespace ibt

IBT_API int ibt_points_in_polygon(const double *poly_xy, int E, const double *pts_xy, int64_t n, uint8_t *out, void *stream)
{
    using namespace ibt;
    if (!poly_xy || !pts_xy || !out || E < 3 || E > GRID_MAX_POLY || n < 0 || reinterpret_cast<uintptr_t>(poly_xy) % 16 != 0 ||
        reinterpret_cast<uintptr_t>(pts_xy) % 16 != 0)
        return IBT_E_INVALID;
    if (n == 0) return IBT_OK;
    const size_t smem = (size_t)E * sizeof(double2);
    if (smem > 48 * 1024) {
        // > 3072 vertices: opt in to more dynamic shared memory, once per device (the attribute is per device; setting it
        // again from a second host thread is harmless)
        static std::atomic<bool> attr_set[64];
        int dev_id = 0;
        IBT_CUDA_TRY(cudaGetDevice(&dev_id));
        if (dev_id < 0 || dev_id >= 64) return IBT_E_INVALID;
        if (!attr_set[dev_id].load(std::memory_order_acquire)) {
            IBT_CUDA_TRY(cudaFuncSetAttribute(points_in_polygon_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GRID_MAX_POLY * 16));
            attr_set[dev_id].store(true, std::memory_order_release);
        }
    }
    points_in_polygon_kernel<<<(unsigned)((n + 255) / 256), 256, smem, static_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<const double2 *>(poly_xy), E, reinterpret_cast<const double2 *>(pts_xy), n, out);
    return check_launch("ibt_points_in_polygon");
}

IBT_API int64_t ibt_grid_bin_workspace_bytes(int64_t n, int cols, int rows)
{
    if (n < 0 || n > (1ll << 28) || cols <= 0 || rows <= 0 || (int64_t)cols * rows > (1ll << 24)) return 0;
    ibt::GridLayout L;
    ibt::grid_layout(n, cols * rows, L);
    return (int64_t)L.total;
}

IBT_API int ibt_grid_bin(const double *x, const double *y, const double *u, const double *v, int64_t n, double topleft_x,
                         double topleft_y, double spacing, int cols, int rows, void *workspace, int64_t workspace_bytes,
                         int32_t *count, double *sum_u, double *sum_v, void *stream)
{
    using namespace ibt;
    if (n < 0 || n > (1ll << 28) || cols <= 0 || rows <= 0 || (int64_t)cols * rows > (1ll << 24) || !(spacing > 0) || !count ||
        !sum_u || !sum_v)
        return IBT_E_INVALID;
    if (n > 0 && (!x || !y || !u || !v || !workspace)) return IBT_E_INVALID;
    const int ncell = cols * rows;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    GridLayout L;
    grid_layout(n, ncell, L);
    if (n > 0 && (workspace_bytes < (int64_t)L.total || reinterpret_cast<uintptr_t>(workspace) % 256 != 0)) return IBT_E_WORKSPACE;
    if (n == 0) {
        IBT_CUDA_TRY(cudaMemsetAsync(count, 0, (size_t)ncell * 4, st));
        IBT_CUDA_TRY(cudaMemsetAsync(sum_u, 0, (size_t)ncell * 8, st));
        IBT_CUDA_TRY(cudaMemsetAsync(sum_v, 0, (size_t)ncell * 8, st));
        return IBT_OK;
    }
    uint8_t *ws = static_cast<uint8_t *>(workspace);
    unsigned long long *keys0 = reinterpret_cast<unsigned long long *>(ws + L.off_keys0);
    unsigned long long *keys1 = reinterpret_cast<unsigned long long *>(ws + L.off_keys1);
    uint32_t *scratch = reinterpret_cast<uint32_t *>(ws + L.off_scratch);
    uint32_t *seg_start = reinterpret_cast<uint32_t *>(ws + L.off_start), *seg_end = reinterpret_cast<uint32_t *>(ws + L.off_end);
    const uint32_t nk = (uint32_t)n * GRID_SLOTS;
    grid_assign_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(x, y, (uint32_t)n, topleft_x, topleft_y, spacing, cols, rows, keys0);
    // keys are in point order already: a stable sort on the cell bytes alone groups them by cell, point order kept
    // (unused slots carry 0xff.. in every byte and end up behind all cells: ncell <= 2^24 < 0xffffff..)
    unsigned long long *sorted = radix_sort_u64_bytes(keys0, keys1, nk, 4, 7, scratch, st);
    IBT_CUDA_TRY(cudaMemsetAsync(seg_start, 0, (size_t)ncell * 4, st));
    IBT_CUDA_TRY(cudaMemsetAsync(seg_end, 0, (size_t)ncell * 4, st));
    grid_segments_kernel<<<(nk + 255) / 256, 256, 0, st>>>(sorted, nk, seg_start, seg_end);
    grid_reduce_kernel<<<(ncell + 127) / 128, 128, 0, st>>>(u, v, sorted, seg_start, seg_end, ncell, count, sum_u, sum_v);
    return check_launch("ibt_grid_bin");
}
