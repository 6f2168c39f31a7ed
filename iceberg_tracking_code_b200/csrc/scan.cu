// Device-wide exclusive prefix sum of uint32 (modulo 2^32), the one scan of the library: destuff offsets, subsequence
// block bases and per-component DC predictions of the JPEG decoder, survivor offsets of the track compaction, digit
// histograms of the grid binning's radix sort.
//
// A row of up to SCAN_ONE_CTA elements is scanned by one CTA in one launch, 1024 elements per step.  Longer rows take
// three launches: tile sums, a one-CTA scan of the tile sums (which also gives the row total), then every tile scanned
// again with its offset added.  Every thread reads its elements before it writes them, so the scan may run in place.
#include "common.cuh"

namespace ibt {

constexpr int SCAN_TILE = 1024;          // elements per CTA in the tile phases (256 threads x 4)
// longest row scanned by one CTA alone: up to 8 steps, the loop costs less than two more launches (B200 at 1000 W: compaction
// of 0.3 M / 2 M tracks 52 / 77 us, 57 / 81 us with three launches from 1025 elements on)
constexpr int SCAN_ONE_CTA = 8 * 1024;

__global__ void __launch_bounds__(256) scan_reduce_kernel(const uint32_t *__restrict__ in, uint32_t *__restrict__ partial, int n,
                                                          int64_t stride)
{
    const uint32_t *row = in + blockIdx.y * stride;
    const int base = blockIdx.x * SCAN_TILE + threadIdx.x * 4;
    uint32_t s = 0;
#pragma unroll
    for (int j = 0; j < 4; j++)
        if (base + j < n) s += row[base + j];
    uint32_t tot;
    cta_exclusive_scan(s, &tot);
    if (threadIdx.x == 0) partial[blockIdx.y * gridDim.x + blockIdx.x] = tot;
}

// one CTA per row walks the whole row, 1024 elements per step
__global__ void __launch_bounds__(1024) scan_rows_kernel(const uint32_t *in, uint32_t *out, int n, int64_t stride,
                                                         uint32_t *__restrict__ total)
{
    const uint32_t *row = in + blockIdx.x * stride;
    uint32_t *orow = out + blockIdx.x * stride;
    uint32_t carry = 0;
    for (int b = 0; b < n; b += 1024) {
        const int i = b + threadIdx.x;
        const uint32_t v = i < n ? row[i] : 0u;
        uint32_t tot;
        const uint32_t ex = cta_exclusive_scan(v, &tot);
        if (i < n) orow[i] = carry + ex;
        carry += tot;
    }
    if (total && threadIdx.x == 0) total[blockIdx.x] = carry;
}

__global__ void __launch_bounds__(256) scan_apply_kernel(const uint32_t *in, const uint32_t *__restrict__ partial, uint32_t *out,
                                                         int n, int64_t stride)
{
    const uint32_t *row = in + blockIdx.y * stride;
    uint32_t *orow = out + blockIdx.y * stride;
    const int base = blockIdx.x * SCAN_TILE + threadIdx.x * 4;
    uint32_t v[4], s = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) { v[j] = base + j < n ? row[base + j] : 0u; s += v[j]; }
    uint32_t ex = cta_exclusive_scan(s, nullptr) + partial[blockIdx.y * gridDim.x + blockIdx.x];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        if (base + j < n) orow[base + j] = ex;
        ex += v[j];
    }
}

size_t scan_partial_words(int n, int rows)
{
    return n > SCAN_ONE_CTA ? (size_t)rows * ((n + SCAN_TILE - 1) / SCAN_TILE) : 0;
}

void launch_scan(const uint32_t *in, uint32_t *out, uint32_t *partial, int n, int rows, int64_t stride, uint32_t *total,
                 cudaStream_t st)
{
    if (n <= SCAN_ONE_CTA) {
        scan_rows_kernel<<<rows, 1024, 0, st>>>(in, out, n, stride, total);
        return;
    }
    const int ntiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    scan_reduce_kernel<<<dim3(ntiles, rows), 256, 0, st>>>(in, partial, n, stride);
    scan_rows_kernel<<<rows, 1024, 0, st>>>(partial, partial, ntiles, ntiles, total);
    scan_apply_kernel<<<dim3(ntiles, rows), 256, 0, st>>>(in, partial, out, n, stride);
}

} // namespace ibt
