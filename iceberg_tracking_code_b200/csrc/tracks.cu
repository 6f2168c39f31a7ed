// Track bookkeeping at a group boundary (s1_lucaskanade_tracking.py:340-359, 362-395): the reference keeps
// tracks as Python lists and drops a track the first time its forward-backward distance reaches 1 px; here the
// group's vertices live in time-major device arrays plus an alive mask, and the survivors are compacted once,
// in seed order, into the (M, T+1, 2) / (M, T) float32 arrays that np.savez writes (SURVEY.md A.8).
#include "common.cuh"

namespace ibt {

constexpr int CB = 256;

__global__ void __launch_bounds__(CB)
alive_count_kernel(const uint8_t *__restrict__ alive, int n, int32_t *__restrict__ block_counts)
{
    const int i = blockIdx.x * CB + threadIdx.x;
    const int c = __syncthreads_count(i < n && alive[i] != 0);
    if (threadIdx.x == 0) block_counts[blockIdx.x] = c;
}

__global__ void __launch_bounds__(CB)
tracks_scatter_kernel(const float2 *__restrict__ tracks_tm, const float *__restrict__ quality_tm,
                      const uint8_t *__restrict__ alive, int n, int T, const int32_t *__restrict__ block_off,
                      float2 *__restrict__ out_tracks, float *__restrict__ out_quality)
{
    __shared__ int32_t wbase[CB / 32];
    const int i = blockIdx.x * CB + threadIdx.x;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const bool a = i < n && alive[i] != 0;
    const uint32_t ballot = __ballot_sync(0xffffffffu, a);
    if (lane == 0) wbase[wid] = __popc(ballot);
    __syncthreads();
    if (threadIdx.x == 0) {
        int32_t run = block_off[blockIdx.x];
        for (int w = 0; w < CB / 32; w++) { const int32_t c = wbase[w]; wbase[w] = run; run += c; }
    }
    __syncthreads();
    if (!a) return;
    const int64_t m = wbase[wid] + __popc(ballot & ((1u << lane) - 1));
    for (int t = 0; t <= T; t++) out_tracks[m * (T + 1) + t] = tracks_tm[(int64_t)t * n + i];
    for (int t = 0; t < T; t++) out_quality[m * T + t] = quality_tm[(int64_t)t * n + i];
}

} // namespace ibt

static int tracks_compact_enqueue(const float *tracks_tm, const float *quality_tm, const uint8_t *alive, int N, int T,
                                  int32_t *scratch, float *out_tracks, float *out_quality, cudaStream_t st)
{
    using namespace ibt;
    if (!tracks_tm || !quality_tm || !alive || !scratch || !out_tracks || !out_quality ||
        reinterpret_cast<uintptr_t>(tracks_tm) % 8 != 0 || reinterpret_cast<uintptr_t>(out_tracks) % 8 != 0)
        return IBT_E_INVALID;
    // scratch: (N + 1) words, block counts -> block offsets in [0, nb), survivor count at [N].  The scan's partial sums, when
    // it needs any (ceil(nb / 1024) words), fit in [nb, N): N > 256 * (nb - 1).
    const int nb = (N + CB - 1) / CB;
    uint32_t *counts = reinterpret_cast<uint32_t *>(scratch);
    alive_count_kernel<<<nb, CB, 0, st>>>(alive, N, scratch);
    launch_scan(counts, counts, counts + nb, nb, 1, 0, counts + N, st);
    tracks_scatter_kernel<<<nb, CB, 0, st>>>(reinterpret_cast<const float2 *>(tracks_tm), quality_tm, alive, N, T, scratch,
                                             reinterpret_cast<float2 *>(out_tracks), out_quality);
    return check_launch("ibt_tracks_compact");
}

IBT_API int ibt_tracks_compact(const float *tracks_tm, const float *quality_tm, const uint8_t *alive, int N, int T,
                               int32_t *scratch, float *out_tracks, float *out_quality, int *out_count, void *stream)
{
    using namespace ibt;
    if (N < 0 || T < 1 || !out_count) return IBT_E_INVALID;
    *out_count = 0;
    if (N == 0) return IBT_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int rc = tracks_compact_enqueue(tracks_tm, quality_tm, alive, N, T, scratch, out_tracks, out_quality, st);
    if (rc) return rc;
    int32_t total = 0;
    IBT_CUDA_TRY(cudaMemcpyAsync(&total, scratch + N, sizeof(total), cudaMemcpyDeviceToHost, st));
    IBT_CUDA_TRY(cudaStreamSynchronize(st));
    *out_count = total;
    return IBT_OK;
}

IBT_API int ibt_tracks_compact_async(const float *tracks_tm, const float *quality_tm, const uint8_t *alive, int N, int T,
                                     int32_t *scratch, float *out_tracks, float *out_quality, void *stream)
{
    if (N < 1 || T < 1) return IBT_E_INVALID;
    return tracks_compact_enqueue(tracks_tm, quality_tm, alive, N, T, scratch, out_tracks, out_quality,
                                  static_cast<cudaStream_t>(stream));
}
