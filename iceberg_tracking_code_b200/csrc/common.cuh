// Shared helpers of libibt.so (sm_100a only).
#pragma once
#include <cuda.h>              // CUtensorMap (types only; the encoder is fetched through cudaGetDriverEntryPoint)
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/ibt.h"

#define IBT_API extern "C" __attribute__((visibility("default")))

namespace ibt {

void set_last_error(cudaError_t e, const char *where);

inline int check_launch(const char *where)
{
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_last_error(e, where); return IBT_E_CUDA; }
    return IBT_OK;
}

#define IBT_CUDA_TRY(expr)                                                        \
    do {                                                                          \
        cudaError_t e__ = (expr);                                                 \
        if (e__ != cudaSuccess) { ::ibt::set_last_error(e__, #expr); return IBT_E_CUDA; } \
    } while (0)

// REFLECT_101 index for any i (period 2(n-1)).  The common cases (inside, or one reflection) cost a few compares;
// indices further out (tiny images under big windows) take the out-of-line modulo path.
__host__ __device__ __noinline__ inline int r101_far(int i, int n)
{
    if (n == 1) return 0;
    const int p = 2 * (n - 1);
    i %= p;
    if (i < 0) i += p;
    return i < n ? i : p - i;
}
__host__ __device__ __forceinline__ int r101(int i, int n)
{
    if (i >= 0 && i < n) return i;
    if (i < 0) i = -i;                   // -1 -> 1
    if (i < n) return i;
    const int j = 2 * (n - 1) - i;       // n -> n-2
    if (j >= 0) return j;
    return r101_far(i, n);
}

#ifndef IBT_MBAR_SOFT
#define IBT_MBAR_SOFT 0
#endif
// ---- TMA / mbarrier helpers (sm_90+ PTX) -------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity)
{
    const unsigned addr = (unsigned)__cvta_generic_to_shared(bar);
    for (int spin = 0; spin < (1 << 26); spin++) {
        unsigned ok;
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
        if (ok) return;
    }
    if (IBT_MBAR_SOFT) return;
    __trap();                                   // a lost TMA must fail loudly, not hang the GPU
}
__device__ __forceinline__ void tma_load_2d(void *smem_dst, const CUtensorMap *tmap, int c0, int c1, uint64_t *bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(c0), "r"(c1),
                 "r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}
__device__ __forceinline__ void tma_prefetch_map(const CUtensorMap *tmap)     // pull the 128-byte descriptor into the TMA unit's cache
{
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// host: 2-D tiled tensor map (zero fill outside the tensor); false if the driver entry point or the encode fails
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline EncodeTiledFn encode_tiled_fn()
{
    // resolved once per process; a function-local static's initialiser runs exactly once even when host threads race here
    static const EncodeTiledFn fn = [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        EncodeTiledFn f = nullptr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            f = reinterpret_cast<EncodeTiledFn>(p);
        (void)cudaGetLastError();
        return f;
    }();
    return fn;
}
inline bool make_map_2d(CUtensorMap *m, CUtensorMapDataType dt, const void *base, int cols, int rows, int64_t pitch_bytes,
                        int box_cols, int box_rows)
{
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn || reinterpret_cast<uintptr_t>(base) % 16 != 0 || pitch_bytes % 16 != 0 || box_cols > 256 || box_rows > 256) return false;
    const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t gstride[1] = {(cuuint64_t)pitch_bytes};
    const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    return fn(m, dt, 2, const_cast<void *>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// ---- programmatic dependent launch (PDL): the kernels of the per-frame chain (gray -> level 0 -> level 1 -> ...) are launched
// with programmatic stream serialisation: a kernel's CTAs are scheduled and run their prologue while the previous kernel
// drains, and block in pdl_wait() until that kernel has completed and its writes are visible.  pdl_launch_dependents() at the
// top of a kernel lets the next launch start as early as possible.  Both are no-ops for kernels launched the ordinary way.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// ---- CTA-wide exclusive scan of one value per thread (blockDim.x <= 1024, multiple of 32) -------------------------------
__device__ __forceinline__ uint32_t cta_exclusive_scan(uint32_t v, uint32_t *total)
{
    __shared__ uint32_t warp_sums[32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    __syncthreads();                                       // warp_sums may still be read by a previous call
    if (lane == 31) warp_sums[w] = inc;
    __syncthreads();
    uint32_t ws = lane < nw ? warp_sums[lane] : 0u;
    uint32_t wi = ws;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, wi, o);
        if (lane >= o) wi += t;
    }
    const uint32_t wbase = __shfl_sync(0xffffffffu, wi - ws, w);
    if (total) *total = __shfl_sync(0xffffffffu, wi, nw - 1);
    return wbase + inc - v;
}

// scan.cu: device-wide exclusive scan of `rows` rows of n uint32 each, `stride` elements apart (1 <= rows <= 65535).
// in == out is allowed.  total (device, optional) receives the total of each row.  partial: scan_partial_words(n, rows)
// words.  Launch errors are left for the caller's check_launch.
size_t scan_partial_words(int n, int rows);
void launch_scan(const uint32_t *in, uint32_t *out, uint32_t *partial, int n, int rows, int64_t stride, uint32_t *total,
                 cudaStream_t st);

constexpr int kNumSMs = 148;             // B200: 2 dies x 74 SMs

} // namespace ibt
