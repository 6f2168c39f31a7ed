// K1: fused pyrDown (5x5 binomial /256) + Scharr derivative for one pyramid level
// (SURVEY.md A.2, A.4).  Replaces the buildOpticalFlowPyramid / calcScharrDeriv work that
// cv2.calcOpticalFlowPyrLK repeats on every call (s1_lucaskanade_tracking.py:323,326).
//
// HBM-bound: per level-l pixel 1 B is read once, 4 B (int16 dx,dy interleaved) and 1/4 B (level l+1) are written.
// Persistent CTAs walk over 128 x (RPW*NW) pixel tiles with a two-stage pipeline (TMA, else cp.async): while the warps filter
// tile t out of one shared-memory buffer, the 16-byte cp.async copies of tile t+1 are in flight into the other
// (tiles touching the left/right image border take a byte path that resolves REFLECT_101; rows reflect by index).
// Each lane slides a 4-pixel-wide strip down RPW rows: per row it reads its word and the two neighbouring words and
// evaluates the horizontal halves of both separable filters with dp4a on funnel-shifted byte windows -- (3,10,3) and
// (-1,0,1) for Scharr, (1,4,6,4,1) for pyrDown -- so no byte is ever unpacked; the vertical halves run on the per-lane
// register history of the previous rows.  Each derivative row leaves as one 16-byte store per lane (512 contiguous
// bytes per warp), each level-(l+1) row as one 2-byte store.  The grid is sized so that every CTA gets the same
// number of tiles (no tail wave).
#include "common.cuh"
#include <cuda.h>
#include <stdlib.h>              // CUtensorMap (types only; the encoder is fetched through cudaGetDriverEntryPoint)

namespace ibt {

constexpr int TW = 128;                 // tile width  (input pixels)
constexpr int HXB = 16;                 // staged bytes left/right of the tile (keeps 16-byte chunks aligned)
constexpr int SPITCH = TW + 2 * HXB;    // 160 bytes per staged row

__device__ __forceinline__ int dp4a_uu(uint32_t a, uint32_t b, int c) { return (int)__dp4a(a, b, (unsigned)c); }
__device__ __forceinline__ int dp4a_us(uint32_t a, int b, int c)
{
    int d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ uint32_t pack_i16(int lo, int hi) { return __byte_perm((uint32_t)lo, (uint32_t)hi, 0x5410); }

// resident CTAs per SM the kernels are compiled for: 4-warp CTAs 7 (register-bound), 1-warp CTAs 24
constexpr int pyr_ctas_per_sm(int nw) { return nw == 4 ? 7 : 24; }

struct PyrArgs {
    const uint8_t *src; int h, w; int64_t pitch;
    uint8_t *deriv; int64_t dpitch;
    uint8_t *down; int64_t downpitch;
    int src_vec_ok, deriv_vec_ok, down_vec_ok;
    int ntx, ntiles;
};

// stage bytes [x0-16, x0+144) of rows y0-2 .. y0+TH into `tile`: every 16-byte chunk that lies inside the row goes
// as cp.async; the columns left of 0 / right of w-1 are filled in later from shared memory itself (reflect_tile)
template <int NW, int RPW>
__device__ __forceinline__ void stage_tile(const PyrArgs &a, int t, uint8_t *tile, int tid)
{
    constexpr int TH = NW * RPW, SROWS = TH + 3, NT = NW * 32;
    const int ty = t / a.ntx, tx = t - ty * a.ntx;
    const int x0 = tx * TW, y0 = ty * TH;
    if (a.src_vec_ok) {
        // thread -> (row r0 + k*RSTEP, chunk c): no division in the loop, one REFLECT_101 row lookup per copy
        constexpr int CH = SPITCH / 16, RSTEP = NT / CH;
        const int r0 = tid / CH, c = tid - r0 * CH;
        const int gx = x0 - HXB + 16 * c;
        if (r0 < RSTEP && gx >= 0 && gx + 16 <= a.pitch) {
            const unsigned sdst = (unsigned)__cvta_generic_to_shared(tile) + 16 * c;
            const uint8_t *g0 = a.src + gx;
#pragma unroll 2
            for (int r = r0; r < SROWS; r += RSTEP) {
                const uint8_t *g = g0 + (int64_t)r101(y0 - 2 + r, a.h) * a.pitch;
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sdst + r * SPITCH), "l"(g) : "memory");
            }
        }
    } else {
        // unaligned image: byte path, only the bytes the filters read (columns x0-4 .. x0+TW+3), REFLECT_101 resolved here
        for (int idx = tid; idx < SROWS * (TW + 8); idx += NT) {
            const int r = idx / (TW + 8), c = idx - r * (TW + 8);
            tile[r * SPITCH + (HXB - 4) + c] = a.src[(int64_t)r101(y0 - 2 + r, a.h) * a.pitch + r101(x0 - 4 + c, a.w)];
        }
    }
}

// REFLECT_101 columns of a staged tile, from the tile itself: -1 -> 1, -2 -> 2, w+k -> w-2-k.  Returns whether it wrote.
template <int NW, int RPW>
__device__ __forceinline__ bool reflect_tile(const PyrArgs &a, int t, uint8_t *tile, int tid)
{
    constexpr int TH = NW * RPW, SROWS = TH + 3, NT = NW * 32;
    const int tx = t % a.ntx;
    const int x0 = tx * TW;
    const bool left = x0 == 0, right = x0 + TW + 4 > a.w;
    if (!a.src_vec_ok || !(left || right)) return false;
    const int org = x0 - HXB;                         // image column of tile byte 0
    for (int r = tid; r < SROWS; r += NT) {
        uint8_t *row = tile + r * SPITCH;
        if (left) {
            row[HXB - 1] = row[HXB + r101(-1, a.w)];
            row[HXB - 2] = row[HXB + r101(-2, a.w)];
        }
        if (right) {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int c = a.w + k;
                if (c - org < SPITCH) {
                    int sc = r101(c, a.w) - org;
                    if (sc < 0) sc = HXB + r101(c, a.w);      // tiny images: fold into the staged range
                    row[c - org] = row[sc];
                }
            }
        }
    }
    return true;
}

// FULL: the tile lies completely inside the image (no per-row / per-column bounds checks)
template <bool DERIV, bool DOWN, int NW, int RPW, bool FULL>
__device__ __forceinline__ void filter_tile(const PyrArgs &a, int t, const uint8_t *tile, int tid)
{
    constexpr int TH = NW * RPW;
    const int ty = t / a.ntx, tx = t - ty * a.ntx;
    const int lane = tid & 31, wy = tid >> 5;
    const int x = tx * TW + 4 * lane;
    const int ybase = ty * TH + RPW * wy;
    const int h = a.h, w = a.w;
    if (!FULL && (x >= w || ybase >= h)) return;
    const int oh = (h + 1) >> 1, ow = (w + 1) >> 1;

    int hx1[4], hx2[4], hs1[4], hs2[4];     // Scharr horizontal halves of the two previous rows
    int hp[4][2];                           // pyrDown horizontal sums of the four previous rows
#pragma unroll
    for (int i = 0; i < 4; i++) { hx1[i] = hx2[i] = hs1[i] = hs2[i] = 0; hp[i][0] = hp[i][1] = 0; }

    const uint32_t *trow = reinterpret_cast<const uint32_t *>(tile + (RPW * wy) * SPITCH + HXB - 4) + lane;
    uint8_t *dp = DERIV ? a.deriv + (int64_t)ybase * a.dpitch + (int64_t)x * 4 : nullptr;
    const bool vec = a.deriv_vec_ok && (FULL || x + 3 < w);
    uint8_t *op = DOWN ? a.down + (int64_t)(ybase >> 1) * a.downpitch + (x >> 1) : nullptr;
    const bool dvec = a.down_vec_ok && (FULL || (x >> 1) + 1 < ow);
#pragma unroll
    for (int j = 0; j <= RPW + 2; j++) {                 // staged rows ybase-2 .. ybase+RPW
        const uint32_t Lw = trow[j * (SPITCH / 4)], O = trow[j * (SPITCH / 4) + 1], Rw = trow[j * (SPITCH / 4) + 2];
        // byte windows: w0 = (x-1..x+2), O = (x..x+3), w2 = (x+1..x+4), w3 = (x+2..x+5)
        const uint32_t w0 = __funnelshift_r(Lw, O, 24);
        const uint32_t w2 = __funnelshift_r(O, Rw, 8);
        const uint32_t w3 = __funnelshift_r(O, Rw, 16);

        if (DERIV && j >= 1) {
            int hx[4], hs[4];
            hs[0] = dp4a_uu(w0, 0x00030A03u, 0); hx[0] = dp4a_us(w0, 0x000100FF, 0);
            hs[1] = dp4a_uu(O, 0x00030A03u, 0);  hx[1] = dp4a_us(O, 0x000100FF, 0);
            hs[2] = dp4a_uu(w2, 0x00030A03u, 0); hx[2] = dp4a_us(w2, 0x000100FF, 0);
            hs[3] = dp4a_uu(w3, 0x00030A03u, 0); hx[3] = dp4a_us(w3, 0x000100FF, 0);
            if (j >= 3) {                                // derivative row of staged row j-1 = image row ybase+j-3
                if (FULL || ybase + j - 3 < h) {
                    uint32_t o[4];
#pragma unroll
                    for (int i = 0; i < 4; i++)
                        o[i] = pack_i16(3 * (hx2[i] + hx[i]) + 10 * hx1[i], hs[i] - hs2[i]);
                    if (vec) {
                        *reinterpret_cast<uint4 *>(dp) = make_uint4(o[0], o[1], o[2], o[3]);
                    } else {
#pragma unroll
                        for (int i = 0; i < 4; i++)
                            if (x + i < w) reinterpret_cast<uint32_t *>(dp)[i] = o[i];
                    }
                }
                dp += a.dpitch;
            }
#pragma unroll
            for (int i = 0; i < 4; i++) { hx2[i] = hx1[i]; hx1[i] = hx[i]; hs2[i] = hs1[i]; hs1[i] = hs[i]; }
        }
        if (DOWN) {
            // output column x/2 is centred on x, x/2+1 on x+2: taps (1,4,6,4,1)
            const uint32_t v0 = __funnelshift_r(Lw, O, 16);               // (x-2 .. x+1)
            const int h0 = dp4a_uu(O, 0x00010000u, dp4a_uu(v0, 0x04060401u, 0));
            const int h1 = dp4a_uu(w3, 0x00010000u, dp4a_uu(O, 0x04060401u, 0));
            if (j >= 4 && (j & 1) == 0) {                // centre row = staged row j-2 = image row ybase+j-4
                if (FULL || ((ybase + j - 4) >> 1) < oh) {
                    const int o0 = (hp[0][0] + h0 + 4 * (hp[1][0] + hp[3][0]) + 6 * hp[2][0] + 128) >> 8;
                    const int o1 = (hp[0][1] + h1 + 4 * (hp[1][1] + hp[3][1]) + 6 * hp[2][1] + 128) >> 8;
                    if (dvec) {
                        *reinterpret_cast<uint16_t *>(op) = (uint16_t)(o0 | (o1 << 8));
                    } else {
                        op[0] = (uint8_t)o0;
                        if ((x >> 1) + 1 < ow) op[1] = (uint8_t)o1;
                    }
                }
                op += a.downpitch;
            }
#pragma unroll
            for (int i = 0; i < 3; i++) { hp[i][0] = hp[i + 1][0]; hp[i][1] = hp[i + 1][1]; }
            hp[3][0] = h0; hp[3][1] = h1;
        }
    }
}

template <bool DERIV, bool DOWN, int NW, int RPW>
__global__ void __launch_bounds__(NW * 32, pyr_ctas_per_sm(NW))
pyr_level_kernel(const __grid_constant__ PyrArgs a)
{
    constexpr int SROWS = NW * RPW + 3;
    __shared__ __align__(16) uint8_t tiles[2][SROWS * SPITCH];
    const int tid = threadIdx.x;
    pdl_launch_dependents();
    pdl_wait();                                           // the source level is the previous launch's output
    int t = blockIdx.x, buf = 0;
    if (t < a.ntiles) stage_tile<NW, RPW>(a, t, tiles[0], tid);
    asm volatile("cp.async.commit_group;" ::: "memory");
    for (; t < a.ntiles; t += gridDim.x) {
        const int tn = t + gridDim.x;
        if (tn < a.ntiles) stage_tile<NW, RPW>(a, tn, tiles[buf ^ 1], tid);       // prefetch the next tile of this CTA
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 1;" ::: "memory");                  // tile t has landed
        __syncthreads();
        if (reflect_tile<NW, RPW>(a, t, tiles[buf], tid)) __syncthreads();
        {
            constexpr int TH = NW * RPW;
            const int ty = t / a.ntx, tx = t - ty * a.ntx;
            const bool full = (tx + 1) * TW <= a.w && (ty + 1) * TH <= a.h;
            if (full) filter_tile<DERIV, DOWN, NW, RPW, true>(a, t, tiles[buf], tid);
            else filter_tile<DERIV, DOWN, NW, RPW, false>(a, t, tiles[buf], tid);
        }
        __syncthreads();                                                      // buffer may be refilled next round
        buf ^= 1;
    }
}


// ---- TMA variant ----------------------------------------------------------------------------------------------
// Same tiles, same filters; the halo tile arrives by ONE cp.async.bulk.tensor.2d per tile (issued by one thread, signalled
// on an mbarrier) instead of per-thread 16-byte cp.async copies: no staging instructions, no per-row index math.  The
// tensor map covers the w x h image; coordinates left / above / right / below it come back as zeros and the
// REFLECT_101 rows and columns are then patched from the tile itself.
// REFLECT_101 rows of a TMA-staged tile (zeros outside the image): rows -2, -1 and h, h+1, copied inside the tile.
template <int NW, int RPW>
__device__ __forceinline__ bool reflect_rows(const PyrArgs &a, int t, uint8_t *tile, int tid)
{
    constexpr int TH = NW * RPW, SROWS = TH + 3, NT = NW * 32;
    const int ty = t / a.ntx;
    const int org = ty * TH - 2;                          // image row of tile row 0
    const bool top = ty == 0, bottom = org + SROWS > a.h;
    if (!(top || bottom)) return false;
    // up to four rows to patch: (dst tile row, src tile row)
    int dst[4], src[4], n = 0;
    if (top) { dst[n] = 0; src[n++] = 4; dst[n] = 1; src[n++] = 3; }
    if (bottom) {
        for (int k = 0; k < 2; k++) {
            const int r = a.h + k - org;
            if (r >= 0 && r < SROWS) { dst[n] = r; src[n++] = a.h - 2 - k - org; }
        }
    }
    for (int i = tid; i < n * (SPITCH / 4); i += NT) {
        const int j = i / (SPITCH / 4), c = i - j * (SPITCH / 4);
        reinterpret_cast<uint32_t *>(tile + dst[j] * SPITCH)[c] = reinterpret_cast<const uint32_t *>(tile + src[j] * SPITCH)[c];
    }
    return true;
}

template <bool DERIV, bool DOWN, int NW, int RPW>
__global__ void __launch_bounds__(NW * 32, pyr_ctas_per_sm(NW))
pyr_level_tma_kernel(const __grid_constant__ PyrArgs a, const __grid_constant__ CUtensorMap tmap)
{
    constexpr int TH = NW * RPW, SROWS = TH + 3;
    constexpr unsigned TILE_BYTES = SROWS * SPITCH;
    constexpr unsigned TILE_ALLOC = (TILE_BYTES + 127) & ~127u;
    __shared__ __align__(128) uint8_t tiles[2][TILE_ALLOC];
    __shared__ __align__(8) uint64_t full[2];
    const int tid = threadIdx.x;
    pdl_launch_dependents();
    if (tid == 0) {
        tma_prefetch_map(&tmap);                          // the descriptor does not depend on the previous launch
        mbar_init(&full[0], 1); mbar_init(&full[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    pdl_wait();                                           // the source level is the previous launch's output
    auto issue = [&](int t, int b) {                      // one thread: arm the barrier, launch the bulk tensor copy
        if (tid == 0) {
            const int ty = t / a.ntx, tx = t - ty * a.ntx;
            fence_proxy_async();                                              // our generic-proxy patches precede the async write
            mbar_expect_tx(&full[b], TILE_BYTES);
            tma_load_2d(tiles[b], &tmap, tx * TW - HXB, ty * TH - 2, &full[b]);
        }
    };
    unsigned phases = 0u;                                 // bit b = parity to wait for on full[b]
    int t = blockIdx.x, buf = 0;
    if (t < a.ntiles) issue(t, 0);
    for (; t < a.ntiles; t += gridDim.x) {
        const int tn = t + gridDim.x;
        if (tn < a.ntiles) issue(tn, buf ^ 1);                                // prefetch the next tile of this CTA
        mbar_wait(&full[buf], (phases >> buf) & 1u);                          // tile t has landed
        phases ^= 1u << buf;
        if (reflect_rows<NW, RPW>(a, t, tiles[buf], tid)) __syncthreads();
        if (reflect_tile<NW, RPW>(a, t, tiles[buf], tid)) __syncthreads();
        {
            const int ty = t / a.ntx, tx = t - ty * a.ntx;
            const bool fullt = (tx + 1) * TW <= a.w && (ty + 1) * TH <= a.h;
            if (fullt) filter_tile<DERIV, DOWN, NW, RPW, true>(a, t, tiles[buf], tid);
            else filter_tile<DERIV, DOWN, NW, RPW, false>(a, t, tiles[buf], tid);
        }
        __syncthreads();                                                      // buffer may be refilled next round
        buf ^= 1;
    }
}

// ---- multi-channel frames (ibt_pyramid_build_multichannel) ------------------------------------------------------------
// A level >= 1 of a cn-channel frame is cn single-channel planes of one geometry, filtered in ONE launch: the tile index also
// selects the channel (tile t = channel t / ntiles, that plane's tile t % ntiles), each plane brings its own PyrArgs and tensor
// map.  Same tiles, helpers and pipelines as pyr_level_kernel / pyr_level_tma_kernel, whose loops are repeated here rather
// than shared: routing the gray kernels through a common body changes their register allocation.
constexpr int PYR_MAX_CN = 4;
struct PyrLevelSet {
    PyrArgs ch[PYR_MAX_CN];
    int cn;
};
struct PyrMapSet { CUtensorMap m[PYR_MAX_CN]; };

__device__ __forceinline__ const PyrArgs &set_tile(const PyrLevelSet &s, int t, int &tc, int &c)
{
    c = t / s.ch[0].ntiles;
    tc = t - c * s.ch[0].ntiles;
    return s.ch[c];
}

template <bool DERIV, bool DOWN, int NW, int RPW>
__global__ void __launch_bounds__(NW * 32, pyr_ctas_per_sm(NW))
pyr_level_set_kernel(const __grid_constant__ PyrLevelSet s)
{
    constexpr int TH = NW * RPW, SROWS = TH + 3;
    __shared__ __align__(16) uint8_t tiles[2][SROWS * SPITCH];
    const int tid = threadIdx.x, ntiles = s.cn * s.ch[0].ntiles;
    pdl_launch_dependents();
    pdl_wait();                                           // the source level is the previous launch's output
    int t = blockIdx.x, buf = 0, tc, c;
    if (t < ntiles) { const PyrArgs &a = set_tile(s, t, tc, c); stage_tile<NW, RPW>(a, tc, tiles[0], tid); }
    asm volatile("cp.async.commit_group;" ::: "memory");
    for (; t < ntiles; t += gridDim.x) {
        const int tn = t + gridDim.x;
        if (tn < ntiles) { const PyrArgs &an = set_tile(s, tn, tc, c); stage_tile<NW, RPW>(an, tc, tiles[buf ^ 1], tid); }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 1;" ::: "memory");                  // tile t has landed
        __syncthreads();
        const PyrArgs &a = set_tile(s, t, tc, c);
        if (reflect_tile<NW, RPW>(a, tc, tiles[buf], tid)) __syncthreads();
        const int ty = tc / a.ntx, tx = tc - ty * a.ntx;
        if ((tx + 1) * TW <= a.w && (ty + 1) * TH <= a.h) filter_tile<DERIV, DOWN, NW, RPW, true>(a, tc, tiles[buf], tid);
        else filter_tile<DERIV, DOWN, NW, RPW, false>(a, tc, tiles[buf], tid);
        __syncthreads();                                                      // buffer may be refilled next round
        buf ^= 1;
    }
}

template <bool DERIV, bool DOWN, int NW, int RPW>
__global__ void __launch_bounds__(NW * 32, pyr_ctas_per_sm(NW))
pyr_level_set_tma_kernel(const __grid_constant__ PyrLevelSet s, const __grid_constant__ PyrMapSet maps)
{
    constexpr int TH = NW * RPW, SROWS = TH + 3;
    constexpr unsigned TILE_BYTES = SROWS * SPITCH;
    constexpr unsigned TILE_ALLOC = (TILE_BYTES + 127) & ~127u;
    __shared__ __align__(128) uint8_t tiles[2][TILE_ALLOC];
    __shared__ __align__(8) uint64_t full[2];
    const int tid = threadIdx.x, ntiles = s.cn * s.ch[0].ntiles;
    pdl_launch_dependents();
    if (tid == 0) {
        for (int c = 0; c < s.cn; c++) tma_prefetch_map(&maps.m[c]);     // the descriptors do not depend on the previous launch
        mbar_init(&full[0], 1); mbar_init(&full[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    pdl_wait();                                           // the source level is the previous launch's output
    auto issue = [&](int t, int b) {                      // one thread: arm the barrier, launch the bulk tensor copy
        if (tid == 0) {
            int tc, c;
            const PyrArgs &a = set_tile(s, t, tc, c);
            const int ty = tc / a.ntx, tx = tc - ty * a.ntx;
            fence_proxy_async();                                              // our generic-proxy patches precede the async write
            mbar_expect_tx(&full[b], TILE_BYTES);
            tma_load_2d(tiles[b], &maps.m[c], tx * TW - HXB, ty * TH - 2, &full[b]);
        }
    };
    unsigned phases = 0u;                                 // bit b = parity to wait for on full[b]
    int t = blockIdx.x, buf = 0;
    if (t < ntiles) issue(t, 0);
    for (; t < ntiles; t += gridDim.x) {
        const int tn = t + gridDim.x;
        if (tn < ntiles) issue(tn, buf ^ 1);                                  // prefetch the next tile of this CTA
        mbar_wait(&full[buf], (phases >> buf) & 1u);                          // tile t has landed
        phases ^= 1u << buf;
        int tc, c;
        const PyrArgs &a = set_tile(s, t, tc, c);
        if (reflect_rows<NW, RPW>(a, tc, tiles[buf], tid)) __syncthreads();
        if (reflect_tile<NW, RPW>(a, tc, tiles[buf], tid)) __syncthreads();
        const int ty = tc / a.ntx, tx = tc - ty * a.ntx;
        if ((tx + 1) * TW <= a.w && (ty + 1) * TH <= a.h) filter_tile<DERIV, DOWN, NW, RPW, true>(a, tc, tiles[buf], tid);
        else filter_tile<DERIV, DOWN, NW, RPW, false>(a, tc, tiles[buf], tid);
        __syncthreads();                                                      // buffer may be refilled next round
        buf ^= 1;
    }
}

// Level 0 of a cn-channel frame: the interleaved (H,W,cn) u8 frame is read once, at any pitch and alignment, and every channel
// gets its level-0 plane, its Scharr planes and its level-1 plane.  Tiles of 128 x 32 pixels (4 warps x 8 rows; a 128 x 64
// tile of 4 channels would not leave room for two CTAs per SM).  16-byte aligned frames (base and pitch) stage the interleaved
// halo tile by cp.async, zero-filling past the end of the row, and de-interleave it once into the cn single-channel tiles that
// filter_tile reads; the REFLECT_101 columns are then patched per channel by reflect_tile.  Any other frame takes the byte
// path, which gathers the pixels channel by channel with REFLECT_101 resolved on load (as pyr_level_kernel does).  The
// interleaved buffer is refilled with the next tile while the channels of this one are filtered.
constexpr int F_NW = 4, F_RPW = 8, F_TH = F_NW * F_RPW, F_SROWS = F_TH + 3;
struct PyrFrameArgs {
    PyrArgs ch[PYR_MAX_CN];         // per channel: its level-0 plane (h, w, pitch), Scharr planes, level-1 plane
    uint8_t *plane[PYR_MAX_CN];     // = ch[c].src, written here
    const uint8_t *frame; int64_t fpitch;
    int frame_vec_ok;               // 16-byte aligned base and pitch: cp.async staging
    int plane_vec_ok;               // every plane has a 4-byte aligned base and pitch: word stores
};

template <int CN>
__device__ __forceinline__ void stage_frame(const PyrFrameArgs &f, int t, uint8_t *stage, int tid)
{
    constexpr int FP = SPITCH * CN, CH = FP / 16, RSTEP = F_NW * 32 / CH;
    const PyrArgs &a = f.ch[0];
    const int ty = t / a.ntx, tx = t - ty * a.ntx;
    const int r0 = tid / CH, c = tid - r0 * CH;
    const int64_t gx = (int64_t)(tx * TW - HXB) * CN + 16 * c, rowb = (int64_t)a.w * CN;
    if (r0 >= RSTEP || gx < 0 || gx >= rowb) return;
    const unsigned n = gx + 16 <= rowb ? 16u : (unsigned)(rowb - gx);       // the rest of the chunk is zero-filled
    const unsigned sdst = (unsigned)__cvta_generic_to_shared(stage) + 16 * c;
    const uint8_t *g0 = f.frame + gx;
    for (int r = r0; r < F_SROWS; r += RSTEP) {
        const uint8_t *g = g0 + (int64_t)r101(ty * F_TH - 2 + r, a.h) * f.fpitch;
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(sdst + r * FP), "l"(g), "r"(n) : "memory");
    }
}

// interleaved staged rows -> CN tiles of the single-channel layout, four pixels (CN words in, one word per channel out) a step
template <int CN>
__device__ __forceinline__ void deinterleave(const uint8_t *stage, uint8_t (*tiles)[F_SROWS * SPITCH], int tid)
{
    constexpr int Q = SPITCH / 4;
    for (int i = tid; i < F_SROWS * Q; i += F_NW * 32) {
        const int r = i / Q, q = i - r * Q;
        const uint32_t *src = reinterpret_cast<const uint32_t *>(stage + r * SPITCH * CN) + q * CN;
        uint32_t w[CN];
#pragma unroll
        for (int k = 0; k < CN; k++) w[k] = src[k];
#pragma unroll
        for (int c = 0; c < CN; c++) {
            uint32_t o = 0;
#pragma unroll
            for (int p = 0; p < 4; p++) {
                const int b = p * CN + c;
                o |= ((w[b >> 2] >> (8 * (b & 3))) & 0xffu) << (8 * p);
            }
            reinterpret_cast<uint32_t *>(tiles[c] + r * SPITCH)[q] = o;
        }
    }
}

// byte path: pixel columns x0-4 .. x0+TW+3 of every channel, REFLECT_101 resolved here
template <int CN>
__device__ __forceinline__ void gather_frame(const PyrFrameArgs &f, int t, uint8_t (*tiles)[F_SROWS * SPITCH], int tid)
{
    const PyrArgs &a = f.ch[0];
    const int ty = t / a.ntx, tx = t - ty * a.ntx;
    for (int idx = tid; idx < F_SROWS * (TW + 8); idx += F_NW * 32) {
        const int r = idx / (TW + 8), c = idx - r * (TW + 8);
        const uint8_t *g = f.frame + (int64_t)r101(ty * F_TH - 2 + r, a.h) * f.fpitch + (int64_t)r101(tx * TW - 4 + c, a.w) * CN;
#pragma unroll
        for (int k = 0; k < CN; k++) tiles[k][r * SPITCH + (HXB - 4) + c] = g[k];
    }
}

// this warp's rows of the level-0 plane, straight from the channel tile
__device__ __forceinline__ void store_plane(const PyrArgs &a, uint8_t *plane, bool vec, int t, const uint8_t *tile, int tid)
{
    const int ty = t / a.ntx, tx = t - ty * a.ntx;
    const int lane = tid & 31, wy = tid >> 5;
    const int x = tx * TW + 4 * lane, y0 = ty * F_TH + F_RPW * wy;
    if (x >= a.w) return;
    const uint8_t *s = tile + (F_RPW * wy + 2) * SPITCH + HXB + 4 * lane;
    uint8_t *p = plane + (int64_t)y0 * a.pitch + x;
    for (int j = 0; j < F_RPW && y0 + j < a.h; j++, s += SPITCH, p += a.pitch) {
        if (vec && x + 3 < a.w) {
            *reinterpret_cast<uint32_t *>(p) = *reinterpret_cast<const uint32_t *>(s);
        } else {
            for (int i = 0; i < 4 && x + i < a.w; i++) p[i] = s[i];
        }
    }
}

template <int CN, bool DERIV, bool DOWN>
__global__ void __launch_bounds__(F_NW * 32)
pyr_frame_kernel(const __grid_constant__ PyrFrameArgs f)
{
    __shared__ __align__(16) uint8_t stage[F_SROWS * SPITCH * CN];           // interleaved rows of the next tile
    __shared__ __align__(16) uint8_t tiles[CN][F_SROWS * SPITCH];
    const int tid = threadIdx.x, ntiles = f.ch[0].ntiles;
    const bool vec = f.frame_vec_ok != 0;
    pdl_launch_dependents();
    pdl_wait();                                           // the frame may be the previous launch's output
    int t = blockIdx.x;
    if (vec && t < ntiles) stage_frame<CN>(f, t, stage, tid);
    asm volatile("cp.async.commit_group;" ::: "memory");
    for (; t < ntiles; t += gridDim.x) {
        if (vec) {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
            __syncthreads();                              // tile t has landed; the channel tiles of t - grid are consumed
            deinterleave<CN>(stage, tiles, tid);
            __syncthreads();                              // the interleaved buffer is free again
            if (t + gridDim.x < ntiles) stage_frame<CN>(f, t + gridDim.x, stage, tid);
            asm volatile("cp.async.commit_group;" ::: "memory");
            bool patched = false;
#pragma unroll
            for (int c = 0; c < CN; c++) patched |= reflect_tile<F_NW, F_RPW>(f.ch[c], t, tiles[c], tid);
            if (patched) __syncthreads();
        } else {
            __syncthreads();                              // the channel tiles of t - grid are consumed
            gather_frame<CN>(f, t, tiles, tid);
            __syncthreads();
        }
        const PyrArgs &a0 = f.ch[0];
        const int ty = t / a0.ntx, tx = t - ty * a0.ntx;
        const bool full = (tx + 1) * TW <= a0.w && (ty + 1) * F_TH <= a0.h;
#pragma unroll
        for (int c = 0; c < CN; c++) {
            store_plane(f.ch[c], f.plane[c], f.plane_vec_ok != 0, t, tiles[c], tid);
            if (DERIV || DOWN) {
                if (full) filter_tile<DERIV, DOWN, F_NW, F_RPW, true>(f.ch[c], t, tiles[c], tid);
                else filter_tile<DERIV, DOWN, F_NW, F_RPW, false>(f.ch[c], t, tiles[c], tid);
            }
        }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}

static bool make_tile_map(CUtensorMap *m, const uint8_t *src, int h, int w, int64_t pitch, int srows)
{
    return make_map_2d(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, src, w, h, pitch, SPITCH, srows);
}

template <bool DERIV, bool DOWN, int NW, int RPW>
static void launch_variant(const PyrArgs &a0, cudaStream_t st)
{
    PyrArgs a = a0;
    constexpr int TH = NW * RPW;
    a.ntx = (a.w + TW - 1) / TW;
    a.ntiles = a.ntx * ((a.h + TH - 1) / TH);
    // persistent CTAs, every CTA the same number of tiles: no partial last wave
    const int resident = kNumSMs * pyr_ctas_per_sm(NW);
    const int per_cta = (a.ntiles + resident - 1) / resident;
    const int blocks = (a.ntiles + per_cta - 1) / per_cta;
    // TMA staging needs a 16-byte aligned image and enough rows / columns for the in-tile reflections
    static const bool no_tma = getenv("IBT_NO_TMA") != nullptr;
    CUtensorMap tmap;
    if (!no_tma && a.src_vec_ok && a.h >= 8 && a.w >= 16 && make_tile_map(&tmap, a.src, a.h, a.w, a.pitch, TH + 3)) {
        (void)launch_pdl(pyr_level_tma_kernel<DERIV, DOWN, NW, RPW>, dim3(blocks), dim3(NW * 32), 0, st, a, tmap);
        return;
    }
    (void)launch_pdl(pyr_level_kernel<DERIV, DOWN, NW, RPW>, dim3(blocks), dim3(NW * 32), 0, st, a);
}

// checks one level step's arguments and fills its PyrArgs (ntx / ntiles are set by the launcher)
static int level_args(const uint8_t *src, int h, int w, int64_t pitch, int16_t *deriv, int64_t dpitch, uint8_t *down,
                      int64_t downpitch, PyrArgs &a)
{
    if (!src || h <= 0 || w <= 0 || pitch < w) return IBT_E_INVALID;
    if (deriv && (dpitch < (int64_t)w * 4 || dpitch % 4 != 0 || reinterpret_cast<uintptr_t>(deriv) % 4 != 0))
        return IBT_E_INVALID;
    if (down && downpitch < (w + 1) / 2) return IBT_E_INVALID;
    a.src = src; a.h = h; a.w = w; a.pitch = pitch;
    a.deriv = reinterpret_cast<uint8_t *>(deriv); a.dpitch = dpitch;
    a.down = down; a.downpitch = downpitch;
    a.src_vec_ok = (reinterpret_cast<uintptr_t>(src) % 16 == 0) && (pitch % 16 == 0);
    a.deriv_vec_ok = deriv && (reinterpret_cast<uintptr_t>(deriv) % 16 == 0) && (dpitch % 16 == 0);
    a.down_vec_ok = down && (reinterpret_cast<uintptr_t>(down) % 2 == 0) && (downpitch % 2 == 0);
    a.ntx = a.ntiles = 0;
    return IBT_OK;
}

static int launch_level(const uint8_t *src, int h, int w, int64_t pitch, int16_t *deriv, int64_t dpitch,
                        uint8_t *down, int64_t downpitch, cudaStream_t st)
{
    if (!src || h <= 0 || w <= 0 || pitch < w) return IBT_E_INVALID;
    if (!deriv && !down) return IBT_OK;
    PyrArgs a;
    const int rc = level_args(src, h, w, pitch, deriv, dpitch, down, downpitch, a);
    if (rc != IBT_OK) return rc;
    // big levels: 128 x 64 tiles (4 warps x 16 rows).  Smaller levels are latency-bound -- a launch lasts as long as one warp
    // needs for its rows -- so they take 1-warp tiles of 4 rows: every SM gets work and no warp walks more than 7 rows
    const bool big = (int64_t)((w + TW - 1) / TW) * ((h + 63) / 64) >= 2 * kNumSMs;
    if (deriv && down) { if (big) launch_variant<true, true, 4, 16>(a, st); else launch_variant<true, true, 1, 4>(a, st); }
    else if (deriv)    { if (big) launch_variant<true, false, 4, 16>(a, st); else launch_variant<true, false, 1, 4>(a, st); }
    else               { if (big) launch_variant<false, true, 4, 16>(a, st); else launch_variant<false, true, 1, 4>(a, st); }
    return check_launch("ibt_pyr_level_u8");
}

// one level of all cn channel planes in one launch (the tile choice of launch_level, counted over the channels)
template <bool DERIV, bool DOWN, int NW, int RPW>
static void launch_set_variant(PyrLevelSet &s, cudaStream_t st)
{
    constexpr int TH = NW * RPW;
    bool tma = getenv("IBT_NO_TMA") == nullptr;
    static thread_local PyrMapSet maps;
    for (int c = 0; c < s.cn; c++) {
        PyrArgs &a = s.ch[c];
        a.ntx = (a.w + TW - 1) / TW;
        a.ntiles = a.ntx * ((a.h + TH - 1) / TH);
        tma = tma && a.src_vec_ok && a.h >= 8 && a.w >= 16 && make_tile_map(&maps.m[c], a.src, a.h, a.w, a.pitch, TH + 3);
    }
    const int ntiles = s.cn * s.ch[0].ntiles;
    const int resident = kNumSMs * pyr_ctas_per_sm(NW);
    const int per_cta = (ntiles + resident - 1) / resident;
    const int blocks = (ntiles + per_cta - 1) / per_cta;
    if (tma) (void)launch_pdl(pyr_level_set_tma_kernel<DERIV, DOWN, NW, RPW>, dim3(blocks), dim3(NW * 32), 0, st, s, maps);
    else (void)launch_pdl(pyr_level_set_kernel<DERIV, DOWN, NW, RPW>, dim3(blocks), dim3(NW * 32), 0, st, s);
}

static void launch_level_set(PyrLevelSet &s, cudaStream_t st)
{
    const PyrArgs &a = s.ch[0];
    const bool deriv = a.deriv != nullptr, down = a.down != nullptr;
    const bool big = (int64_t)((a.w + TW - 1) / TW) * ((a.h + 63) / 64) * s.cn >= 2 * kNumSMs;
    if (deriv && down) { if (big) launch_set_variant<true, true, 4, 16>(s, st); else launch_set_variant<true, true, 1, 4>(s, st); }
    else if (deriv)    { if (big) launch_set_variant<true, false, 4, 16>(s, st); else launch_set_variant<true, false, 1, 4>(s, st); }
    else               { if (big) launch_set_variant<false, true, 4, 16>(s, st); else launch_set_variant<false, true, 1, 4>(s, st); }
}

template <int CN, bool DERIV, bool DOWN>
static void launch_frame_variant(const PyrFrameArgs &f, int ntiles, cudaStream_t st)
{
    static int per_sm[64] = {0};                          // resident CTAs per SM, per device (shared memory grows with CN)
    int dev = 0;
    (void)cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) dev = 0;
    if (per_sm[dev] == 0) {
        int n = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, pyr_frame_kernel<CN, DERIV, DOWN>, F_NW * 32, 0) != cudaSuccess || n < 1)
            n = 1;
        per_sm[dev] = n;
    }
    const int resident = kNumSMs * per_sm[dev];
    const int per_cta = (ntiles + resident - 1) / resident;
    const int blocks = (ntiles + per_cta - 1) / per_cta;
    (void)launch_pdl(pyr_frame_kernel<CN, DERIV, DOWN>, dim3(blocks), dim3(F_NW * 32), 0, st, f);
}

template <int CN>
static void launch_frame(const PyrFrameArgs &f, int ntiles, cudaStream_t st)
{
    const bool deriv = f.ch[0].deriv != nullptr, down = f.ch[0].down != nullptr;
    if (deriv && down) launch_frame_variant<CN, true, true>(f, ntiles, st);
    else if (deriv)    launch_frame_variant<CN, true, false>(f, ntiles, st);
    else if (down)     launch_frame_variant<CN, false, true>(f, ntiles, st);
    else               launch_frame_variant<CN, false, false>(f, ntiles, st);
}

static int build_multichannel(const uint8_t *frame, int64_t fpitch, int cn, const ibt_pyramid_t *const *pyr, int with_derivs,
                              cudaStream_t st)
{
    if (!frame || cn < 2 || cn > PYR_MAX_CN || !pyr) return IBT_E_INVALID;
    for (int c = 0; c < cn; c++)
        if (!pyr[c]) return IBT_E_INVALID;
    const ibt_pyramid_t &p0 = *pyr[0];
    const int L = p0.nlevels;
    if (L < 1 || L > IBT_MAX_LEVELS || p0.rows[0] <= 0 || p0.cols[0] <= 0 || fpitch < (int64_t)p0.cols[0] * cn)
        return IBT_E_INVALID;
    for (int c = 0; c < cn; c++) {
        const ibt_pyramid_t &p = *pyr[c];
        if (p.nlevels != L) return IBT_E_INVALID;
        for (int l = 0; l < L; l++) {
            if (p.rows[l] != p0.rows[l] || p.cols[l] != p0.cols[l] || !p.img[l]) return IBT_E_INVALID;
            if (l + 1 < L && (p.rows[l + 1] != (p.rows[l] + 1) / 2 || p.cols[l + 1] != (p.cols[l] + 1) / 2)) return IBT_E_INVALID;
            if (with_derivs && !p.deriv[l]) return IBT_E_INVALID;
        }
    }
    // every level's arguments are checked before the first launch
    PyrFrameArgs f;
    static thread_local PyrLevelSet sets[IBT_MAX_LEVELS];
    f.frame = frame; f.fpitch = fpitch;
    f.frame_vec_ok = (reinterpret_cast<uintptr_t>(frame) % 16 == 0) && (fpitch % 16 == 0);
    f.plane_vec_ok = 1;
    for (int l = 0; l < L; l++) {
        sets[l].cn = cn;
        for (int c = 0; c < cn; c++) {
            const ibt_pyramid_t &p = *pyr[c];
            const bool last = l + 1 == L;
            PyrArgs &a = l == 0 ? f.ch[c] : sets[l].ch[c];
            const int rc = level_args(p.img[l], p.rows[l], p.cols[l], p.img_pitch[l],
                                      with_derivs ? const_cast<int16_t *>(p.deriv[l]) : nullptr, with_derivs ? p.deriv_pitch[l] : 0,
                                      last ? nullptr : const_cast<uint8_t *>(p.img[l + 1]), last ? 0 : p.img_pitch[l + 1], a);
            if (rc != IBT_OK) return rc;
        }
    }
    const int ntx = (p0.cols[0] + TW - 1) / TW, ntiles = ntx * ((p0.rows[0] + F_TH - 1) / F_TH);
    for (int c = 0; c < cn; c++) {
        PyrArgs &a = f.ch[c];
        f.plane[c] = const_cast<uint8_t *>(a.src);
        f.plane_vec_ok &= (reinterpret_cast<uintptr_t>(a.src) % 4 == 0) && (a.pitch % 4 == 0);
        a.src_vec_ok = f.frame_vec_ok;                    // reflect_tile: REFLECT_101 columns are patched in the tile
        a.ntx = ntx; a.ntiles = ntiles;
    }
    if (cn == 2) launch_frame<2>(f, ntiles, st);
    else if (cn == 3) launch_frame<3>(f, ntiles, st);
    else launch_frame<4>(f, ntiles, st);
    for (int l = 1; l < L; l++)
        if (with_derivs || l + 1 < L) launch_level_set(sets[l], st);
    return check_launch("ibt_pyramid_build_multichannel");
}

} // namespace ibt

IBT_API int ibt_pyramid_levels(int H, int W, int winW, int winH, int maxLevel, int *sizes_hw)
{
    if (H <= 0 || W <= 0 || maxLevel < 0 || maxLevel >= IBT_MAX_LEVELS || !sizes_hw) return IBT_E_INVALID;
    int l = 0, h = H, w = W;
    sizes_hw[0] = h; sizes_hw[1] = w;
    while (l < maxLevel) {
        const int nh = (h + 1) / 2, nw = (w + 1) / 2;
        if (!(nw > winW && nh > winH)) break;
        h = nh; w = nw; ++l;
        sizes_hw[2 * l] = h; sizes_hw[2 * l + 1] = w;
    }
    return l;
}

IBT_API int ibt_pyr_level_u8(const uint8_t *src, int h, int w, int64_t src_pitch, int16_t *deriv, int64_t deriv_pitch,
                             uint8_t *down, int64_t down_pitch, void *stream)
{
    return ibt::launch_level(src, h, w, src_pitch, deriv, deriv_pitch, down, down_pitch, static_cast<cudaStream_t>(stream));
}

IBT_API int ibt_pyramid_build(const ibt_pyramid_t *pyr, int with_derivs, void *stream)
{
    if (!pyr || pyr->nlevels < 1 || pyr->nlevels > IBT_MAX_LEVELS) return IBT_E_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    for (int l = 0; l < pyr->nlevels; l++) {
        const bool last = (l + 1 == pyr->nlevels);
        if (!last && (pyr->rows[l + 1] != (pyr->rows[l] + 1) / 2 || pyr->cols[l + 1] != (pyr->cols[l] + 1) / 2))
            return IBT_E_INVALID;
        int16_t *d = with_derivs ? const_cast<int16_t *>(pyr->deriv[l]) : nullptr;
        if (with_derivs && !d) return IBT_E_INVALID;
        uint8_t *dn = last ? nullptr : const_cast<uint8_t *>(pyr->img[l + 1]);
        if (!last && !dn) return IBT_E_INVALID;
        int rc = ibt::launch_level(pyr->img[l], pyr->rows[l], pyr->cols[l], pyr->img_pitch[l], d,
                                   with_derivs ? pyr->deriv_pitch[l] : 0, dn, last ? 0 : pyr->img_pitch[l + 1], st);
        if (rc != IBT_OK) return rc;
    }
    return IBT_OK;
}

IBT_API int ibt_pyramid_build_multichannel(const uint8_t *frame, int64_t frame_pitch, int cn, const ibt_pyramid_t *const *pyr,
                                           int with_derivs, void *stream)
{
    return ibt::build_multichannel(frame, frame_pitch, cn, pyr, with_derivs, static_cast<cudaStream_t>(stream));
}
