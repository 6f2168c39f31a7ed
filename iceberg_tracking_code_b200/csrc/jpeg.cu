// K5: baseline JPEG -> RGB / gray on the GPU (SURVEY.md 8a row a1, 8f rank 1).
// Replaces `np.array(Image.open(image))` (+ the cv2.cvtColor that follows it) at s1_lucaskanade_tracking.py:310-311,
// s0_1_test_lucaskanade_tracking.py:79-80: Pillow's bundled libjpeg-turbo with default settings (islow IDCT, fancy
// upsampling, 16-bit fixed-point YCbCr->RGB), reproduced bit for bit.  The file travels to the GPU compressed
// (a few MB instead of 72 MB of RGB per 24 MP frame) and the tracker consumes the gray plane in place.
//
//   destuff       remove the 0x00 after every 0xFF of the entropy-coded segment (count / scan / write); bytes are stored
//                 so that a 32-bit load returns them in bit-stream (big-endian) order
//   Huffman       decoded speculatively (restart markers, if any, are not needed for parallelism): thread i owns bits
//                 [i*S, (i+1)*S) and starts from a guessed decoder state (see jpg_sync_probe for the guess).  Huffman
//                 streams self-synchronise: after a few symbols a decoder that started in the wrong state is in the
//                 right one.  Rounds: every thread whose entry state changed decodes its subsequence again and hands its
//                 exit state (bit position, block in MCU, zig-zag index) to its successor, until nothing changes
//                 (thread 0's entry state is exact, so the fixed point is the sequential decode: correctness never
//                 depends on self-synchronisation, only the number of rounds does).  Then an exclusive scan of the
//                 blocks completed per subsequence gives every thread its output block, and one more pass writes the
//                 coefficients (natural order, int16; DC still differential).
//   DC            per-component prefix sum of the DC differences over MCUs (scan) + within the MCU (IDCT kernel)
//   IDCT          one thread per 8x8 block in PLANE order (a warp stores 256 contiguous bytes per row): dequantise,
//                 libjpeg "islow" integer IDCT in registers, saturate to u8
//   colour        8 pixels per thread, one kernel per sampling mode: fancy h2v2 / h2v1 chroma upsampling, YCbCr->RGB,
//                 optional fused cvtColor gray
#include "common.cuh"
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <atomic>

namespace ibt {

// subsequence length S = 2^sbits stream bits per decoder thread, chosen per file (jpeg_sbits): every pass costs the latency
// of one thread walking S bits, dense files need ~15 kbit / S repair rounds, sparse files have too few subsequences at a large S
constexpr int JPG_LUT_BITS = 10;
constexpr int JPG_Q = 4;                 // pieces per subsequence in the coefficient pass
constexpr int JPG_CHUNK = 4096;          // destuff: bytes per CTA (256 threads x 16)

struct __align__(16) JpgTables {          // device copy in the workspace (~27 KB): one (DC, AC) table pair per component
    uint32_t lut[6][1 << JPG_LUT_BITS];  // [comp*2 + ac]: symbol | len << 8 | (len + extra bits) << 16; 0 = longer code
    uint32_t limit[6][17];               // left-justified 16-bit value of the first code longer than l
    int32_t valoff[6][17];               // vals index = valoff[l] + (w16 >> (16 - l))
    uint8_t vals[6][256];
    uint8_t blk_comp[16];
    int nblk_mcu;
    uint32_t compmap;                    // component of block b of the MCU in bits [2b, 2b+1]
    uint32_t pad[2];
};

struct JpgGeom {
    int ncomp, W, H;
    int hs[3], vs[3], blkoff[3];
    int mcux, mcuy, nblk_mcu;
    int bw[3], bh[3];                    // blocks per plane row / column
    int pw[3], ph[3];                    // plane size (samples, whole blocks)
    int dw[3], dh[3];                    // real downsampled size
    int hmax, vmax;
    int hsub[3], vsub[3];                // hmax / hs[c], vmax / vs[c] (1 or 2)
    int restart_interval;                // MCUs per restart interval (0 = none): DC predictions restart there
    uint8_t *plane[3];
    uint16_t quant[3][64];               // per component, natural order
};

__constant__ uint8_t c_zigzag[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                     41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                     30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

// ---- destuff ------------------------------------------------------------------------------------------------
// byte j of the segment is dropped iff it is the 0x00 that follows a 0xFF, or belongs to an RSTn marker (FF D0..D7);
// rmask marks the first byte of each RSTn marker (the next restart interval starts at the output position reached there)
__device__ __forceinline__ uint32_t destuff_keepmask(const uint8_t *__restrict__ src, int64_t n, int64_t j0, uint8_t *b, uint32_t &rmask)
{
    uint32_t keep = 0;
    rmask = 0;
    uint8_t prev = j0 > 0 && j0 <= n ? src[j0 - 1] : 0;
    uint8_t c = j0 < n ? src[j0] : 0;
#pragma unroll
    for (int j = 0; j < 16; j++) {
        const int64_t g = j0 + j;
        const uint8_t nx = g + 1 < n ? src[g + 1] : 0;
        b[j] = c;
        const bool stuffing = c == 0x00 && prev == 0xFF;
        const bool rst0 = c == 0xFF && nx >= 0xD0 && nx <= 0xD7;
        const bool rst1 = prev == 0xFF && c >= 0xD0 && c <= 0xD7;
        if (g < n && !(stuffing || rst0 || rst1)) keep |= 1u << j;
        if (g < n && rst0) rmask |= 1u << j;
        prev = c;
        c = nx;
    }
    return keep;
}
__global__ void __launch_bounds__(256) jpg_destuff_count(const uint8_t *__restrict__ src, int64_t n, uint32_t *__restrict__ counts)
{
    uint8_t b[16];
    uint32_t rmask;
    const int64_t j0 = (int64_t)blockIdx.x * JPG_CHUNK + threadIdx.x * 16;
    const uint32_t keep = destuff_keepmask(src, n, j0, b, rmask);
    uint32_t tot;
    cta_exclusive_scan(__popc(keep), &tot);
    if (threadIdx.x == 0) counts[blockIdx.x] = tot;
}
// dst byte k lives at address k ^ 3: a 32-bit load then holds four stream bytes most-significant first.
// rst (restart intervals only): bit k set = a restart interval starts at destuffed byte k.
__global__ void __launch_bounds__(256) jpg_destuff_write(const uint8_t *__restrict__ src, int64_t n, const uint32_t *__restrict__ offsets,
                                                         uint8_t *__restrict__ dst, uint32_t *__restrict__ meta, uint32_t *__restrict__ rst)
{
    uint8_t b[16];
    uint32_t rmask;
    const int64_t j0 = (int64_t)blockIdx.x * JPG_CHUNK + threadIdx.x * 16;
    const uint32_t keep = destuff_keepmask(src, n, j0, b, rmask);
    uint32_t tot;
    uint32_t o = cta_exclusive_scan(__popc(keep), &tot) + offsets[blockIdx.x];
#pragma unroll
    for (int j = 0; j < 16; j++) {
        if (rst && (rmask >> j & 1u)) atomicOr(&rst[o >> 5], 1u << (o & 31u));
        if (keep >> j & 1u) { dst[o ^ 3u] = b[j]; o++; }
    }
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) meta[0] = offsets[blockIdx.x] + tot;      // destuffed bytes
}

// ---- Huffman ---------------------------------------------------------------------------------------------------
struct __align__(16) JpgSmemTables {
    uint32_t lut[6][1 << JPG_LUT_BITS];
    uint32_t limit[6][17];
    int32_t valoff[6][17];
    uint8_t vals[6][256];
    uint8_t blk_comp[16];
    uint8_t zigzag[64];
};
__device__ __forceinline__ void load_tables(JpgSmemTables &S, const JpgTables *__restrict__ T)
{
    // the tables sit in global memory (L2-resident after the first CTA): 16-byte coalesced copies
    const uint4 *src = reinterpret_cast<const uint4 *>(T);
    uint4 *dst = reinterpret_cast<uint4 *>(&S);
    constexpr int nq = (int)(offsetof(JpgTables, nblk_mcu) / 16);
    static_assert(offsetof(JpgTables, nblk_mcu) % 16 == 0, "layout");
    static_assert(offsetof(JpgSmemTables, zigzag) == offsetof(JpgTables, nblk_mcu), "layout");
    for (int i = threadIdx.x; i < nq; i += blockDim.x) dst[i] = __ldg(src + i);
    if (threadIdx.x < 64) S.zigzag[threadIdx.x] = c_zigzag[threadIdx.x];
    __syncthreads();
}

// Decode symbols from bit `pos` while pos < end.  State (pos, blk = block inside the MCU, k = next zig-zag index,
// 0 = DC expected).  done counts completed blocks.  WRITE: coefficients go to coef[(base + done) * 64 + natural index].
// One thread walks one subsequence, so the loop is a latency chain: window -> LUT (shared memory) -> advance.  The body
// is branch-free (a warp holds 32 unrelated decoders), the stream window lives in three registers with the next word
// already in flight, and the DC case is folded into the AC rule (run 0, index k + run = 0).
template <bool WRITE>
__device__ __forceinline__ void huff_run(const uint32_t *__restrict__ words, const JpgSmemTables &S, const uint32_t compmap,
                                         const int nblk_mcu, uint32_t &pos, int &blk, int &k, const uint32_t end, uint32_t &done,
                                         int16_t *__restrict__ coef, const uint32_t base, const uint32_t nblocks,
                                         const uint32_t *__restrict__ rst)
{
    constexpr int LUTN = 1 << JPG_LUT_BITS;
    uint32_t wcur = pos >> 5;
    const uint32_t *wp = words + wcur + 2;
    uint32_t hi = wp[-2], lo = wp[-1], nxt = wp[0];
    const uint32_t *lut0 = &S.lut[0][0];
    int set2 = (int)((compmap >> (2 * blk)) & 3u) * 2;               // table pair of the current block
    while (pos < end) {
        const uint32_t win = __funnelshift_l(lo, hi, pos);          // shift amount taken mod 32
        const int tbl = set2 + (k > 0);
        uint32_t e = lut0[tbl * LUTN + (win >> (32 - JPG_LUT_BITS))];
        if (__builtin_expect(e == 0u, 0)) {                         // code longer than the LUT: canonical length search
            const uint32_t w16 = win >> 16;
            const uint32_t *lim = S.limit[tbl];
            int len = JPG_LUT_BITS + 1;
#pragma unroll
            for (int l = JPG_LUT_BITS + 1; l < 16; l++) len += w16 >= lim[l];
            // w16 >= lim[16]: not a code (only a mis-synchronised decoder gets here): 16 bits, symbol 0
            const uint32_t sym = w16 >= lim[16] ? 0u : S.vals[tbl][(S.valoff[tbl][len] + (int)(w16 >> (16 - len))) & 255];
            e = sym | (uint32_t)len << 8 | (uint32_t)(len + (sym & 15u)) << 16;
        }
        const int s = (int)(e & 15u), r = (int)((e >> 4) & 15u);
        const int kz = k + r;                                       // zig-zag index of this coefficient (DC: 0)
        if (WRITE) {
            const uint32_t b = base + done;
            if (s != 0 && kz <= 63 && b < nblocks) {
                const int len = (int)((e >> 8) & 255u);
                const uint32_t v = (win << len) >> (32 - s);
                const int val = v < (1u << (s - 1)) ? (int)v - (1 << s) + 1 : (int)v;
                coef[(size_t)b * 64 + S.zigzag[kz]] = (int16_t)val;
            }
        }
        pos += e >> 16;
        const bool fin = (k != 0 && s == 0 && r != 15) || kz >= 63;  // EOB, or the block is full
        k = fin ? 0 : kz + 1;
        done += fin ? 1u : 0u;
        const int b1 = blk + 1 == nblk_mcu ? 0 : blk + 1;
        blk = fin ? b1 : blk;
        set2 = (int)((compmap >> (2 * blk)) & 3u) * 2;
        uint32_t wnew = pos >> 5;
        if (wnew != wcur) { hi = lo; lo = nxt; nxt = *++wp; wcur = wnew; }
        if (rst != nullptr && fin && blk == 0) {
            // An MCU is complete.  If a restart interval starts at the next byte boundary and only padding (1-bits: no
            // code word is all ones, T.81 C.2) lies before it, this was the last MCU of its interval: skip the padding.
            // (The RSTn marker itself was removed by the destuff pass; the DC predictions restart in jpg_idct.)
            const uint32_t bp = (pos + 7u) >> 3;
            if (rst[bp >> 5] >> (bp & 31u) & 1u) {
                const uint32_t n = 8u * bp - pos;
                const uint32_t w = __funnelshift_l(lo, hi, pos);
                if (n == 0u || (w >> (32u - n)) == (1u << n) - 1u) {
                    pos = 8u * bp;
                    wnew = pos >> 5;
                    if (wnew != wcur) { hi = lo; lo = nxt; nxt = *++wp; wcur = wnew; }
                }
            }
        }
    }
}

// entry state of subsequence i: pos | (blk * 64 + k) << 32
__global__ void __launch_bounds__(256) jpg_sync_init(unsigned long long *__restrict__ start, uint8_t *__restrict__ dirty, int nsub, int sbits)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nsub) return;
    start[i] = (unsigned long long)i << sbits;
    dirty[i] = 1;
    dirty[nsub + i] = 0;
}
// Better first guesses.  A decoder that starts at an arbitrary bit locks on to the code words within a few symbols and to
// the zig-zag index at the next end-of-block, but the block's place inside the MCU (which table pair comes next) stays a
// guess, and a wrong guess loses the lock again at the next luma/chroma change.  So subsequence i is first decoded once per
// possible place h = 0 .. blocks-per-MCU - 1; where at least two of these decoders end in the same state (two unrelated
// wrong decoders practically never agree) that state becomes the entry state of subsequence i + 1, else h = 0's exit is
// used as before.  Still only a guess -- the rounds below verify every subsequence and repair what is wrong.  Measured at
// 24 MP with S = 1024: 4 -> 2 rounds on the iceberg scene (0.51 -> 0.49 ms), 16 -> 14 on the noise texture, where a guessed
// decoder re-synchronises with probability 1/2 per subsequence (the 90 us of the probe are just paid back there).
__global__ void __launch_bounds__(128) jpg_sync_probe(const uint32_t *__restrict__ words, const uint32_t *__restrict__ meta,
                                                      const JpgTables *__restrict__ T, unsigned long long *__restrict__ exits,
                                                      int nsub, int P, const uint32_t *__restrict__ rst, int sbits)
{
    __shared__ JpgSmemTables S;
    load_tables(S, T);
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= nsub * P) return;
    const int i = g / P, h = g - i * P;
    const unsigned long long total_bits = (unsigned long long)meta[0] * 8ull;
    const unsigned long long lo = (unsigned long long)i << sbits, S_bits = 1ull << sbits;
    if (lo >= total_bits) { exits[g] = ~0ull; return; }
    const unsigned long long hi = lo + S_bits < total_bits ? lo + S_bits : total_bits;
    uint32_t pos = (uint32_t)lo, done = 0;
    int blk = h, k = 0;
    huff_run<false>(words, S, T->compmap, T->nblk_mcu, pos, blk, k, (uint32_t)hi, done, nullptr, 0, 0, rst);
    exits[g] = (unsigned long long)pos | ((unsigned long long)(blk * 64 + k) << 32);
}
__global__ void __launch_bounds__(256) jpg_sync_vote(const unsigned long long *__restrict__ exits, unsigned long long *__restrict__ start,
                                                     uint8_t *__restrict__ dirty, int nsub, int P)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nsub) return;
    dirty[i] = 1;
    dirty[nsub + i] = 0;
    if (i == 0) start[0] = 0ull;
    if (i + 1 >= nsub) return;
    const unsigned long long *e = exits + (size_t)i * P;
    unsigned long long best = e[0];                       // subsequence 0: h = 0 IS the true decoder
    if (i > 0) {
        int best_n = 1;
        for (int a = 0; a < P; a++) {
            int n = 0;
            for (int b = 0; b < P; b++) n += e[b] == e[a];
            if (n > best_n) { best_n = n; best = e[a]; }
        }
    }
    start[i + 1] = best;
}

// One round: threads whose entry state changed decode their subsequence and publish the exit state to their successor.
__global__ void __launch_bounds__(128) jpg_sync_round(const uint32_t *__restrict__ words, const uint32_t *__restrict__ meta,
                                                      const JpgTables *__restrict__ T, unsigned long long *__restrict__ start,
                                                      unsigned long long *__restrict__ qstart, uint8_t *__restrict__ dirty,
                                                      uint32_t *__restrict__ nblk, int nsub, int round,
                                                      uint32_t *__restrict__ changed_slot, const uint32_t *__restrict__ rst, int sbits)
{
    __shared__ JpgSmemTables S;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    uint8_t *din = dirty + (round & 1) * nsub, *dout = dirty + ((round + 1) & 1) * nsub;
    // nothing to do in this CTA?  (the common case after the second round)
    const bool mine = i < nsub && din[i];
    if (!__syncthreads_or(mine)) return;
    load_tables(S, T);
    if (!mine) return;
    din[i] = 0;
    const unsigned long long total_bits = (unsigned long long)meta[0] * 8ull;
    const unsigned long long lo = (unsigned long long)i << sbits, S_bits = 1ull << sbits;
    if (lo >= total_bits) {
        for (int q = 0; q < JPG_Q; q++) { nblk[(size_t)i * JPG_Q + q] = 0; qstart[(size_t)i * JPG_Q + q] = ~0ull; }
        return;
    }
    const unsigned long long hi = lo + S_bits < total_bits ? lo + S_bits : total_bits;
    const unsigned long long st = start[i];
    uint32_t pos = (uint32_t)st;
    int blk = (int)(st >> 38), k = (int)(st >> 32) & 63;
    // decoded in JPG_Q pieces: the state at the entry of every piece and the blocks completed inside it are kept, so that
    // the coefficient pass can run with JPG_Q times as many (and as short) decoders.  A thread's last decode starts from
    // its final entry state, so what it leaves behind is final too.
    const unsigned long long piece = S_bits / JPG_Q;
#pragma unroll 1
    for (int q = 0; q < JPG_Q; q++) {
        const unsigned long long qlo = lo + q * piece, qhi = qlo + piece < hi ? qlo + piece : hi;
        qstart[(size_t)i * JPG_Q + q] = (unsigned long long)pos | ((unsigned long long)(blk * 64 + k) << 32);
        uint32_t done = 0;
        if (qlo < hi) huff_run<false>(words, S, T->compmap, T->nblk_mcu, pos, blk, k, (uint32_t)qhi, done, nullptr, 0, 0, rst);
        nblk[(size_t)i * JPG_Q + q] = done;
    }
    if (i + 1 < nsub && hi < total_bits) {
        const unsigned long long out = (unsigned long long)pos | ((unsigned long long)(blk * 64 + k) << 32);
        if (start[i + 1] != out) {
            start[i + 1] = out;
            dout[i + 1] = 1;
            atomicAdd(changed_slot, 1u);
        }
    }
}
// Coefficient pass: one thread per PIECE (S / JPG_Q bits) from the entry state the last sync decode left there.
__global__ void __launch_bounds__(128) jpg_huff_write(const uint32_t *__restrict__ words, const uint32_t *__restrict__ meta,
                                                      const JpgTables *__restrict__ T, const unsigned long long *__restrict__ qstart,
                                                      const uint32_t *__restrict__ base, int16_t *__restrict__ coef, int nsub,
                                                      uint32_t nblocks, const uint32_t *__restrict__ rst, int sbits)
{
    __shared__ JpgSmemTables S;
    load_tables(S, T);
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= nsub * JPG_Q) return;
    const int i = g / JPG_Q, q = g - i * JPG_Q;
    const unsigned long long total_bits = (unsigned long long)meta[0] * 8ull;
    const unsigned long long lo = (unsigned long long)i << sbits, S_bits = 1ull << sbits;
    if (lo >= total_bits) return;
    const unsigned long long hi = lo + S_bits < total_bits ? lo + S_bits : total_bits;
    const unsigned long long piece = S_bits / JPG_Q;
    const unsigned long long qlo = lo + q * piece, qhi = qlo + piece < hi ? qlo + piece : hi;
    if (qlo >= hi) return;
    const unsigned long long st = qstart[g];
    uint32_t pos = (uint32_t)st;
    int blk = (int)(st >> 38), k = (int)(st >> 32) & 63;
    uint32_t done = 0;
    huff_run<true>(words, S, T->compmap, T->nblk_mcu, pos, blk, k, (uint32_t)qhi, done, coef, base[g], nblocks, rst);
}

// ---- DC differences -> per-MCU sums per component (rows of dcs: [comp][nmcu]) ------------------------------------------------
__global__ void __launch_bounds__(256) jpg_dc_sums(const int16_t *__restrict__ coef, const __grid_constant__ JpgGeom G,
                                                   uint32_t *__restrict__ dcs, int nmcu)
{
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= nmcu) return;
    for (int c = 0; c < G.ncomp; c++) {
        int s = 0;
        const int nb = G.hs[c] * G.vs[c];
        for (int j = 0; j < nb; j++) s += coef[((size_t)m * G.nblk_mcu + G.blkoff[c] + j) * 64];
        dcs[(size_t)c * nmcu + m] = (uint32_t)s;
    }
}

// ---- libjpeg "islow" inverse DCT (jidctint.c): 13-bit constants, PASS1_BITS = 2 ------------------------------------------------
template <int SHIFT>
__device__ __forceinline__ void idct8(int i0, int i1, int i2, int i3, int i4, int i5, int i6, int i7, int *o)
{
    int z2 = i2, z3 = i6;
    int z1 = (z2 + z3) * 4433;
    int tmp2 = z1 + z3 * (-15137);
    int tmp3 = z1 + z2 * 6270;
    int tmp0 = (i0 + i4) * 8192;
    int tmp1 = (i0 - i4) * 8192;
    const int tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
    tmp0 = i7; tmp1 = i5; tmp2 = i3; tmp3 = i1;
    z1 = tmp0 + tmp3; z2 = tmp1 + tmp2; z3 = tmp0 + tmp2;
    int z4 = tmp1 + tmp3;
    const int z5 = (z3 + z4) * 9633;
    tmp0 *= 2446; tmp1 *= 16819; tmp2 *= 25172; tmp3 *= 12299;
    z1 *= -7373; z2 *= -20995; z3 *= -16069; z4 *= -3196;
    z3 += z5; z4 += z5;
    tmp0 += z1 + z3; tmp1 += z2 + z4; tmp2 += z2 + z3; tmp3 += z1 + z4;
    constexpr int R = 1 << (SHIFT - 1);
    o[0] = (tmp10 + tmp3 + R) >> SHIFT; o[7] = (tmp10 - tmp3 + R) >> SHIFT;
    o[1] = (tmp11 + tmp2 + R) >> SHIFT; o[6] = (tmp11 - tmp2 + R) >> SHIFT;
    o[2] = (tmp12 + tmp1 + R) >> SHIFT; o[5] = (tmp12 - tmp1 + R) >> SHIFT;
    o[3] = (tmp13 + tmp0 + R) >> SHIFT; o[4] = (tmp13 - tmp0 + R) >> SHIFT;
}
__device__ __forceinline__ uint32_t sat_u8(int v) { return (uint32_t)__vimin_s32_relu(v, 255); }     // max(min(v, 255), 0), one VIMNMX

// one thread per block, blocks numbered in plane order per component (component 0 first)
__global__ void __launch_bounds__(128) jpg_idct(const int16_t *__restrict__ coef, const uint32_t *__restrict__ dcpre,
                                                const __grid_constant__ JpgGeom G, int nmcu, int total_blocks)
{
    __shared__ int sq[3][64];
    for (int i = threadIdx.x; i < 3 * 64; i += blockDim.x) sq[i / 64][i % 64] = G.quant[i / 64][i % 64];
    __syncthreads();
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total_blocks) return;
    int c = 0;
    while (c < G.ncomp - 1 && t >= G.bw[c] * G.bh[c]) { t -= G.bw[c] * G.bh[c]; c++; }
    const int by = t / G.bw[c], bx = t - by * G.bw[c];
    const int h = G.hs[c], v = G.vs[c];
    const int m = (by / v) * G.mcux + bx / h;
    const int jl = (by % v) * h + (bx % h);
    const size_t b0 = (size_t)m * G.nblk_mcu + G.blkoff[c];
    int dc = (int)dcpre[(size_t)c * nmcu + m];
    if (G.restart_interval) dc -= (int)dcpre[(size_t)c * nmcu + m - m % G.restart_interval];
    for (int j = 0; j <= jl; j++) dc += coef[(b0 + j) * 64];
    const uint4 *src = reinterpret_cast<const uint4 *>(coef + (b0 + jl) * 64);
    int ws[64];
    {
        int in[64];
#pragma unroll
        for (int r = 0; r < 8; r++) {
            const uint4 q = __ldg(src + r);
            const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int j = 0; j < 4; j++) {
                in[r * 8 + 2 * j] = (int)(short)(w[j] & 0xffffu) * sq[c][r * 8 + 2 * j];
                in[r * 8 + 2 * j + 1] = ((int)w[j] >> 16) * sq[c][r * 8 + 2 * j + 1];
            }
        }
        in[0] = dc * sq[c][0];
#pragma unroll
        for (int col = 0; col < 8; col++) {
            int o[8];
            idct8<11>(in[col], in[8 + col], in[16 + col], in[24 + col], in[32 + col], in[40 + col], in[48 + col], in[56 + col], o);
#pragma unroll
            for (int r = 0; r < 8; r++) ws[r * 8 + col] = o[r];
        }
    }
    uint8_t *dst = G.plane[c] + (size_t)by * 8 * G.pw[c] + bx * 8;
#pragma unroll
    for (int r = 0; r < 8; r++) {
        int o[8];
        idct8<18>(ws[r * 8], ws[r * 8 + 1], ws[r * 8 + 2], ws[r * 8 + 3], ws[r * 8 + 4], ws[r * 8 + 5], ws[r * 8 + 6], ws[r * 8 + 7], o);
        uint2 px;
        px.x = sat_u8(o[0] + 128) | sat_u8(o[1] + 128) << 8 | sat_u8(o[2] + 128) << 16 | sat_u8(o[3] + 128) << 24;
        px.y = sat_u8(o[4] + 128) | sat_u8(o[5] + 128) << 8 | sat_u8(o[6] + 128) << 16 | sat_u8(o[7] + 128) << 24;
        *reinterpret_cast<uint2 *>(dst + (size_t)r * G.pw[c]) = px;
    }
}

// ---- chroma upsampling (jdsample.c "fancy") + YCbCr -> RGB (jdcolor.c) + optional cvtColor gray ---------------------------------
// six neighbouring samples of one chroma row: columns cx0-1 .. cx0+4 (cx0 a multiple of 4), clamped to [0, dw-1]
__device__ __forceinline__ void chroma_row6(const uint8_t *__restrict__ row, int cx0, int dw, int *v)
{
    if (cx0 > 0 && cx0 + 4 <= dw - 1) {
        const uint32_t w = *reinterpret_cast<const uint32_t *>(row + cx0);
        v[0] = row[cx0 - 1]; v[1] = w & 255; v[2] = (w >> 8) & 255; v[3] = (w >> 16) & 255; v[4] = w >> 24; v[5] = row[cx0 + 4];
    } else {
#pragma unroll
        for (int j = 0; j < 6; j++) v[j] = row[min(max(cx0 - 1 + j, 0), dw - 1)];
    }
}
// 8 chroma samples for pixels x0..x0+7 (x0 a multiple of 8) of row y; HSUB x VSUB = luma samples per chroma sample
template <int HSUB, int VSUB>
__device__ __forceinline__ void chroma8(const JpgGeom &G, int c, int x0, int y, int *out)
{
    const uint8_t *P = G.plane[c];
    const int pw = G.pw[c], dw = G.dw[c], dh = G.dh[c];
    constexpr int hsub = HSUB, vsub = VSUB;
    if (hsub == 1) {
        const uint2 w = *reinterpret_cast<const uint2 *>(P + (size_t)y * pw + x0);
#pragma unroll
        for (int j = 0; j < 4; j++) { out[j] = (w.x >> (8 * j)) & 255; out[4 + j] = (w.y >> (8 * j)) & 255; }
        return;
    }
    const int cx0 = x0 >> 1;
    int a[6];
    if (vsub == 1) {
        chroma_row6(P + (size_t)y * pw, cx0, dw, a);
        if (dw <= 2) {                                             // h2v1_upsample: plain replication
#pragma unroll
            for (int j = 0; j < 8; j++) out[j] = a[1 + (j >> 1)];
            return;
        }
#pragma unroll
        for (int j = 0; j < 4; j++) {
            out[2 * j] = (3 * a[1 + j] + a[j] + 1) >> 2;
            out[2 * j + 1] = (3 * a[1 + j] + a[2 + j] + 2) >> 2;
        }
        return;
    }
    const int cy = y >> 1;
    chroma_row6(P + (size_t)cy * pw, cx0, dw, a);
    if (dw <= 2) {                                                 // h2v2_upsample: plain replication
#pragma unroll
        for (int j = 0; j < 8; j++) out[j] = a[1 + (j >> 1)];
        return;
    }
    int f[6];
    chroma_row6(P + (size_t)min(max((y & 1) ? cy + 1 : cy - 1, 0), dh - 1) * pw, cx0, dw, f);
#pragma unroll
    for (int j = 0; j < 6; j++) a[j] = 3 * a[j] + f[j];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        out[2 * j] = (3 * a[1 + j] + a[j] + 8) >> 4;
        out[2 * j + 1] = (3 * a[1 + j] + a[2 + j] + 7) >> 4;
    }
}

template <int SH, int NCOMP, int HSUB, int VSUB>
__global__ void __launch_bounds__(256) jpg_color(const __grid_constant__ JpgGeom G, uint8_t *__restrict__ rgb, int64_t rgb_pitch,
                                                 uint8_t *__restrict__ gray, int64_t gray_pitch, int k0, int k1, int k2)
{
    const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * 8;
    const int y = blockIdx.y;
    if (x0 >= G.W) return;
    const uint2 yw = *reinterpret_cast<const uint2 *>(G.plane[0] + (size_t)y * G.pw[0] + x0);
    uint32_t R[8], Gc[8], B[8], g[8];
    if (NCOMP == 1) {
#pragma unroll
        for (int j = 0; j < 8; j++) g[j] = ((j < 4 ? yw.x : yw.y) >> (8 * (j & 3))) & 255u;
    } else {
        int cb[8], cr[8];
        chroma8<HSUB, VSUB>(G, 1, x0, y, cb);
        chroma8<HSUB, VSUB>(G, 2, x0, y, cr);
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const int Y = (int)(((j < 4 ? yw.x : yw.y) >> (8 * (j & 3))) & 255u), b = cb[j] - 128, r = cr[j] - 128;
            R[j] = sat_u8(Y + ((91881 * r + 32768) >> 16));
            Gc[j] = sat_u8(Y + ((-22554 * b + 32768 - 46802 * r) >> 16));
            B[j] = sat_u8(Y + ((116130 * b + 32768) >> 16));
            g[j] = (R[j] * k0 + Gc[j] * k1 + B[j] * k2 + (1u << (SH - 1))) >> SH;      // channel 0 takes the "B" weight (s1:311)
        }
    }
    const bool full = x0 + 8 <= G.W;
    if (gray) {
        uint8_t *d = gray + (size_t)y * gray_pitch + x0;
        if (full && ((reinterpret_cast<uintptr_t>(d) & 7) == 0))
            *reinterpret_cast<uint2 *>(d) = make_uint2(g[0] | g[1] << 8 | g[2] << 16 | g[3] << 24, g[4] | g[5] << 8 | g[6] << 16 | g[7] << 24);
        else
            for (int j = 0; j < 8 && x0 + j < G.W; j++) d[j] = (uint8_t)g[j];
    }
    if (NCOMP == 3 && rgb) {
        uint8_t *d = rgb + (size_t)y * rgb_pitch + (size_t)x0 * 3;
        if (full && ((reinterpret_cast<uintptr_t>(d) & 7) == 0)) {
            uint2 *w = reinterpret_cast<uint2 *>(d);
            w[0] = make_uint2(R[0] | Gc[0] << 8 | B[0] << 16 | R[1] << 24, Gc[1] | B[1] << 8 | R[2] << 16 | Gc[2] << 24);
            w[1] = make_uint2(B[2] | R[3] << 8 | Gc[3] << 16 | B[3] << 24, R[4] | Gc[4] << 8 | B[4] << 16 | R[5] << 24);
            w[2] = make_uint2(Gc[5] | B[5] << 8 | R[6] << 16 | Gc[6] << 24, B[6] | R[7] << 8 | Gc[7] << 16 | B[7] << 24);
        } else {
            for (int j = 0; j < 8 && x0 + j < G.W; j++) { d[3 * j] = (uint8_t)R[j]; d[3 * j + 1] = (uint8_t)Gc[j]; d[3 * j + 2] = (uint8_t)B[j]; }
        }
    }
}

// ---- save-and-reopen round trip of the cropping pre-pass (camtools.py:80,102,232 -> s1:310) ----------------------------------
// `img_crop.save(outpath)` re-encodes every cropped frame with Pillow's defaults (libjpeg-turbo: quality 75, 4:2:0, islow DCT)
// and the tracking loop reads that file back.  Entropy coding is lossless, so the pixels the reference tracks are
//   decode( quantise( FDCT( downsample( RGB->YCbCr( crop ))))).
// jpg_enc_planes: jccolor.c rgb_ycc_convert (16-bit fixed point) + jcsample.c box filters (alternating bias) with libjpeg's edge
//                 replication (jcprepct.c / expand_right_edge), written straight into the decoder's plane layout;
// jpg_enc_requant: one thread per 8x8 block, in place: jfdctint.c forward DCT, jcdctmgr.c quantisation (divisor 8q, magnitude
//                 rounded half up), dequantisation and the islow inverse DCT of jpg_idct;
// then the decoder's own jpg_color kernel (fancy upsampling, YCbCr->RGB, gray).
struct JpgEncQ {
    uint16_t q[2][64];                    // luma / chroma tables, natural order
    uint32_t magic[2][64];                // floor(2^32 / (8 q)) + 1: exact quotients for numerators < 2^20
};

// 8 RGB pixels of row `row` (already clamped) starting at column x0; columns past W - 1 replicate the last one
__device__ __forceinline__ void enc_load8(const uint8_t *__restrict__ rgb, int64_t pitch, int row, int x0, int W, uint32_t *px)
{
    const uint8_t *p = rgb + (size_t)row * pitch + (size_t)x0 * 3;
    if (x0 + 10 <= W) {                                          // the 28 bytes of the seven aligned words stay inside the row
        const uintptr_t a = reinterpret_cast<uintptr_t>(p);
        const uint32_t *w = reinterpret_cast<const uint32_t *>(a & ~(uintptr_t)3);
        const uint32_t sh = (uint32_t)(a & 3u) * 8u;
        uint32_t v[7];
#pragma unroll
        for (int j = 0; j < 7; j++) v[j] = __ldg(w + j);
        uint32_t b[6];
#pragma unroll
        for (int j = 0; j < 6; j++) b[j] = __funnelshift_r(v[j], v[j + 1], sh);
#pragma unroll
        for (int j = 0; j < 8; j++) {                             // pixel j = bytes 3j .. 3j+2 of the 24
            const int o = 3 * j, wi = o >> 2, bi = (o & 3) * 8;
            const uint32_t t = bi == 0 ? b[wi] : __funnelshift_r(b[wi], wi + 1 < 6 ? b[wi + 1] : 0u, bi);
            px[j] = t & 0xffffffu;
        }
    } else {
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const uint8_t *q = rgb + (size_t)row * pitch + (size_t)min(x0 + j, W - 1) * 3;
            px[j] = (uint32_t)q[0] | (uint32_t)q[1] << 8 | (uint32_t)q[2] << 16;
        }
    }
}
__device__ __forceinline__ void enc_ycc(uint32_t p, int &Y, int &Cb, int &Cr)
{
    const int r = p & 255, g = (p >> 8) & 255, b = (p >> 16) & 255;
    Y = (19595 * r + 38470 * g + 7471 * b + 32768) >> 16;
    Cb = (-11059 * r - 21709 * g + 32768 * b + (128 << 16) + 32767) >> 16;
    Cr = (32768 * r - 27439 * g - 5329 * b + (128 << 16) + 32767) >> 16;
}

// thread = 8 luma columns x VS luma rows (one chroma row); grid.y = chroma plane rows
template <int HS, int VS>
__global__ void __launch_bounds__(256) jpg_enc_planes(const uint8_t *__restrict__ rgb, int64_t pitch, const __grid_constant__ JpgGeom G)
{
    const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * 8;
    const int gy = blockIdx.y;
    if (x0 >= G.pw[0]) return;
    const int W = G.W, H = G.H;
    // chroma row gy: rows past the last real row group copy that group (jcprepct.c pads the DOWNSAMPLED rows)
    const int ce = min(gy, G.dh[1] - 1);
    int cb[VS][8], cr[VS][8], yy[VS][8];
    int srow[VS];
#pragma unroll
    for (int r = 0; r < VS; r++) {
        srow[r] = min(VS * ce + r, H - 1);
        uint32_t px[8];
        enc_load8(rgb, pitch, srow[r], x0, W, px);
#pragma unroll
        for (int j = 0; j < 8; j++) enc_ycc(px[j], yy[r][j], cb[r][j], cr[r][j]);
    }
    // luma rows VS*gy + r take source row min(VS*gy + r, H - 1): the same rows except in the padding below an even-height image
#pragma unroll
    for (int r = 0; r < VS; r++) {
        const int lrow = min(VS * gy + r, H - 1);
        if (lrow != srow[r]) {
            uint32_t px[8];
            enc_load8(rgb, pitch, lrow, x0, W, px);
            int d0, d1;
#pragma unroll
            for (int j = 0; j < 8; j++) enc_ycc(px[j], yy[r][j], d0, d1);
        }
        uint2 o;
        o.x = (uint32_t)yy[r][0] | (uint32_t)yy[r][1] << 8 | (uint32_t)yy[r][2] << 16 | (uint32_t)yy[r][3] << 24;
        o.y = (uint32_t)yy[r][4] | (uint32_t)yy[r][5] << 8 | (uint32_t)yy[r][6] << 16 | (uint32_t)yy[r][7] << 24;
        *reinterpret_cast<uint2 *>(G.plane[0] + (size_t)(VS * gy + r) * G.pw[0] + x0) = o;
    }
    if (HS == 1) {
        uint2 ob, orr;
        ob.x = (uint32_t)cb[0][0] | (uint32_t)cb[0][1] << 8 | (uint32_t)cb[0][2] << 16 | (uint32_t)cb[0][3] << 24;
        ob.y = (uint32_t)cb[0][4] | (uint32_t)cb[0][5] << 8 | (uint32_t)cb[0][6] << 16 | (uint32_t)cb[0][7] << 24;
        orr.x = (uint32_t)cr[0][0] | (uint32_t)cr[0][1] << 8 | (uint32_t)cr[0][2] << 16 | (uint32_t)cr[0][3] << 24;
        orr.y = (uint32_t)cr[0][4] | (uint32_t)cr[0][5] << 8 | (uint32_t)cr[0][6] << 16 | (uint32_t)cr[0][7] << 24;
        *reinterpret_cast<uint2 *>(G.plane[1] + (size_t)gy * G.pw[1] + x0) = ob;
        *reinterpret_cast<uint2 *>(G.plane[2] + (size_t)gy * G.pw[2] + x0) = orr;
    } else {
        uint32_t ob = 0, orr = 0;
#pragma unroll
        for (int j = 0; j < 4; j++) {                             // chroma column x0/2 + j: bias 1,2,1,2 (h2v2) / 0,1,0,1 (h2v1)
            int sb = cb[0][2 * j] + cb[0][2 * j + 1], sr = cr[0][2 * j] + cr[0][2 * j + 1];
            if (VS == 2) {
                sb += cb[VS - 1][2 * j] + cb[VS - 1][2 * j + 1] + 1 + (j & 1);
                sr += cr[VS - 1][2 * j] + cr[VS - 1][2 * j + 1] + 1 + (j & 1);
                sb >>= 2; sr >>= 2;
            } else {
                sb = (sb + (j & 1)) >> 1; sr = (sr + (j & 1)) >> 1;
            }
            ob |= (uint32_t)sb << (8 * j);
            orr |= (uint32_t)sr << (8 * j);
        }
        *reinterpret_cast<uint32_t *>(G.plane[1] + (size_t)gy * G.pw[1] + (x0 >> 1)) = ob;
        *reinterpret_cast<uint32_t *>(G.plane[2] + (size_t)gy * G.pw[2] + (x0 >> 1)) = orr;
    }
}

// jfdctint.c, one 8-point pass.  PASS 1: rows, outputs scaled up by 2^PASS1_BITS; PASS 2: columns, scaled back (overall x8)
template <int PASS>
__device__ __forceinline__ void fdct8(int &d0, int &d1, int &d2, int &d3, int &d4, int &d5, int &d6, int &d7)
{
    const int t0 = d0 + d7, t7 = d0 - d7, t1 = d1 + d6, t6 = d1 - d6, t2 = d2 + d5, t5 = d2 - d5, t3 = d3 + d4, t4 = d3 - d4;
    const int t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
    constexpr int SH = PASS == 1 ? 11 : 15, R = 1 << (SH - 1);
    if (PASS == 1) { d0 = (t10 + t11) * 4; d4 = (t10 - t11) * 4; }
    else { d0 = (t10 + t11 + 2) >> 2; d4 = (t10 - t11 + 2) >> 2; }
    int z1 = (t12 + t13) * 4433;
    d2 = (z1 + t13 * 6270 + R) >> SH;
    d6 = (z1 + t12 * (-15137) + R) >> SH;
    z1 = t4 + t7;
    int z2 = t5 + t6, z3 = t4 + t6, z4 = t5 + t7;
    const int z5 = (z3 + z4) * 9633;
    const int a4 = t4 * 2446, a5 = t5 * 16819, a6 = t6 * 25172, a7 = t7 * 12299;
    z1 *= -7373; z2 *= -20995; z3 *= -16069; z4 *= -3196;
    z3 += z5; z4 += z5;
    d7 = (a4 + z1 + z3 + R) >> SH;
    d5 = (a5 + z2 + z4 + R) >> SH;
    d3 = (a6 + z2 + z3 + R) >> SH;
    d1 = (a7 + z1 + z4 + R) >> SH;
}

__global__ void __launch_bounds__(128) jpg_enc_requant(const __grid_constant__ JpgGeom G, const __grid_constant__ JpgEncQ Q, int total_blocks)
{
    __shared__ int sq[2][64];
    __shared__ uint32_t sm[2][64];
    for (int i = threadIdx.x; i < 128; i += blockDim.x) { sq[i >> 6][i & 63] = Q.q[i >> 6][i & 63]; sm[i >> 6][i & 63] = Q.magic[i >> 6][i & 63]; }
    __syncthreads();
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total_blocks) return;
    int c = 0;
    while (c < G.ncomp - 1 && t >= G.bw[c] * G.bh[c]) { t -= G.bw[c] * G.bh[c]; c++; }
    const int by = t / G.bw[c], bx = t - by * G.bw[c];
    const int tq = c ? 1 : 0;
    uint8_t *blk = G.plane[c] + (size_t)by * 8 * G.pw[c] + bx * 8;
    int w[64];
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const uint2 v = *reinterpret_cast<const uint2 *>(blk + (size_t)r * G.pw[c]);
#pragma unroll
        for (int j = 0; j < 4; j++) {
            w[r * 8 + j] = (int)((v.x >> (8 * j)) & 255u) - 128;
            w[r * 8 + 4 + j] = (int)((v.y >> (8 * j)) & 255u) - 128;
        }
        fdct8<1>(w[r * 8], w[r * 8 + 1], w[r * 8 + 2], w[r * 8 + 3], w[r * 8 + 4], w[r * 8 + 5], w[r * 8 + 6], w[r * 8 + 7]);
    }
    int ws[64];
#pragma unroll
    for (int col = 0; col < 8; col++) {
        fdct8<2>(w[col], w[8 + col], w[16 + col], w[24 + col], w[32 + col], w[40 + col], w[48 + col], w[56 + col]);
        // quantise (magnitude + half the divisor, truncating division by 8q) and dequantise
#pragma unroll
        for (int r = 0; r < 8; r++) {
            const int i = r * 8 + col, q = sq[tq][i], v = w[i];
            const uint32_t a = (uint32_t)abs(v) + (uint32_t)(q * 4);
            const int m = (int)__umulhi(a, sm[tq][i]) * q;
            w[i] = v < 0 ? -m : m;
        }
        int o[8];
        idct8<11>(w[col], w[8 + col], w[16 + col], w[24 + col], w[32 + col], w[40 + col], w[48 + col], w[56 + col], o);
#pragma unroll
        for (int r = 0; r < 8; r++) ws[r * 8 + col] = o[r];
    }
#pragma unroll
    for (int r = 0; r < 8; r++) {
        int o[8];
        idct8<18>(ws[r * 8], ws[r * 8 + 1], ws[r * 8 + 2], ws[r * 8 + 3], ws[r * 8 + 4], ws[r * 8 + 5], ws[r * 8 + 6], ws[r * 8 + 7], o);
        uint2 px;
        px.x = sat_u8(o[0] + 128) | sat_u8(o[1] + 128) << 8 | sat_u8(o[2] + 128) << 16 | sat_u8(o[3] + 128) << 24;
        px.y = sat_u8(o[4] + 128) | sat_u8(o[5] + 128) << 8 | sat_u8(o[6] + 128) << 16 | sat_u8(o[7] + 128) << 24;
        *reinterpret_cast<uint2 *>(blk + (size_t)r * G.pw[c]) = px;
    }
}

// ---- host ---------------------------------------------------------------------------------------------------------------
static const uint8_t h_zigzag[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                     41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                     30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

static int jpeg_validate(const ibt_jpeg_info_t *I)
{
    if (!I || I->width <= 0 || I->height <= 0 || I->width > 65535 || I->height > 65535) return IBT_E_INVALID;
    if (I->ncomp != 1 && I->ncomp != 3) return IBT_E_UNSUPPORTED;
    if (I->restart_interval < 0) return IBT_E_INVALID;
    if (I->scan_bytes <= 0 || I->scan_offset < 0 || I->scan_bytes > 0x1fffffff) return IBT_E_INVALID;
    for (int c = 0; c < I->ncomp; c++) {
        if (I->hsamp[c] < 1 || I->vsamp[c] < 1 || I->qsel[c] < 0 || I->qsel[c] > 3 || I->dcsel[c] < 0 || I->dcsel[c] > 3 ||
            I->acsel[c] < 0 || I->acsel[c] > 3)
            return IBT_E_INVALID;
    }
    if (I->ncomp == 3) {
        if (I->hsamp[1] != 1 || I->vsamp[1] != 1 || I->hsamp[2] != 1 || I->vsamp[2] != 1) return IBT_E_UNSUPPORTED;
        const int h = I->hsamp[0], v = I->vsamp[0];
        if (!((h == 1 && v == 1) || (h == 2 && v == 1) || (h == 2 && v == 2))) return IBT_E_UNSUPPORTED;
    }
    return IBT_OK;
}

// S = 2^sbits: at most ~16 k subsequences per file while 256 <= S <= 2048 (IBT_JPEG_SBITS overrides: the sweep in profiles/)
static int jpeg_sbits(const ibt_jpeg_info_t *I)
{
    static const int forced = getenv("IBT_JPEG_SBITS") ? atoi(getenv("IBT_JPEG_SBITS")) : 0;
    if (forced >= 7 && forced <= 12) return forced;
    const long long bits = (long long)I->scan_bytes * 8;
    int sb = 8;
    while (sb < 11 && (bits >> sb) > 16000) sb++;
    return sb;
}

struct JpgLayout {
    JpgGeom G;
    int nmcu, nblocks, nsub, nchunks, sbits;
    size_t off_stream, off_counts, off_offsets, off_meta, off_tables, off_rst, off_exits, off_changed, off_start, off_qstart, off_dirty, off_nblk, off_base, off_partial,
        off_coef, off_dcs, off_dcpre, off_plane[3], total;
    size_t stream_bytes, coef_bytes, rst_bytes;
};
constexpr int JPG_MAX_ROUNDS_BATCH = 64;
static std::atomic<bool> jpeg_probe_enabled{true};        // ibt_jpeg_set_probe

static void jpeg_layout(const ibt_jpeg_info_t *I, JpgLayout &L)
{
    memset(&L, 0, sizeof(L));
    JpgGeom &G = L.G;
    G.ncomp = I->ncomp; G.W = I->width; G.H = I->height;
    G.restart_interval = I->restart_interval;
    G.hmax = G.vmax = 1;
    for (int c = 0; c < I->ncomp; c++) {
        G.hs[c] = I->ncomp == 1 ? 1 : I->hsamp[c];
        G.vs[c] = I->ncomp == 1 ? 1 : I->vsamp[c];
        if (G.hs[c] > G.hmax) G.hmax = G.hs[c];
        if (G.vs[c] > G.vmax) G.vmax = G.vs[c];
    }
    G.mcux = (G.W + 8 * G.hmax - 1) / (8 * G.hmax);
    G.mcuy = (G.H + 8 * G.vmax - 1) / (8 * G.vmax);
    int off = 0;
    for (int c = 0; c < I->ncomp; c++) {
        G.blkoff[c] = off;
        off += G.hs[c] * G.vs[c];
        G.bw[c] = G.mcux * G.hs[c]; G.bh[c] = G.mcuy * G.vs[c];
        G.pw[c] = G.bw[c] * 8; G.ph[c] = G.bh[c] * 8;
        G.dw[c] = (G.W * G.hs[c] + G.hmax - 1) / G.hmax;
        G.dh[c] = (G.H * G.vs[c] + G.vmax - 1) / G.vmax;
        G.hsub[c] = G.hmax / G.hs[c]; G.vsub[c] = G.vmax / G.vs[c];
        for (int i = 0; i < 64; i++) G.quant[c][i] = I->quant[I->qsel[c]][i];
    }
    G.nblk_mcu = off;
    L.nmcu = G.mcux * G.mcuy;
    L.nblocks = L.nmcu * G.nblk_mcu;
    L.sbits = jpeg_sbits(I);
    L.nsub = (int)((I->scan_bytes * 8 + (1ll << L.sbits) - 1) >> L.sbits);
    L.nchunks = (int)((I->scan_bytes + JPG_CHUNK - 1) / JPG_CHUNK);
    size_t o = 0;
    auto take = [&](size_t bytes) { const size_t r = o; o += (bytes + 255) & ~(size_t)255; return r; };
    L.stream_bytes = ((size_t)I->scan_bytes + 64 + 3) & ~(size_t)3;
    L.off_stream = take(L.stream_bytes);
    L.off_counts = take((size_t)L.nchunks * 4);
    L.off_offsets = take((size_t)L.nchunks * 4);
    L.off_meta = take(64);
    L.off_tables = take(sizeof(JpgTables));
    L.rst_bytes = I->restart_interval ? ((L.stream_bytes / 8 + 8 + 3) & ~(size_t)3) : 0;
    L.off_rst = take(L.rst_bytes);
    L.off_exits = take((size_t)L.nsub * G.nblk_mcu * 8);
    L.off_changed = take(JPG_MAX_ROUNDS_BATCH * 4);
    L.off_start = take((size_t)L.nsub * 8);
    L.off_dirty = take((size_t)L.nsub * 2);
    L.off_nblk = take((size_t)L.nsub * JPG_Q * 4);
    L.off_base = take((size_t)L.nsub * JPG_Q * 4);
    L.off_qstart = take((size_t)L.nsub * JPG_Q * 8);
    L.off_partial = take(std::max({scan_partial_words(L.nchunks, 1), scan_partial_words(L.nsub * JPG_Q, 1),
                                   scan_partial_words(L.nmcu, 3)}) * 4);
    L.coef_bytes = (size_t)L.nblocks * 64 * 2;
    L.off_coef = take(L.coef_bytes);
    L.off_dcs = take((size_t)3 * L.nmcu * 4);
    L.off_dcpre = take((size_t)3 * L.nmcu * 4);
    for (int c = 0; c < I->ncomp; c++) L.off_plane[c] = take((size_t)G.pw[c] * G.ph[c]);
    L.total = o;
}

static int build_tables(const ibt_jpeg_info_t *I, const JpgGeom &G, JpgTables &T)
{
    memset(&T, 0, sizeof(T));
    for (int c = 0; c < I->ncomp; c++)
        for (int ac = 0; ac < 2; ac++) {
            const uint8_t *bits = ac ? I->ac_bits[I->acsel[c]] : I->dc_bits[I->dcsel[c]];
            const uint8_t *vals = ac ? I->ac_vals[I->acsel[c]] : I->dc_vals[I->dcsel[c]];
            const int t = c * 2 + ac, nvals_max = ac ? 256 : 16;
            int code = 0, k = 0;
            for (int l = 1; l <= 16; l++) {
                const int n = bits[l - 1];
                if (k + n > nvals_max || code + n > (1 << l)) return IBT_E_INVALID;
                T.valoff[t][l] = k - code;
                for (int i = 0; i < n; i++, code++, k++) {
                    if (!ac && vals[k] > 15) return IBT_E_INVALID;          // DC categories are 0..11 (T.81 F.1.2.1)
                    T.vals[t][k] = vals[k];
                    if (l <= JPG_LUT_BITS) {
                        const int lo = code << (JPG_LUT_BITS - l), cnt = 1 << (JPG_LUT_BITS - l);
                        for (int j = 0; j < cnt; j++)
                            T.lut[t][lo + j] = (uint32_t)vals[k] | (uint32_t)l << 8 | (uint32_t)(l + (vals[k] & 15)) << 16;
                    }
                }
                T.limit[t][l] = (uint32_t)code << (16 - l);
                code <<= 1;
            }
            if (k == 0) return IBT_E_INVALID;
        }
    T.nblk_mcu = G.nblk_mcu;
    for (int c = 0; c < I->ncomp; c++)
        for (int j = 0; j < G.hs[c] * G.vs[c]; j++) {
            T.blk_comp[G.blkoff[c] + j] = (uint8_t)c;
            T.compmap |= (uint32_t)c << (2 * (G.blkoff[c] + j));
        }
    return IBT_OK;
}

// geometry of the file Pillow would write for a W x H RGB image with luma sampling hs x vs
static void recompress_layout(int W, int H, int hs, int vs, JpgLayout &L)
{
    ibt_jpeg_info_t I;
    memset(&I, 0, sizeof(I));
    I.width = W; I.height = H; I.ncomp = 3;
    I.hsamp[0] = hs; I.vsamp[0] = vs; I.hsamp[1] = I.vsamp[1] = I.hsamp[2] = I.vsamp[2] = 1;
    I.scan_bytes = 1;
    jpeg_layout(&I, L);
    size_t o = 0;
    for (int c = 0; c < 3; c++) { L.off_plane[c] = o; o += ((size_t)L.G.pw[c] * L.G.ph[c] + 255) & ~(size_t)255; }
    L.total = o;
}

} // namespace ibt

// ---- HOST: marker parsing (ITU-T T.81 Annex B) ------------------------------------------------------------------------------
IBT_API int ibt_jpeg_parse(const uint8_t *d, int64_t n, ibt_jpeg_info_t *I)
{
    if (!d || !I || n < 4) return IBT_E_INVALID;
    memset(I, 0, sizeof(*I));
    if (d[0] != 0xFF || d[1] != 0xD8) return IBT_E_INVALID;
    int64_t p = 2;
    int comp_id[3] = {0, 0, 0};
    bool have_sof = false, have_q[4] = {false, false, false, false}, have_dc[4] = {false, false, false, false},
         have_ac[4] = {false, false, false, false};
    for (;;) {
        if (p + 4 > n || d[p] != 0xFF) return IBT_E_INVALID;
        while (p < n && d[p] == 0xFF) p++;
        if (p >= n) return IBT_E_INVALID;
        const int m = d[p++];
        if (m == 0xD8 || (m >= 0xD0 && m <= 0xD7) || m == 0x01) continue;
        if (m == 0xD9 || p + 2 > n) return IBT_E_INVALID;
        const int len = (d[p] << 8) | d[p + 1];
        if (len < 2 || p + len > n) return IBT_E_INVALID;
        const uint8_t *s = d + p + 2;
        const int sl = len - 2;
        if (m == 0xC0 || m == 0xC1) {
            if (sl < 6) return IBT_E_INVALID;
            if (s[0] != 8) return IBT_E_UNSUPPORTED;
            I->height = (s[1] << 8) | s[2];
            I->width = (s[3] << 8) | s[4];
            I->ncomp = s[5];
            if (I->ncomp != 1 && I->ncomp != 3) return IBT_E_UNSUPPORTED;
            if (sl < 6 + 3 * I->ncomp) return IBT_E_INVALID;
            for (int i = 0; i < I->ncomp; i++) {
                comp_id[i] = s[6 + 3 * i];
                I->hsamp[i] = s[7 + 3 * i] >> 4;
                I->vsamp[i] = s[7 + 3 * i] & 15;
                I->qsel[i] = s[8 + 3 * i] & 3;
            }
            have_sof = true;
        } else if (m >= 0xC2 && m <= 0xCF && m != 0xC4 && m != 0xC8 && m != 0xCC) {
            return IBT_E_UNSUPPORTED;                       // progressive, lossless, arithmetic, differential
        } else if (m == 0xC4) {
            int o = 0;
            while (o < sl) {
                if (o + 17 > sl) return IBT_E_INVALID;
                const int tc = s[o] >> 4, th = s[o] & 15;
                if (tc > 1 || th > 3) return IBT_E_INVALID;
                int cnt = 0;
                for (int l = 0; l < 16; l++) cnt += s[o + 1 + l];
                if (cnt > (tc ? 256 : 16) || o + 17 + cnt > sl) return IBT_E_INVALID;
                uint8_t *bits = tc ? I->ac_bits[th] : I->dc_bits[th];
                uint8_t *vals = tc ? I->ac_vals[th] : I->dc_vals[th];
                memcpy(bits, s + o + 1, 16);
                memset(vals, 0, tc ? 256 : 16);
                memcpy(vals, s + o + 17, cnt);
                (tc ? have_ac : have_dc)[th] = true;
                o += 17 + cnt;
            }
        } else if (m == 0xDB) {
            int o = 0;
            while (o < sl) {
                const int pq = s[o] >> 4, tq = s[o] & 15;
                if (tq > 3 || pq > 1) return IBT_E_INVALID;
                o++;
                if (o + 64 * (pq + 1) > sl) return IBT_E_INVALID;
                for (int i = 0; i < 64; i++) {
                    I->quant[tq][ibt::h_zigzag[i]] = (uint16_t)(pq ? ((s[o] << 8) | s[o + 1]) : s[o]);
                    o += pq + 1;
                }
                have_q[tq] = true;
            }
        } else if (m == 0xDD) {
            if (sl < 2) return IBT_E_INVALID;
            I->restart_interval = (s[0] << 8) | s[1];
        } else if (m == 0xDA) {
            if (!have_sof || sl < 1) return IBT_E_INVALID;
            const int ns = s[0];
            if (ns != I->ncomp) return IBT_E_UNSUPPORTED;   // one interleaved scan only
            if (sl < 1 + 2 * ns + 3) return IBT_E_INVALID;
            for (int i = 0; i < ns; i++) {
                if (s[1 + 2 * i] != comp_id[i]) return IBT_E_UNSUPPORTED;
                I->dcsel[i] = s[2 + 2 * i] >> 4;
                I->acsel[i] = s[2 + 2 * i] & 15;
                if (I->dcsel[i] > 3 || I->acsel[i] > 3) return IBT_E_INVALID;
            }
            p += len;
            break;
        }
        p += len;
    }
    for (int i = 0; i < I->ncomp; i++)
        if (!have_q[I->qsel[i]] || !have_dc[I->dcsel[i]] || !have_ac[I->acsel[i]]) return IBT_E_INVALID;
    // the entropy-coded segment ends at the first marker that is neither stuffing (FF 00) nor RSTn
    I->scan_offset = p;
    int64_t q = p;
    for (;;) {
        const uint8_t *f = q < n ? static_cast<const uint8_t *>(memchr(d + q, 0xFF, (size_t)(n - q))) : nullptr;
        if (!f) { q = n; break; }
        q = f - d;
        if (q + 1 >= n) { q = n; break; }
        const int nx = d[q + 1];
        if (nx == 0x00 || (nx >= 0xD0 && nx <= 0xD7)) { q += 2; continue; }
        if (nx == 0xFF) { q += 1; continue; }
        break;
    }
    I->scan_bytes = q - p;
    if (I->scan_bytes <= 0) return IBT_E_INVALID;
    return ibt::jpeg_validate(I);
}

IBT_API int64_t ibt_jpeg_workspace_bytes(const ibt_jpeg_info_t *I)
{
    if (ibt::jpeg_validate(I) != IBT_OK) return 0;
    ibt::JpgLayout L;
    ibt::jpeg_layout(I, L);
    return (int64_t)L.total;
}

// Shared body of ibt_jpeg_decode / ibt_jpeg_decode_async.  fixed_rounds == 0: synchronous form (rounds in batches, the host
// reads the change counters after each batch and stops at the fixed point).  fixed_rounds > 0: exactly that many rounds are
// enqueued (a round after the fixed point changes nothing and costs a few microseconds), the change counters travel to
// h_pinned[0 .. fixed_rounds) and the function returns without waiting: the caller checks them later.
static int jpeg_decode_impl(const uint8_t *d_file, const ibt_jpeg_info_t *I, void *d_ws, int64_t ws_bytes, uint8_t *d_rgb,
                            int64_t rgb_pitch, uint8_t *d_gray, int64_t gray_pitch, int coeffset, int *out_rounds,
                            int fixed_rounds, uint8_t *h_pinned, void *stream)
{
    using namespace ibt;
    int rc = jpeg_validate(I);
    if (rc) return rc;
    if (!d_file || !d_ws || (!d_rgb && !d_gray)) return IBT_E_INVALID;
    if (d_rgb && (I->ncomp != 3 || rgb_pitch < (int64_t)I->width * 3)) return IBT_E_INVALID;
    if (d_gray && gray_pitch < I->width) return IBT_E_INVALID;
    if (coeffset != IBT_GRAY_CV4_15BIT && coeffset != IBT_GRAY_CV3_14BIT) return IBT_E_INVALID;
    if (reinterpret_cast<uintptr_t>(d_ws) % 256 != 0) return IBT_E_INVALID;
    if (fixed_rounds < 0 || fixed_rounds > JPG_MAX_ROUNDS_BATCH) return IBT_E_INVALID;
    static thread_local JpgLayout L;                        // ~1 KB of geometry, reused as a kernel parameter below
    jpeg_layout(I, L);
    if ((size_t)ws_bytes < L.total) return IBT_E_WORKSPACE;
    // pinned staging: [0, 256) round counters read back, then the Huffman tables on their way to the device.  The synchronous
    // form owns a per-thread buffer (it synchronises the stream before it returns, so the staging is free again at the next
    // call); the asynchronous form uses the caller's (free again when the caller has seen the stream pass this decode).
    if (!h_pinned) {
        static thread_local uint8_t *h_own = nullptr;
        if (!h_own) IBT_CUDA_TRY(cudaHostAlloc(reinterpret_cast<void **>(&h_own), 256 + sizeof(JpgTables), cudaHostAllocDefault));
        h_pinned = h_own;
    }
    uint32_t *h_flag = reinterpret_cast<uint32_t *>(h_pinned);
    JpgTables &T = *reinterpret_cast<JpgTables *>(h_pinned + 256);
    rc = build_tables(I, L.G, T);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    uint8_t *ws = static_cast<uint8_t *>(d_ws);
    uint8_t *sbytes = ws + L.off_stream;
    const uint32_t *words = reinterpret_cast<const uint32_t *>(sbytes);
    uint32_t *counts = reinterpret_cast<uint32_t *>(ws + L.off_counts), *offsets = reinterpret_cast<uint32_t *>(ws + L.off_offsets);
    uint32_t *meta = reinterpret_cast<uint32_t *>(ws + L.off_meta), *changed = reinterpret_cast<uint32_t *>(ws + L.off_changed);
    unsigned long long *start = reinterpret_cast<unsigned long long *>(ws + L.off_start);
    uint8_t *dirty = ws + L.off_dirty;
    unsigned long long *qstart = reinterpret_cast<unsigned long long *>(ws + L.off_qstart);
    uint32_t *nblk = reinterpret_cast<uint32_t *>(ws + L.off_nblk), *base = reinterpret_cast<uint32_t *>(ws + L.off_base);
    uint32_t *partial = reinterpret_cast<uint32_t *>(ws + L.off_partial);
    int16_t *coef = reinterpret_cast<int16_t *>(ws + L.off_coef);
    uint32_t *dcs = reinterpret_cast<uint32_t *>(ws + L.off_dcs), *dcpre = reinterpret_cast<uint32_t *>(ws + L.off_dcpre);
    for (int c = 0; c < I->ncomp; c++) L.G.plane[c] = ws + L.off_plane[c];
    const uint8_t *scan = d_file + I->scan_offset;

    const JpgTables *dT = reinterpret_cast<const JpgTables *>(ws + L.off_tables);
    IBT_CUDA_TRY(cudaMemcpyAsync(ws + L.off_tables, &T, sizeof(JpgTables), cudaMemcpyHostToDevice, st));
    // 1. destuff
    IBT_CUDA_TRY(cudaMemsetAsync(sbytes, 0, L.stream_bytes, st));
    IBT_CUDA_TRY(cudaMemsetAsync(coef, 0, L.coef_bytes, st));
    jpg_destuff_count<<<L.nchunks, 256, 0, st>>>(scan, I->scan_bytes, counts);
    launch_scan(counts, offsets, partial, L.nchunks, 1, 0, nullptr, st);
    uint32_t *rst = L.rst_bytes ? reinterpret_cast<uint32_t *>(ws + L.off_rst) : nullptr;
    if (rst) IBT_CUDA_TRY(cudaMemsetAsync(rst, 0, L.rst_bytes, st));
    jpg_destuff_write<<<L.nchunks, 256, 0, st>>>(scan, I->scan_bytes, offsets, sbytes, meta, rst);

    // 2. synchronisation rounds; the host reads the per-round change counters once per batch
    static const bool no_probe = getenv("IBT_JPEG_NO_PROBE") != nullptr;       // A/B switch for the measurements in profiles/
    if (L.G.nblk_mcu > 1 && !no_probe && jpeg_probe_enabled.load(std::memory_order_relaxed)) {
        unsigned long long *exits = reinterpret_cast<unsigned long long *>(ws + L.off_exits);
        const int P = L.G.nblk_mcu;
        jpg_sync_probe<<<(L.nsub * P + 127) / 128, 128, 0, st>>>(words, meta, dT, exits, L.nsub, P, rst, L.sbits);
        jpg_sync_vote<<<(L.nsub + 255) / 256, 256, 0, st>>>(exits, start, dirty, L.nsub, P);
    } else {
        jpg_sync_init<<<(L.nsub + 255) / 256, 256, 0, st>>>(start, dirty, L.nsub, L.sbits);
    }
    const int sync_ctas = (L.nsub + 127) / 128;
    if (fixed_rounds > 0) {
        IBT_CUDA_TRY(cudaMemsetAsync(changed, 0, JPG_MAX_ROUNDS_BATCH * 4, st));
        for (int r = 0; r < fixed_rounds; r++)
            jpg_sync_round<<<sync_ctas, 128, 0, st>>>(words, meta, dT, start, qstart, dirty, nblk, L.nsub, r, changed + r, rst, L.sbits);
        IBT_CUDA_TRY(cudaMemcpyAsync(h_flag, changed, (size_t)fixed_rounds * 4, cudaMemcpyDeviceToHost, st));
        rc = check_launch("jpeg sync");
        if (rc) return rc;
    } else {
        // first batch: the caller's hint (rounds the previous, similar file needed) + 2, else 8
        int round = 0, batch = 8, rounds_used = -1;
        if (out_rounds && *out_rounds > 0) batch = *out_rounds + 2 > JPG_MAX_ROUNDS_BATCH ? JPG_MAX_ROUNDS_BATCH : *out_rounds + 2;
        while (rounds_used < 0) {
            IBT_CUDA_TRY(cudaMemsetAsync(changed, 0, JPG_MAX_ROUNDS_BATCH * 4, st));
            for (int r = 0; r < batch; r++)
                jpg_sync_round<<<sync_ctas, 128, 0, st>>>(words, meta, dT, start, qstart, dirty, nblk, L.nsub, round + r, changed + r, rst, L.sbits);
            IBT_CUDA_TRY(cudaMemcpyAsync(h_flag, changed, (size_t)batch * 4, cudaMemcpyDeviceToHost, st));
            IBT_CUDA_TRY(cudaStreamSynchronize(st));
            for (int r = 0; r < batch; r++)
                if (h_flag[r] == 0) { rounds_used = round + r + 1; break; }     // a round without changes: fixed point reached
            round += batch;
            if (round > L.nsub + 8) break;                                     // cannot happen: one subsequence settles per round
            batch = batch * 2 > JPG_MAX_ROUNDS_BATCH ? JPG_MAX_ROUNDS_BATCH : batch * 2;
        }
        rc = check_launch("jpeg sync");
        if (rc) return rc;
        if (rounds_used < 0) return IBT_E_INVALID;
        if (out_rounds) *out_rounds = rounds_used;
    }

    // 3. output block of every subsequence, coefficient pass
    launch_scan(nblk, base, partial, L.nsub * JPG_Q, 1, 0, nullptr, st);
    jpg_huff_write<<<(L.nsub * JPG_Q + 127) / 128, 128, 0, st>>>(words, meta, dT, qstart, base, coef, L.nsub, (uint32_t)L.nblocks, rst, L.sbits);

    // 4. DC prediction: prefix sums over MCUs per component
    jpg_dc_sums<<<(L.nmcu + 255) / 256, 256, 0, st>>>(coef, L.G, dcs, L.nmcu);
    launch_scan(dcs, dcpre, partial, L.nmcu, I->ncomp, L.nmcu, nullptr, st);

    // 5. inverse DCT into the component planes, 6. upsampling + colour conversion (+ gray)
    jpg_idct<<<(L.nblocks + 127) / 128, 128, 0, st>>>(coef, dcpre, L.G, L.nmcu, L.nblocks);
    const dim3 cgrid((unsigned)((I->width + 8 * 256 - 1) / (8 * 256)), (unsigned)I->height);
    const int mode = I->ncomp == 1 ? 0 : (L.G.hmax == 1 ? 1 : (L.G.vmax == 1 ? 2 : 3));        // grey, 4:4:4, 4:2:2, 4:2:0
#define IBT_JPG_COLOR(SH, K0, K1, K2)                                                                                              \
    switch (mode) {                                                                                                                \
    case 0: jpg_color<SH, 1, 1, 1><<<cgrid, 256, 0, st>>>(L.G, d_rgb, rgb_pitch, d_gray, gray_pitch, K0, K1, K2); break;           \
    case 1: jpg_color<SH, 3, 1, 1><<<cgrid, 256, 0, st>>>(L.G, d_rgb, rgb_pitch, d_gray, gray_pitch, K0, K1, K2); break;           \
    case 2: jpg_color<SH, 3, 2, 1><<<cgrid, 256, 0, st>>>(L.G, d_rgb, rgb_pitch, d_gray, gray_pitch, K0, K1, K2); break;           \
    default: jpg_color<SH, 3, 2, 2><<<cgrid, 256, 0, st>>>(L.G, d_rgb, rgb_pitch, d_gray, gray_pitch, K0, K1, K2); break;          \
    }
    if (coeffset == IBT_GRAY_CV4_15BIT) { IBT_JPG_COLOR(15, 3735, 19235, 9798) }
    else { IBT_JPG_COLOR(14, 1868, 9617, 4899) }
#undef IBT_JPG_COLOR
    return check_launch("ibt_jpeg_decode");
}

IBT_API int ibt_jpeg_decode(const uint8_t *d_file, const ibt_jpeg_info_t *I, void *d_ws, int64_t ws_bytes, uint8_t *d_rgb,
                            int64_t rgb_pitch, uint8_t *d_gray, int64_t gray_pitch, int coeffset, int *out_rounds, void *stream)
{
    return jpeg_decode_impl(d_file, I, d_ws, ws_bytes, d_rgb, rgb_pitch, d_gray, gray_pitch, coeffset, out_rounds, 0, nullptr, stream);
}

IBT_API int64_t ibt_jpeg_async_host_bytes(void) { return 256 + (int64_t)sizeof(ibt::JpgTables); }

IBT_API int ibt_jpeg_decode_async(const uint8_t *d_file, const ibt_jpeg_info_t *I, void *d_ws, int64_t ws_bytes, uint8_t *d_rgb,
                                  int64_t rgb_pitch, uint8_t *d_gray, int64_t gray_pitch, int coeffset, int rounds,
                                  void *h_pinned, int64_t h_pinned_bytes, void *stream)
{
    if (rounds < 1 || !h_pinned || h_pinned_bytes < ibt_jpeg_async_host_bytes()) return IBT_E_INVALID;
    return jpeg_decode_impl(d_file, I, d_ws, ws_bytes, d_rgb, rgb_pitch, d_gray, gray_pitch, coeffset, nullptr, rounds,
                            static_cast<uint8_t *>(h_pinned), stream);
}

// ---- ibt_jpeg_recompress --------------------------------------------------------------------------------------------------
static const uint8_t k_std_luma_q[64] = {16, 11, 10, 16, 24,  40,  51,  61,  12, 12, 14, 19, 26,  58,  60,  55,
                                         14, 13, 16, 24, 40,  57,  69,  56,  14, 17, 22, 29, 51,  87,  80,  62,
                                         18, 22, 37, 56, 68,  109, 103, 77,  24, 35, 55, 64, 81,  104, 113, 92,
                                         49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99};
static const uint8_t k_std_chroma_q[64] = {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99,
                                           24, 26, 56, 99, 99, 99, 99, 99, 47, 66, 99, 99, 99, 99, 99, 99,
                                           99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99,
                                           99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99};

static bool recompress_args_ok(int W, int H, int hs, int vs)
{
    if (W <= 0 || H <= 0 || W > 65535 || H > 65535) return false;
    return (hs == 1 && vs == 1) || (hs == 2 && vs == 1) || (hs == 2 && vs == 2);
}

IBT_API int64_t ibt_jpeg_recompress_workspace_bytes(int width, int height, int hsamp, int vsamp)
{
    if (!recompress_args_ok(width, height, hsamp, vsamp)) return 0;
    ibt::JpgLayout L;
    ibt::recompress_layout(width, height, hsamp, vsamp, L);
    return (int64_t)L.total;
}

IBT_API int ibt_jpeg_recompress(const uint8_t *d_rgb_in, int64_t in_pitch, int width, int height, int quality, int hsamp, int vsamp,
                                void *d_ws, int64_t ws_bytes, uint8_t *d_rgb, int64_t rgb_pitch, uint8_t *d_gray, int64_t gray_pitch,
                                int coeffset, void *stream)
{
    using namespace ibt;
    if (!recompress_args_ok(width, height, hsamp, vsamp)) return IBT_E_INVALID;
    if (!d_rgb_in || !d_ws || (!d_rgb && !d_gray) || in_pitch < (int64_t)width * 3) return IBT_E_INVALID;
    if (d_rgb && rgb_pitch < (int64_t)width * 3) return IBT_E_INVALID;
    if (d_gray && gray_pitch < width) return IBT_E_INVALID;
    if (coeffset != IBT_GRAY_CV4_15BIT && coeffset != IBT_GRAY_CV3_14BIT) return IBT_E_INVALID;
    if (reinterpret_cast<uintptr_t>(d_ws) % 256 != 0) return IBT_E_INVALID;
    static thread_local JpgLayout L;
    recompress_layout(width, height, hsamp, vsamp, L);
    if ((size_t)ws_bytes < L.total) return IBT_E_WORKSPACE;
    // jcparam.c: jpeg_quality_scaling + jpeg_add_quant_table(force_baseline)
    if (quality <= 0) quality = 1;
    if (quality > 100) quality = 100;
    const int scale = quality < 50 ? 5000 / quality : 200 - quality * 2;
    JpgEncQ Q;
    for (int t = 0; t < 2; t++)
        for (int i = 0; i < 64; i++) {
            long v = ((long)(t ? k_std_chroma_q[i] : k_std_luma_q[i]) * scale + 50) / 100;
            v = v < 1 ? 1 : (v > 255 ? 255 : v);
            Q.q[t][i] = (uint16_t)v;
            Q.magic[t][i] = (uint32_t)(0x100000000ull / (unsigned long long)(v * 8)) + 1u;
            L.G.quant[t][i] = (uint16_t)v;
        }
    for (int i = 0; i < 64; i++) L.G.quant[2][i] = L.G.quant[1][i];
    uint8_t *ws = static_cast<uint8_t *>(d_ws);
    for (int c = 0; c < 3; c++) L.G.plane[c] = ws + L.off_plane[c];
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const dim3 pgrid((unsigned)((L.G.pw[0] / 8 + 255) / 256), (unsigned)L.G.ph[1]);
    if (hsamp == 1) jpg_enc_planes<1, 1><<<pgrid, 256, 0, st>>>(d_rgb_in, in_pitch, L.G);
    else if (vsamp == 1) jpg_enc_planes<2, 1><<<pgrid, 256, 0, st>>>(d_rgb_in, in_pitch, L.G);
    else jpg_enc_planes<2, 2><<<pgrid, 256, 0, st>>>(d_rgb_in, in_pitch, L.G);
    int total_blocks = 0;
    for (int c = 0; c < 3; c++) total_blocks += L.G.bw[c] * L.G.bh[c];
    jpg_enc_requant<<<(total_blocks + 127) / 128, 128, 0, st>>>(L.G, Q, total_blocks);
    const dim3 cgrid((unsigned)((width + 8 * 256 - 1) / (8 * 256)), (unsigned)height);
    const int mode = hsamp == 1 ? 1 : (vsamp == 1 ? 2 : 3);
#define IBT_JPG_COLOR(SH, K0, K1, K2)                                                                                              \
    switch (mode) {                                                                                                                \
    case 1: jpg_color<SH, 3, 1, 1><<<cgrid, 256, 0, st>>>(L.G, d_rgb, rgb_pitch, d_gray, gray_pitch, K0, K1, K2); break;           \
    case 2: jpg_color<SH, 3, 2, 1><<<cgrid, 256, 0, st>>>(L.G, d_rgb, rgb_pitch, d_gray, gray_pitch, K0, K1, K2); break;           \
    default: jpg_color<SH, 3, 2, 2><<<cgrid, 256, 0, st>>>(L.G, d_rgb, rgb_pitch, d_gray, gray_pitch, K0, K1, K2); break;          \
    }
    if (coeffset == IBT_GRAY_CV4_15BIT) { IBT_JPG_COLOR(15, 3735, 19235, 9798) }
    else { IBT_JPG_COLOR(14, 1868, 9617, 4899) }
#undef IBT_JPG_COLOR
    return check_launch("ibt_jpeg_recompress");
}

IBT_API int ibt_jpeg_set_probe(int enabled)
{
    ibt::jpeg_probe_enabled.store(enabled != 0, std::memory_order_relaxed);
    return IBT_OK;
}
