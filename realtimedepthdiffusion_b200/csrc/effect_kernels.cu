// GPUDepthEffect kernels: desaturation, haze, defocus -- separately or fused into
// one read of image + gray + depth.
//
// Arithmetic contract (from the PTX of the reference, SURVEY.md Appendix A):
//   desaturation: f = div.rn(d, 255); out_c = cvt.rzi(fma(f, gray, (1 - f) * orig_c)) & 0xFF
//   haze        : t = expf(div.rn(-2 d, 255)); out_c = cvt.rzi(fma(t, orig_c, (1 - t) * 255)) & 0xFF
//   defocus     : K = (int)(0.025 * (double)sqrtf((float)(rows^2 + cols^2)));
//                 a = cvt.rzi.s32.f64((double)(K * d) / 255.0); h = a / 2;
//                 mean of orig over [y-h, y+h) x [x-h, x+h) clipped to the image,
//                 out_c = cvt.rzi(div.rn(sum_c, count)) & 0xFF; empty window -> copy orig.
// The reference gathers the window tap by tap (up to 110^2 taps per pixel at 4K) in
// fp32; those sums are exact integers while count * 255 < 2^24, so an integer
// summed-area table reproduces them bit for bit with 4 corner reads.  Windows
// larger than that (only possible beyond ~10K-pixel diagonals) fall back to the
// reference's raster-order fp32 accumulation to stay bit-exact.
//
// ref: src/GPUDepthEffect.cu:8-123.

#include "rtdd_internal.h"

#include <math.h>

namespace rtdd {

__device__ __forceinline__ unsigned int f2u8(float v) { return __float2uint_rz(v) & 0xFFu; }
__device__ __forceinline__ int rtdd_div_up_dev(int a, int b) { return (a + b - 1) / b; }

// ---------------------------------------------------------------------------
// summed-area table of the BGR image: S[y][x] = sum over rows < y, cols < x,
// (rows+1) x (cols+1) uint4 {B, G, R, 0}; u32 wrap-around is harmless because
// every window sum that is used is < 2^32.
// Pass 0 (round 2, three small kernels): per group of SAT_G rows, the column sums of the IMAGE strip, prefixed along x = what the
//         group adds to every table row below it; an exclusive scan over the groups turns them into each group's start values
//         (1.5 MB at 4K).
// Pass A: row prefix sums.  Pass B: column prefix within a group, STARTING from the group's start values -- so the table is
// final and a lookup is ONE 16-byte read per corner (round 1 added a per-group offset at every lookup: 8 reads per pixel).
// ---------------------------------------------------------------------------
#define SAT_G 16

__global__ void __launch_bounds__(256)
sat_rows_kernel(const uint8_t *__restrict__ orig, size_t origPitch, uint4 *__restrict__ sat, int rows, int cols)
{
    // one CTA per image row; chunks of 1024 pixels (4 per thread); ONE barrier per chunk: the warp totals are double buffered and
    // every thread accumulates the running carry itself
    __shared__ uint3 sWarp[2][8];
    const int y = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int satPitch = cols + 1;
    uint4 *outRow = sat + (size_t)(y + 1) * satPitch;
    if (y == 0)
        for (int x = threadIdx.x; x <= cols; x += blockDim.x) sat[x] = make_uint4(0, 0, 0, 0);
    if (threadIdx.x == 0) outRow[0] = make_uint4(0, 0, 0, 0);
    const uint8_t *row = orig + (size_t)y * origPitch;
    const bool vec = ((((uintptr_t)orig | origPitch) & 3u) == 0);
    uint3 carry = make_uint3(0, 0, 0);
    int buf = 0;
    for (int base = 0; base < cols; base += 256 * 4, buf ^= 1) {
        const int x0 = base + threadIdx.x * 4;
        unsigned int b[4] = {0, 0, 0, 0}, g[4] = {0, 0, 0, 0}, r[4] = {0, 0, 0, 0};
        if (vec && x0 + 4 <= cols) {
            const unsigned int *p = (const unsigned int *)(row + 3 * x0);
            const unsigned int w[3] = {__ldg(p), __ldg(p + 1), __ldg(p + 2)};
#pragma unroll
            for (int i = 0; i < 12; i++) {
                const unsigned int v = (w[i >> 2] >> (8 * (i & 3))) & 0xFFu;
                if (i % 3 == 0) b[i / 3] = v; else if (i % 3 == 1) g[i / 3] = v; else r[i / 3] = v;
            }
        } else {
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int x = x0 + i;
                if (x < cols) { b[i] = __ldg(row + 3 * x); g[i] = __ldg(row + 3 * x + 1); r[i] = __ldg(row + 3 * x + 2); }
            }
        }
#pragma unroll
        for (int i = 1; i < 4; i++) { b[i] += b[i - 1]; g[i] += g[i - 1]; r[i] += r[i - 1]; }
        uint3 tot = make_uint3(b[3], g[3], r[3]);
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned int tb = __shfl_up_sync(0xFFFFFFFFu, tot.x, d);
            const unsigned int tg = __shfl_up_sync(0xFFFFFFFFu, tot.y, d);
            const unsigned int tr = __shfl_up_sync(0xFFFFFFFFu, tot.z, d);
            if (lane >= d) { tot.x += tb; tot.y += tg; tot.z += tr; }
        }
        if (lane == 31) sWarp[buf][warp] = tot;
        __syncthreads();
        uint3 off = carry, all = make_uint3(0, 0, 0);
#pragma unroll
        for (int w = 0; w < 8; w++) {
            const uint3 t = sWarp[buf][w];
            if (w < warp) { off.x += t.x; off.y += t.y; off.z += t.z; }
            all.x += t.x; all.y += t.y; all.z += t.z;
        }
        // exclusive prefix of this thread = inclusive warp scan - own total + offsets
        off.x += tot.x - b[3]; off.y += tot.y - g[3]; off.z += tot.z - r[3];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int x = x0 + i;
            if (x < cols) outRow[x + 1] = make_uint4(off.x + b[i], off.y + g[i], off.z + r[i], 0u);
        }
        carry.x += all.x; carry.y += all.y; carry.z += all.z;
    }
}

// Pass 0a: aux[g][x + 1] = sum over the rows of group g of image column x (per channel).  Grid: (column chunks, groups).
__global__ void __launch_bounds__(128)
sat_group_colsums_kernel(const uint8_t *__restrict__ orig, size_t origPitch, uint4 *__restrict__ aux, int rows, int cols)
{
    const int g = blockIdx.y;
    const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    const int satPitch = cols + 1;
    uint4 *outRow = aux + (size_t)g * satPitch;
    if (blockIdx.x == 0 && threadIdx.x == 0) outRow[0] = make_uint4(0, 0, 0, 0);
    if (x0 >= cols) return;
    const int yBeg = g * SAT_G, yEnd = min(yBeg + SAT_G, rows);
    const bool vec = ((((uintptr_t)orig | origPitch) & 3u) == 0) && (x0 + 4 <= cols);
    unsigned int b[4] = {0, 0, 0, 0}, gg[4] = {0, 0, 0, 0}, r[4] = {0, 0, 0, 0};
#pragma unroll 8
    for (int y = yBeg; y < yEnd; y++) {
        const uint8_t *row = orig + (size_t)y * origPitch + 3 * x0;
        if (vec) {
            const unsigned int w0 = __ldg((const unsigned int *)row), w1 = __ldg((const unsigned int *)row + 1), w2 = __ldg((const unsigned int *)row + 2);
            const unsigned int w[3] = {w0, w1, w2};
#pragma unroll
            for (int i = 0; i < 12; i++) {
                const unsigned int v = (w[i >> 2] >> (8 * (i & 3))) & 0xFFu;
                if (i % 3 == 0) b[i / 3] += v; else if (i % 3 == 1) gg[i / 3] += v; else r[i / 3] += v;
            }
        } else {
            for (int i = 0; i < 4 && x0 + i < cols; i++) { b[i] += __ldg(row + 3 * i); gg[i] += __ldg(row + 3 * i + 1); r[i] += __ldg(row + 3 * i + 2); }
        }
    }
    for (int i = 0; i < 4 && x0 + i < cols; i++) outRow[x0 + i + 1] = make_uint4(b[i], gg[i], r[i], 0u);
}

// Pass 0b: inclusive prefix along x of every aux row, in place (one CTA per group): aux[g][x] = what group g adds to column x of
// every table row below it.  Pass 0c (sat_aux_kernel) then scans over the groups.
__global__ void __launch_bounds__(256)
sat_group_prefix_kernel(uint4 *__restrict__ aux, int cols)
{
    __shared__ uint3 sWarp[8];
    __shared__ uint3 sCarry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint4 *row = aux + (size_t)blockIdx.x * (cols + 1);
    if (threadIdx.x == 0) sCarry = make_uint3(0, 0, 0);
    __syncthreads();
    for (int base = 1; base <= cols; base += 256 * 4) {
        const int x0 = base + threadIdx.x * 4;
        uint4 v[4];
#pragma unroll
        for (int i = 0; i < 4; i++) v[i] = (x0 + i <= cols) ? row[x0 + i] : make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int i = 1; i < 4; i++) { v[i].x += v[i - 1].x; v[i].y += v[i - 1].y; v[i].z += v[i - 1].z; }
        uint3 tot = make_uint3(v[3].x, v[3].y, v[3].z);
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned int tb = __shfl_up_sync(0xFFFFFFFFu, tot.x, d);
            const unsigned int tg = __shfl_up_sync(0xFFFFFFFFu, tot.y, d);
            const unsigned int tr = __shfl_up_sync(0xFFFFFFFFu, tot.z, d);
            if (lane >= d) { tot.x += tb; tot.y += tg; tot.z += tr; }
        }
        if (lane == 31) sWarp[warp] = tot;
        __syncthreads();
        uint3 off = sCarry;
        for (int w = 0; w < warp; w++) { off.x += sWarp[w].x; off.y += sWarp[w].y; off.z += sWarp[w].z; }
        off.x += tot.x - v[3].x; off.y += tot.y - v[3].y; off.z += tot.z - v[3].z;
#pragma unroll
        for (int i = 0; i < 4; i++)
            if (x0 + i <= cols) row[x0 + i] = make_uint4(off.x + v[i].x, off.y + v[i].y, off.z + v[i].z, 0u);
        __syncthreads();
        if (threadIdx.x == 255) sCarry = make_uint3(off.x + v[3].x, off.y + v[3].y, off.z + v[3].z);
        __syncthreads();
    }
}

// Passes A + B in one (round 2): one CTA of 1024 threads per group of SAT_G rows writes the FINAL table rows of its group.  A
// thread owns 4 columns per 4096-column chunk and keeps their running column sums in registers, starting from the group's start
// values (aux after passes 0a-0c); per image row it forms the row prefix of its pixels (local prefix, warp scan, one
// shared-memory hand-off between the 32 warps -- ONE barrier per row, the warp totals are double buffered), adds it to the
// column sums and stores the table row.  The table is written exactly once (133 MB at 4K) and never read during the build;
// round 1's two passes wrote it twice and read it once.
#define SAT_CHUNKS 4                      // 4 x 4096 = 16384 columns at most
template <int NCH>                        // chunks of 4096 columns a thread carries column sums for (12 registers each)
__global__ void __launch_bounds__(1024, 1)
sat_fused_kernel(const uint8_t *__restrict__ orig, size_t origPitch, uint4 *__restrict__ sat, const uint4 *__restrict__ aux, int rows, int cols)
{
    __shared__ uint3 sWarp[2][32];
    const int g = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int satPitch = cols + 1;
    const int yBeg = g * SAT_G, yEnd = min(yBeg + SAT_G, rows);
    const int nchunks = rtdd_div_up_dev(cols, 4096);        // <= NCH
    const bool vecOk = ((((uintptr_t)orig | origPitch) & 3u) == 0);
    if (g == 0)
        for (int x = threadIdx.x; x <= cols; x += blockDim.x) sat[x] = make_uint4(0, 0, 0, 0);      // table row 0
    uint3 acc[NCH][4];
#pragma unroll
    for (int c = 0; c < NCH; c++)
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int x = c * 4096 + threadIdx.x * 4 + i;
            const uint4 v = (c < nchunks && x < cols) ? __ldg(aux + (size_t)g * satPitch + x + 1) : make_uint4(0, 0, 0, 0);
            acc[c][i] = make_uint3(v.x, v.y, v.z);
        }
    int buf = 0;
    // the 12 pixel bytes of a thread's 4 columns, one row ahead: a row's loads are in flight while the previous row is scanned
    // (without this a row cost ~4 us: DRAM latency + the scan, serially)
    auto load_words = [&](int y, int c, unsigned int (&w)[3]) {
        const int x0 = c * 4096 + threadIdx.x * 4;
        const uint8_t *row = orig + (size_t)y * origPitch;
        w[0] = w[1] = w[2] = 0u;
        if (y >= yEnd || c >= nchunks || x0 >= cols) return;
        if (vecOk && x0 + 4 <= cols) {
            const unsigned int *p = (const unsigned int *)(row + 3 * x0);
            w[0] = __ldg(p); w[1] = __ldg(p + 1); w[2] = __ldg(p + 2);
        } else {
            unsigned int bytes[12];
#pragma unroll
            for (int i = 0; i < 12; i++) bytes[i] = (x0 + i / 3 < cols) ? (unsigned int)__ldg(row + 3 * x0 + i) : 0u;
#pragma unroll
            for (int i = 0; i < 12; i++) w[i >> 2] |= bytes[i] << (8 * (i & 3));
        }
    };
    unsigned int nxt[NCH][3];
#pragma unroll
    for (int c = 0; c < NCH; c++) load_words(yBeg, c, nxt[c]);
    for (int y = yBeg; y < yEnd; y++) {
        uint4 *outRow = sat + (size_t)(y + 1) * satPitch;
        if (threadIdx.x == 0) outRow[0] = make_uint4(0, 0, 0, 0);
        unsigned int cur[NCH][3];
#pragma unroll
        for (int c = 0; c < NCH; c++) { cur[c][0] = nxt[c][0]; cur[c][1] = nxt[c][1]; cur[c][2] = nxt[c][2]; }
#pragma unroll
        for (int c = 0; c < NCH; c++) load_words(y + 1, c, nxt[c]);
        uint3 carry = make_uint3(0, 0, 0);
#pragma unroll
        for (int c = 0; c < NCH; c++) {
            if (c >= nchunks) break;
            const int x0 = c * 4096 + threadIdx.x * 4;
            unsigned int b[4], gg[4], r[4];
#pragma unroll
            for (int i = 0; i < 12; i++) {
                const unsigned int v = (cur[c][i >> 2] >> (8 * (i & 3))) & 0xFFu;
                if (i % 3 == 0) b[i / 3] = v; else if (i % 3 == 1) gg[i / 3] = v; else r[i / 3] = v;
            }
#pragma unroll
            for (int i = 1; i < 4; i++) { b[i] += b[i - 1]; gg[i] += gg[i - 1]; r[i] += r[i - 1]; }
            uint3 tot = make_uint3(b[3], gg[3], r[3]);
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned int tb = __shfl_up_sync(0xFFFFFFFFu, tot.x, d);
                const unsigned int tg = __shfl_up_sync(0xFFFFFFFFu, tot.y, d);
                const unsigned int tr = __shfl_up_sync(0xFFFFFFFFu, tot.z, d);
                if (lane >= d) { tot.x += tb; tot.y += tg; tot.z += tr; }
            }
            if (lane == 31) sWarp[buf][warp] = tot;
            __syncthreads();
            // every warp scans the 32 warp totals itself: lane l holds the inclusive prefix over warps 0..l
            uint3 wt = sWarp[buf][lane];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned int tb = __shfl_up_sync(0xFFFFFFFFu, wt.x, d);
                const unsigned int tg = __shfl_up_sync(0xFFFFFFFFu, wt.y, d);
                const unsigned int tr = __shfl_up_sync(0xFFFFFFFFu, wt.z, d);
                if (lane >= d) { wt.x += tb; wt.y += tg; wt.z += tr; }
            }
            const unsigned int pbx = __shfl_sync(0xFFFFFFFFu, wt.x, warp > 0 ? warp - 1 : 0);
            const unsigned int pgx = __shfl_sync(0xFFFFFFFFu, wt.y, warp > 0 ? warp - 1 : 0);
            const unsigned int prx = __shfl_sync(0xFFFFFFFFu, wt.z, warp > 0 ? warp - 1 : 0);
            const unsigned int allb = __shfl_sync(0xFFFFFFFFu, wt.x, 31), allg = __shfl_sync(0xFFFFFFFFu, wt.y, 31), allr = __shfl_sync(0xFFFFFFFFu, wt.z, 31);
            uint3 off = carry;
            if (warp > 0) { off.x += pbx; off.y += pgx; off.z += prx; }
            off.x += tot.x - b[3]; off.y += tot.y - gg[3]; off.z += tot.z - r[3];     // exclusive prefix of this thread's first pixel
#pragma unroll
            for (int i = 0; i < 4; i++) {
                acc[c][i].x += off.x + b[i]; acc[c][i].y += off.y + gg[i]; acc[c][i].z += off.z + r[i];
                if (x0 + i < cols) outRow[x0 + i + 1] = make_uint4(acc[c][i].x, acc[c][i].y, acc[c][i].z, 0u);
            }
            carry.x += allb; carry.y += allg; carry.z += allr;
            buf ^= 1;
        }
    }
}

// Pass B of the two-pass form (images wider than 16384 columns): column prefix inside group g, starting from the group's start values
__global__ void __launch_bounds__(128)
sat_cols_kernel(uint4 *__restrict__ sat, const uint4 *__restrict__ aux, int rows, int cols)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int g = blockIdx.y;
    if (x > cols) return;
    const int satPitch = cols + 1;
    const int yBeg = g * SAT_G + 1;
    const int yEnd = min(yBeg + SAT_G, rows + 1);
    uint4 acc = __ldg(aux + (size_t)g * satPitch + x);
#pragma unroll 8
    for (int y = yBeg; y < yEnd; y++) {
        uint4 *p = sat + (size_t)y * satPitch + x;
        const uint4 v = *p;
        acc.x += v.x; acc.y += v.y; acc.z += v.z;
        *p = acc;
    }
}

// Pass 0c: exclusive scan over the groups, per column: aux[g][x] := sum of aux[g'][x] for g' < g.  One CTA = 32 columns x 8 warps;
// warp w owns a segment of the groups: segment totals first (independent loads), a shared-memory hand-off, then the running
// sums (the serial 135-step loop per column of the first version took 70 us at 4K)
__global__ void __launch_bounds__(256)
sat_aux_kernel(uint4 *__restrict__ aux, int groups, int cols)
{
    __shared__ uint3 sTot[8][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x = blockIdx.x * 32 + lane;
    const int satPitch = cols + 1;
    const int seg = (groups + 7) / 8;
    const int g0 = warp * seg, g1 = min(g0 + seg, groups);
    uint3 tot = make_uint3(0, 0, 0);
    if (x <= cols) {
#pragma unroll 4
        for (int g = g0; g < g1; g++) {
            const uint4 v = aux[(size_t)g * satPitch + x];
            tot.x += v.x; tot.y += v.y; tot.z += v.z;
        }
    }
    sTot[warp][lane] = tot;
    __syncthreads();
    if (x > cols) return;
    uint3 acc = make_uint3(0, 0, 0);
    for (int w = 0; w < warp; w++) { acc.x += sTot[w][lane].x; acc.y += sTot[w][lane].y; acc.z += sTot[w][lane].z; }
#pragma unroll 4
    for (int g = g0; g < g1; g++) {
        uint4 *p = aux + (size_t)g * satPitch + x;
        const uint4 v = *p;
        *p = make_uint4(acc.x, acc.y, acc.z, 0u);          // exclusive: start values of group g
        acc.x += v.x; acc.y += v.y; acc.z += v.z;
    }
}

__device__ __forceinline__ uint4 sat_at(const uint4 *__restrict__ sat, const uint4 *__restrict__ aux, int satPitch, int y, int x)
{
    (void)aux;                                   // group start values are folded into the table at build time
    return __ldg(sat + (size_t)y * satPitch + x);     // row 0 of the table is zero
}

// ---------------------------------------------------------------------------
// the per-pixel effect kernel: any subset of {desaturation, haze, defocus} from a
// single read of orig (3 B) + gray (1 B) + depth (4 B).  One thread = 4 pixels;
// when every plane is 4-byte aligned (16 for depth) the 12 colour bytes move as
// three 32-bit words.
// ---------------------------------------------------------------------------
template <bool ALIGNED>
__device__ __forceinline__ void load_bgr4(const uint8_t *__restrict__ p, int n, unsigned int (&c)[4][3])
{
    if (ALIGNED && n == 4) {
        const unsigned int w0 = __ldg((const unsigned int *)p);
        const unsigned int w1 = __ldg((const unsigned int *)p + 1);
        const unsigned int w2 = __ldg((const unsigned int *)p + 2);
        const unsigned int w[3] = {w0, w1, w2};
#pragma unroll
        for (int i = 0; i < 12; i++) c[i / 3][i % 3] = (w[i >> 2] >> (8 * (i & 3))) & 0xFFu;
    } else {
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
            for (int k = 0; k < 3; k++) c[i][k] = (i < n) ? (unsigned int)__ldg(p + 3 * i + k) : 0u;
    }
}

template <bool ALIGNED>
__device__ __forceinline__ void store_bgr4(uint8_t *__restrict__ p, int n, const unsigned int (&c)[4][3])
{
    if (ALIGNED && n == 4) {
        unsigned int w[3] = {0u, 0u, 0u};
#pragma unroll
        for (int i = 0; i < 12; i++) w[i >> 2] |= c[i / 3][i % 3] << (8 * (i & 3));
        ((unsigned int *)p)[0] = w[0]; ((unsigned int *)p)[1] = w[1]; ((unsigned int *)p)[2] = w[2];
    } else {
#pragma unroll
        for (int i = 0; i < 4; i++)
            if (i < n) { p[3 * i] = (uint8_t)c[i][0]; p[3 * i + 1] = (uint8_t)c[i][1]; p[3 * i + 2] = (uint8_t)c[i][2]; }
    }
}

template <bool ALIGNED, bool DESAT, bool HAZE, bool DEFOCUS>
__global__ void __launch_bounds__(256)
effects_kernel(const uint8_t *__restrict__ orig, size_t origPitch, const uint8_t *__restrict__ gray, size_t grayPitch,
               const float *__restrict__ depth, size_t depthPitch,
               uint8_t *__restrict__ desat, size_t desatPitch, uint8_t *__restrict__ haze, size_t hazePitch,
               uint8_t *__restrict__ defocus, size_t defocusPitch,
               const uint4 *__restrict__ sat, const uint4 *__restrict__ aux, int K, int rows, int cols, int yBegin, int yEnd, int satRow0, int satRows)
{
    // Rows [yBegin, yEnd) of the image are produced (the whole image: 0, rows; a row strip of one GPU: rtdd_effects_rows).  The
    // summed-area table covers image rows [satRow0, satRow0 + satRows); a box that leaves it takes the raster path below.
    const int x4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    const int y = yBegin + blockIdx.y * blockDim.y + threadIdx.y;
    if (x4 >= cols || y >= yEnd) return;
    const int n = min(4, cols - x4);

    unsigned int c[4][3];
    load_bgr4<ALIGNED>(orig + (size_t)y * origPitch + 3 * x4, n, c);
    float d[4];
    {
        const float *dRow = (const float *)((const char *)depth + (size_t)y * depthPitch) + x4;
        if (ALIGNED && n == 4) {
            const float4 v = __ldg((const float4 *)dRow);
            d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
        } else {
#pragma unroll
            for (int i = 0; i < 4; i++) d[i] = (i < n) ? __ldg(dRow + i) : 0.0f;
        }
    }

    if (DESAT) {
        unsigned int g[4];
        const uint8_t *gRow = gray + (size_t)y * grayPitch + x4;
        if (ALIGNED && n == 4) {
            const unsigned int w = __ldg((const unsigned int *)gRow);
#pragma unroll
            for (int i = 0; i < 4; i++) g[i] = (w >> (8 * i)) & 0xFFu;
        } else {
#pragma unroll
            for (int i = 0; i < 4; i++) g[i] = (i < n) ? (unsigned int)__ldg(gRow + i) : 0u;
        }
        unsigned int o[4][3];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const float f = __fdiv_rn(d[i], 255.0f);
            const float f1 = __fsub_rn(1.0f, f);
            const float fg = (float)g[i];
#pragma unroll
            for (int k = 0; k < 3; k++) o[i][k] = f2u8(__fmaf_rn(f, fg, __fmul_rn(f1, (float)c[i][k])));
        }
        store_bgr4<ALIGNED>(desat + (size_t)y * desatPitch + 3 * x4, n, o);
    }

    if (HAZE) {
        unsigned int o[4][3];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const float t = expf(__fdiv_rn(__fmul_rn(d[i], -2.0f), 255.0f));
            const float h = __fmul_rn(__fsub_rn(1.0f, t), 255.0f);
#pragma unroll
            for (int k = 0; k < 3; k++) o[i][k] = f2u8(__fmaf_rn(t, (float)c[i][k], h));
        }
        store_bgr4<ALIGNED>(haze + (size_t)y * hazePitch + 3 * x4, n, o);
    }

    if (DEFOCUS) {
        const int satPitch = cols + 1;
        unsigned int o[4][3];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int x = x4 + i;
            const float kd = __fmul_rn((float)K, d[i]);
            const int a = __double2int_rz(__ddiv_rn((double)kd, 255.0));
            const int h = a / 2;
            o[i][0] = c[i][0]; o[i][1] = c[i][1]; o[i][2] = c[i][2];
            if (i < n && h > 0) {
                const int x0 = max(x - h, 0), x1 = min(x + h, cols);
                const int y0 = max(y - h, 0), y1 = min(y + h, rows);
                // (h > 0 guarantees a non-empty clipped window for an in-image pixel)
                const int count = (x1 - x0) * (y1 - y0);
                float sb, sg, sr;
                if (count <= 65793 && y0 >= satRow0 && y1 <= satRow0 + satRows) {      // count * 255 < 2^24: the reference's fp32 sums are exact integers
                    const uint4 s11 = sat_at(sat, aux, satPitch, y1 - satRow0, x1);
                    const uint4 s01 = sat_at(sat, aux, satPitch, y0 - satRow0, x1);
                    const uint4 s10 = sat_at(sat, aux, satPitch, y1 - satRow0, x0);
                    const uint4 s00 = sat_at(sat, aux, satPitch, y0 - satRow0, x0);
                    sb = (float)(s11.x - s01.x - s10.x + s00.x);
                    sg = (float)(s11.y - s01.y - s10.y + s00.y);
                    sr = (float)(s11.z - s01.z - s10.z + s00.z);
                } else {                   // huge window (or one beyond a strip's table): replay the reference's raster-order fp32 accumulation
                    sb = 0.0f; sg = 0.0f; sr = 0.0f;
                    for (int py = y0; py < y1; py++) {
                        const uint8_t *r = orig + (size_t)py * origPitch;
                        for (int px = x0; px < x1; px++) {
                            sb = __fadd_rn(sb, (float)__ldg(r + 3 * px));
                            sg = __fadd_rn(sg, (float)__ldg(r + 3 * px + 1));
                            sr = __fadd_rn(sr, (float)__ldg(r + 3 * px + 2));
                        }
                    }
                }
                const float fc = (float)count;
                o[i][0] = f2u8(__fdiv_rn(sb, fc));
                o[i][1] = f2u8(__fdiv_rn(sg, fc));
                o[i][2] = f2u8(__fdiv_rn(sr, fc));
            }
        }
        store_bgr4<ALIGNED>(defocus + (size_t)y * defocusPitch + 3 * x4, n, o);
    }
}

static bool aligned4(const void *p, size_t pitch) { return (((uintptr_t)p | pitch) & 3u) == 0; }
static bool aligned16(const void *p, size_t pitch) { return (((uintptr_t)p | pitch) & 15u) == 0; }

template <bool DESAT, bool HAZE, bool DEFOCUS>
static cudaError_t launch_effects(cudaStream_t s, const uint8_t *orig, size_t origPitch, const uint8_t *gray, size_t grayPitch,
                                  const float *depth, size_t depthPitch, uint8_t *desat, size_t desatPitch,
                                  uint8_t *haze, size_t hazePitch, uint8_t *defocus, size_t defocusPitch,
                                  const uint4 *sat, const uint4 *aux, int K, int rows, int cols, int yBegin = 0, int yEnd = -1,
                                  int satRow0 = 0, int satRows = -1)
{
    if (yEnd < 0) yEnd = rows;
    if (satRows < 0) satRows = rows;
    bool al = aligned4(orig, origPitch) && aligned16(depth, depthPitch);
    if (DESAT) al = al && aligned4(gray, grayPitch) && aligned4(desat, desatPitch);
    if (HAZE) al = al && aligned4(haze, hazePitch);
    if (DEFOCUS) al = al && aligned4(defocus, defocusPitch);
    dim3 block(32, 8);
    if (yEnd <= yBegin) return cudaSuccess;
    dim3 grid(rtdd_div_up(rtdd_div_up(cols, 4), block.x), rtdd_div_up(yEnd - yBegin, block.y));
    if (al)
        effects_kernel<true, DESAT, HAZE, DEFOCUS><<<grid, block, 0, s>>>(orig, origPitch, gray, grayPitch, depth, depthPitch,
            desat, desatPitch, haze, hazePitch, defocus, defocusPitch, sat, aux, K, rows, cols, yBegin, yEnd, satRow0, satRows);
    else
        effects_kernel<false, DESAT, HAZE, DEFOCUS><<<grid, block, 0, s>>>(orig, origPitch, gray, grayPitch, depth, depthPitch,
            desat, desatPitch, haze, hazePitch, defocus, defocusPitch, sat, aux, K, rows, cols, yBegin, yEnd, satRow0, satRows);
    return cudaGetLastError();
}

cudaError_t launch_desaturate(cudaStream_t s, const uint8_t *orig, size_t origPitch, const uint8_t *gray, size_t grayPitch,
                              const float *depth, size_t depthPitch, uint8_t *out, size_t outPitch, int rows, int cols)
{
    return launch_effects<true, false, false>(s, orig, origPitch, gray, grayPitch, depth, depthPitch, out, outPitch,
                                              nullptr, 0, nullptr, 0, nullptr, nullptr, 0, rows, cols);
}

cudaError_t launch_haze(cudaStream_t s, const uint8_t *orig, size_t origPitch, const float *depth, size_t depthPitch,
                        uint8_t *out, size_t outPitch, int rows, int cols)
{
    return launch_effects<false, true, false>(s, orig, origPitch, nullptr, 0, depth, depthPitch, nullptr, 0,
                                              out, outPitch, nullptr, 0, nullptr, nullptr, 0, rows, cols);
}

// ref: src/GPUDepthEffect.cu:42 -- evaluated on the host with the same IEEE sqrtf / fp64 multiply
int defocus_kernel_size(int rows, int cols)
{
    const float s = sqrtf((float)(unsigned int)(rows * rows + cols * cols));
    return (int)(0.025 * (double)s);
}

static int sat_groups(int rows) { return rtdd_div_up(rows, SAT_G); }

size_t defocus_scratch_bytes(int rows, int cols)
{
    return ((size_t)(rows + 1) + sat_groups(rows)) * (size_t)(cols + 1) * sizeof(uint4);
}

// the summed-area table depends on the image only: a caller that knows the image is unchanged builds it once
// (rtdd_frame_effects).  Tried: a single table pass (column sums kept in registers while one CTA per 8-row group walks
// down and scans along x; table written once, no per-lookup offset) -- correct, but its serial rows with two CTA barriers
// each made it slower than these three streaming passes (4K defocus 0.270 vs 0.248 ms), so it was not kept.
cudaError_t launch_sat_build(cudaStream_t s, void *scratch, const uint8_t *orig, size_t origPitch, int rows, int cols, int *launched)
{
    uint4 *sat = (uint4 *)scratch;
    uint4 *aux = sat + (size_t)(rows + 1) * (cols + 1);
    const int groups = sat_groups(rows);
    sat_group_colsums_kernel<<<dim3(rtdd_div_up(rtdd_div_up(cols, 4), 128), groups), 128, 0, s>>>(orig, origPitch, aux, rows, cols);
    sat_group_prefix_kernel<<<groups, 256, 0, s>>>(aux, cols);
    sat_aux_kernel<<<rtdd_div_up(cols + 1, 32), 256, 0, s>>>(aux, groups, cols);
    *launched = 4;
    if (cols <= 4096) {
        sat_fused_kernel<1><<<groups, 1024, 0, s>>>(orig, origPitch, sat, aux, rows, cols);
    } else if (cols <= 8192) {
        sat_fused_kernel<2><<<groups, 1024, 0, s>>>(orig, origPitch, sat, aux, rows, cols);
    } else if (cols <= 4096 * SAT_CHUNKS) {
        sat_fused_kernel<SAT_CHUNKS><<<groups, 1024, 0, s>>>(orig, origPitch, sat, aux, rows, cols);
    } else {                 // wider than 16384 columns: the two streaming passes of round 1
        sat_rows_kernel<<<rows, 256, 0, s>>>(orig, origPitch, sat, rows, cols);
        sat_cols_kernel<<<dim3(rtdd_div_up(cols + 1, 128), groups), 128, 0, s>>>(sat, aux, rows, cols);
        *launched = 5;
    }
    return cudaGetLastError();
}

cudaError_t launch_defocus(cudaStream_t s, void *scratch, const uint8_t *orig, size_t origPitch, const uint8_t *gray, size_t grayPitch,
                           const float *depth, size_t depthPitch, uint8_t *defocus, size_t defocusPitch,
                           uint8_t *desat, size_t desatPitch, uint8_t *haze, size_t hazePitch,
                           int rows, int cols, int *launched, bool buildSat, int yBegin, int yEnd, int satRow0, int satRows)
{
    // all planes are the FULL image planes; the summed-area table covers image rows [satRow0, satRow0 + satRows)
    if (yEnd < 0) yEnd = rows;
    if (satRows < 0) { satRow0 = 0; satRows = rows; }
    uint4 *sat = (uint4 *)scratch;
    uint4 *aux = sat + (size_t)(satRows + 1) * (cols + 1);
    const int K = defocus_kernel_size(rows, cols);
    *launched = 0;
    if (buildSat) {
        cudaError_t e = launch_sat_build(s, scratch, orig + (size_t)satRow0 * origPitch, origPitch, satRows, cols, launched);
        if (e != cudaSuccess) return e;
    }
    *launched += 1;
    if (desat && haze)
        return launch_effects<true, true, true>(s, orig, origPitch, gray, grayPitch, depth, depthPitch, desat, desatPitch,
                                                haze, hazePitch, defocus, defocusPitch, sat, aux, K, rows, cols, yBegin, yEnd, satRow0, satRows);
    return launch_effects<false, false, true>(s, orig, origPitch, nullptr, 0, depth, depthPitch, nullptr, 0, nullptr, 0,
                                              defocus, defocusPitch, sat, aux, K, rows, cols, yBegin, yEnd, satRow0, satRows);
}

// ---------------------------------------------------------------------------
// refocus (extension, no reference counterpart): box blur whose side grows with the distance of a pixel's depth from a focus
// plane, over the same summed-area table as defocus.
//   d' = clamp(d, 0, 255) (NaN -> 0); e = max(|d' - f| - w, 0); a = cvt.rzi.s32.f64((double)((float)A * e) / 255.0); h = a / 2;
//   h == 0: copy; else out_c = floor(S_c / N) over [y-h, y+h) x [x-h, x+h) clipped to the image (N pixels).
// A <= 4096 keeps N <= 2^24 and every window sum below 2^32, so the u32 table is exact for every window and there is no raster
// path.  For N <= 65793 (N * 255 < 2^24) the floor is taken as cvt.rzi(div.rn((float)S, (float)N)) -- the defocus pass's
// arithmetic, so f = 0, w = 0, A = K reproduces defocus bit for bit -- and above that as a u32 divide.
// A kernel of its own rather than a fourth flag of effects_kernel: the box rule and the mean rule both differ, so the shared
// kernel would branch on which caller it serves.
// ---------------------------------------------------------------------------
template <bool ALIGNED>
__global__ void __launch_bounds__(256)
refocus_kernel(const uint8_t *__restrict__ orig, size_t origPitch, const float *__restrict__ depth, size_t depthPitch,
               uint8_t *__restrict__ out, size_t outPitch, const uint4 *__restrict__ sat, int rows, int cols,
               float focus, const float *__restrict__ focusAt, float band, int aperture)
{
    const int x4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x4 >= cols || y >= rows) return;
    const int n = min(4, cols - x4);
    // "click to focus": the depth under the chosen pixel, read here so that no host round trip sits between solve and refocus
    if (focusAt) focus = fminf(fmaxf(__ldg(focusAt), 0.0f), 255.0f);

    unsigned int c[4][3];
    load_bgr4<ALIGNED>(orig + (size_t)y * origPitch + 3 * x4, n, c);
    float d[4];
    {
        const float *dRow = (const float *)((const char *)depth + (size_t)y * depthPitch) + x4;
        if (ALIGNED && n == 4) {
            const float4 v = __ldg((const float4 *)dRow);
            d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
        } else {
#pragma unroll
            for (int i = 0; i < 4; i++) d[i] = (i < n) ? __ldg(dRow + i) : 0.0f;
        }
    }

    const int satPitch = cols + 1;
    unsigned int o[4][3];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int x = x4 + i;
        const float dc = fminf(fmaxf(d[i], 0.0f), 255.0f);
        const float e = fmaxf(__fsub_rn(fabsf(__fsub_rn(dc, focus)), band), 0.0f);
        const int a = __double2int_rz(__ddiv_rn((double)__fmul_rn((float)aperture, e), 255.0));
        const int h = a / 2;
        o[i][0] = c[i][0]; o[i][1] = c[i][1]; o[i][2] = c[i][2];
        if (i < n && h > 0) {
            const int x0 = max(x - h, 0), x1 = min(x + h, cols);
            const int y0 = max(y - h, 0), y1 = min(y + h, rows);
            const unsigned int count = (unsigned int)((x1 - x0) * (y1 - y0));
            const uint4 s11 = sat_at(sat, nullptr, satPitch, y1, x1);
            const uint4 s01 = sat_at(sat, nullptr, satPitch, y0, x1);
            const uint4 s10 = sat_at(sat, nullptr, satPitch, y1, x0);
            const uint4 s00 = sat_at(sat, nullptr, satPitch, y0, x0);
            const unsigned int sb = s11.x - s01.x - s10.x + s00.x;
            const unsigned int sg = s11.y - s01.y - s10.y + s00.y;
            const unsigned int sr = s11.z - s01.z - s10.z + s00.z;
            if (count <= 65793u) {
                const float fc = (float)count;
                o[i][0] = f2u8(__fdiv_rn((float)sb, fc));
                o[i][1] = f2u8(__fdiv_rn((float)sg, fc));
                o[i][2] = f2u8(__fdiv_rn((float)sr, fc));
            } else {
                o[i][0] = sb / count; o[i][1] = sg / count; o[i][2] = sr / count;
            }
        }
    }
    store_bgr4<ALIGNED>(out + (size_t)y * outPitch + 3 * x4, n, o);
}

cudaError_t launch_refocus(cudaStream_t s, const void *scratch, const uint8_t *orig, size_t origPitch, const float *depth, size_t depthPitch,
                           uint8_t *out, size_t outPitch, int rows, int cols, float focus, const float *focusAt, float band, int aperture)
{
    const uint4 *sat = (const uint4 *)scratch;
    const bool al = aligned4(orig, origPitch) && aligned16(depth, depthPitch) && aligned4(out, outPitch);
    dim3 block(32, 8);
    dim3 grid(rtdd_div_up(rtdd_div_up(cols, 4), block.x), rtdd_div_up(rows, block.y));
    if (al)
        refocus_kernel<true><<<grid, block, 0, s>>>(orig, origPitch, depth, depthPitch, out, outPitch, sat, rows, cols, focus, focusAt, band, aperture);
    else
        refocus_kernel<false><<<grid, block, 0, s>>>(orig, origPitch, depth, depthPitch, out, outPitch, sat, rows, cols, focus, focusAt, band, aperture);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// stereo (extension, no reference counterpart): left and right views and a red-cyan anaglyph, the image taken as the centre view.
//   d' = clamp(d, 0, 255) (NaN -> 0, -0 -> +0); s = cvt.rzi.s32.f64((double)((float)D * (d' - c)) / 255.0); hL = s / 2; hR = s - hL.
//   Source x lands on tL = x - hL in the left view and on tR = x + hR in the right one.  A target column takes the landing source
//   with the smallest d'; a hole takes the covered neighbour (nearest on each side) whose winner is farther, the left one on a tie;
//   a row with no covered column keeps the image's own pixels.
// Every output row depends on its own source row only, so one CTA takes one row and keeps the row's per-column state in shared
// memory, per view: a z-buffer of d' bits (d' >= 0 with -0 made +0, so the bits order like the values), the winning source
// column, and a two-level bitmap of covered columns (a bit per column, a bit per non-empty word) that finds the nearest covered
// column on either side of a hole in a few instructions, with no scan over the row.  Sources of equal d' have equal s and so
// never land on the same target: the winner of a column is unique, and a u32 atomicMin of the bits followed by "the source whose
// bits equal the minimum writes its x" is exact in any order.  12 B per column + the bitmaps: 196 KB at 16384 columns.
// ---------------------------------------------------------------------------
constexpr int STEREO_THREADS = 512;
constexpr unsigned int STEREO_EMPTY = 0xFFFFFFFFu;       // z-buffer value of a column no source landed on

__device__ __forceinline__ float stereo_depth(float d) { return __fadd_rn(fminf(fmaxf(d, 0.0f), 255.0f), 0.0f); }

// s = cvt.rzi.s32.f64((double)q / 255.0) with q = __fmul_rn(D, d' - c), taken as trunc(q) / 255 in integers: the same value for
// every float q, because the quotient is an integer n exactly when q = 255 n, and otherwise lies at least 2^-31 from every integer
// (|q| >= 1 is a multiple of 2^-23) while its fp64 rounding error is below 2^-42 (|q| / 255 <= 1024).  No fp64 divide in the
// loop, and no call into its slow path.
__device__ __forceinline__ int stereo_parallax(float dc, float conv, float D)
{
    return __float2int_rz(__fmul_rn(D, __fsub_rn(dc, conv))) / 255;
}

// largest covered column <= t, or -1.  b0: a bit per column; b1: a bit per non-zero word of b0; top: a bit per non-zero word of b1
__device__ __forceinline__ int stereo_prev(const unsigned int *b0, const unsigned int *b1, unsigned int top, int t)
{
    int w = t >> 5;
    unsigned int m = b0[w] & (0xFFFFFFFFu >> (31 - (t & 31)));
    if (m) return (w << 5) + 31 - __clz(m);
    int w1 = w >> 5;
    m = b1[w1] & ((1u << (w & 31)) - 1u);
    if (!m) {
        const unsigned int mt = top & ((1u << w1) - 1u);
        if (!mt) return -1;
        w1 = 31 - __clz(mt);
        m = b1[w1];
    }
    w = (w1 << 5) + 31 - __clz(m);
    return (w << 5) + 31 - __clz(b0[w]);
}

// smallest covered column >= t, or -1
__device__ __forceinline__ int stereo_next(const unsigned int *b0, const unsigned int *b1, unsigned int top, int t)
{
    int w = t >> 5;
    unsigned int m = b0[w] & (0xFFFFFFFFu << (t & 31));
    if (m) return (w << 5) + __ffs(m) - 1;
    int w1 = w >> 5;
    m = b1[w1] & (0xFFFFFFFEu << (w & 31));
    if (!m) {
        const unsigned int mt = top & (0xFFFFFFFEu << w1);
        if (!mt) return -1;
        w1 = __ffs(mt) - 1;
        m = b1[w1];
    }
    w = (w1 << 5) + __ffs(m) - 1;
    return (w << 5) + __ffs(b0[w]) - 1;
}

// the source column whose pixel one view shows at target column t
__device__ __forceinline__ int stereo_source(const unsigned int *key, const unsigned short *win, const unsigned int *b0,
                                             const unsigned int *b1, unsigned int top, int t)
{
    if (key[t] != STEREO_EMPTY) return win[t];
    const int l = stereo_prev(b0, b1, top, t), r = stereo_next(b0, b1, top, t);
    if (r < 0) return l < 0 ? t : win[l];
    return (l >= 0 && key[l] >= key[r]) ? win[l] : win[r];
}

static size_t stereo_smem_bytes(int cols)
{
    return (size_t)12 * cols + (size_t)8 * ((cols + 31) / 32) + 128;
}

template <bool ALIGNED>
__global__ void __launch_bounds__(STEREO_THREADS)
stereo_kernel(const uint8_t *__restrict__ orig, size_t origPitch, const float *__restrict__ depth, size_t depthPitch,
              uint8_t *__restrict__ left, size_t leftPitch, uint8_t *__restrict__ right, size_t rightPitch,
              uint8_t *__restrict__ anaglyph, size_t anaglyphPitch, int cols, float conv, const float *__restrict__ convAt, int maxDisparity)
{
    extern __shared__ __align__(16) unsigned char stereo_smem[];
    const int W = (cols + 31) >> 5, W1 = (W + 31) >> 5;            // W1 <= 16 for cols <= 16384
    unsigned int *key = (unsigned int *)stereo_smem;                // [2][cols] view 0 = left, 1 = right
    unsigned int *b0 = key + 2 * cols;                              // [2][W]
    unsigned int *b1 = b0 + 2 * W;                                  // [2][16]
    unsigned short *win = (unsigned short *)(b1 + 32);              // [2][cols]
    const int y = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const bool needL = left || anaglyph, needR = right || anaglyph;
    // "click to converge": the depth under the chosen pixel, read here so that no host round trip sits between solve and stereo
    if (convAt) conv = stereo_depth(__ldg(convAt));
    const float D = (float)maxDisparity;
    const uint8_t *src = orig + (size_t)y * origPitch;
    const float *dRow = (const float *)((const char *)depth + (size_t)y * depthPitch);

    for (int t = tid; t < 2 * cols; t += STEREO_THREADS) key[t] = STEREO_EMPTY;
    __syncthreads();
    for (int x = tid; x < cols; x += STEREO_THREADS) {
        const float dc = stereo_depth(__ldg(dRow + x));
        const int s = stereo_parallax(dc, conv, D), hL = s / 2;
        const int tL = x - hL, tR = x + (s - hL);
        if (needL && (unsigned)tL < (unsigned)cols) atomicMin(key + tL, __float_as_uint(dc));
        if (needR && (unsigned)tR < (unsigned)cols) atomicMin(key + cols + tR, __float_as_uint(dc));
    }
    __syncthreads();
    for (int x = tid; x < cols; x += STEREO_THREADS) {             // the row's depth is in L1 now
        const float dc = stereo_depth(__ldg(dRow + x));
        const int s = stereo_parallax(dc, conv, D), hL = s / 2;
        const int tL = x - hL, tR = x + (s - hL);
        if (needL && (unsigned)tL < (unsigned)cols && key[tL] == __float_as_uint(dc)) win[tL] = (unsigned short)x;
        if (needR && (unsigned)tR < (unsigned)cols && key[cols + tR] == __float_as_uint(dc)) win[cols + tR] = (unsigned short)x;
    }
    for (int t = tid; t < 32 * W; t += STEREO_THREADS) {            // whole warps: both bounds are multiples of 32
        const unsigned int mL = __ballot_sync(0xFFFFFFFFu, t < cols && key[t] != STEREO_EMPTY);
        const unsigned int mR = __ballot_sync(0xFFFFFFFFu, t < cols && key[cols + t] != STEREO_EMPTY);
        if (lane == 0) { b0[t >> 5] = mL; b0[W + (t >> 5)] = mR; }
    }
    __syncthreads();
    for (int w = tid; w < 32 * W1; w += STEREO_THREADS) {
        const unsigned int mL = __ballot_sync(0xFFFFFFFFu, w < W && b0[w] != 0u);
        const unsigned int mR = __ballot_sync(0xFFFFFFFFu, w < W && b0[W + w] != 0u);
        if (lane == 0) { b1[w >> 5] = mL; b1[16 + (w >> 5)] = mR; }
    }
    __syncthreads();
    const unsigned int topL = __ballot_sync(0xFFFFFFFFu, lane < W1 && b1[lane] != 0u);
    const unsigned int topR = __ballot_sync(0xFFFFFFFFu, lane < W1 && b1[16 + lane] != 0u);

    for (int x4 = 4 * tid; x4 < cols; x4 += 4 * STEREO_THREADS) {
        const int n = min(4, cols - x4);
        unsigned int cl[4][3], cr[4][3];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            cl[i][0] = cl[i][1] = cl[i][2] = cr[i][0] = cr[i][1] = cr[i][2] = 0u;
            if (i < n) {
                if (needL) {
                    const uint8_t *p = src + 3 * stereo_source(key, win, b0, b1, topL, x4 + i);
                    cl[i][0] = __ldg(p); cl[i][1] = __ldg(p + 1); cl[i][2] = __ldg(p + 2);
                }
                if (needR) {
                    const uint8_t *p = src + 3 * stereo_source(key + cols, win + cols, b0 + W, b1 + 16, topR, x4 + i);
                    cr[i][0] = __ldg(p); cr[i][1] = __ldg(p + 1); cr[i][2] = __ldg(p + 2);
                }
            }
        }
        if (left) store_bgr4<ALIGNED>(left + (size_t)y * leftPitch + 3 * x4, n, cl);
        if (right) store_bgr4<ALIGNED>(right + (size_t)y * rightPitch + 3 * x4, n, cr);
        if (anaglyph) {
#pragma unroll
            for (int i = 0; i < 4; i++) cr[i][2] = cl[i][2];            // B, G of the right view, R of the left one
            store_bgr4<ALIGNED>(anaglyph + (size_t)y * anaglyphPitch + 3 * x4, n, cr);
        }
    }
}

cudaError_t configure_stereo()
{
    const int bytes = (int)stereo_smem_bytes(RTDD_STEREO_MAX_COLS);
    cudaError_t e = cudaFuncSetAttribute(stereo_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(stereo_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    return e;
}

cudaError_t launch_stereo(cudaStream_t s, const uint8_t *orig, size_t origPitch, const float *depth, size_t depthPitch,
                          uint8_t *left, size_t leftPitch, uint8_t *right, size_t rightPitch, uint8_t *anaglyph, size_t anaglyphPitch,
                          int rows, int cols, float conv, const float *convAt, int maxDisparity)
{
    const bool al = (!left || aligned4(left, leftPitch)) && (!right || aligned4(right, rightPitch)) &&
                    (!anaglyph || aligned4(anaglyph, anaglyphPitch));
    const size_t smem = stereo_smem_bytes(cols);
    if (al)
        stereo_kernel<true><<<rows, STEREO_THREADS, smem, s>>>(orig, origPitch, depth, depthPitch, left, leftPitch, right, rightPitch,
                                                               anaglyph, anaglyphPitch, cols, conv, convAt, maxDisparity);
    else
        stereo_kernel<false><<<rows, STEREO_THREADS, smem, s>>>(orig, origPitch, depth, depthPitch, left, leftPitch, right, rightPitch,
                                                                anaglyph, anaglyphPitch, cols, conv, convAt, maxDisparity);
    return cudaGetLastError();
}

}  // namespace rtdd
