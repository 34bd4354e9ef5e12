// ball_query_grid.cu -- multi-scale ball query through a per-scene uniform xy grid (large n, small radius).
//
// Same results as ball_query.cu / the reference kernel (src/ball_query_gpu.cu:9-45): the first `nsample`
// point indices IN ORIGINAL INDEX ORDER with d2 < radius^2, first-hit padding, zero rows when empty.  The
// brute-force scan tests all n points per centre (143.9 M pair tests per KITTI scene); here
//   1. one CTA per (scene, window of BG_WIN consecutive point ids) bins that window's points into square cells
//      of edge c >= 1.01 * r_max (counting sort in shared memory) and writes them cell-major as float4
//      (x, y, z, original index); every window uses the same scene-wide cell geometry;
//   2. one warp per centre tests only the 3 x 3 cell neighbourhood (three contiguous runs of the cell-major
//      array), marks every hit in a per-warp BITMAP indexed by original point index (shared memory), and
//      reads the bitmap back in index order -- which is exactly the reference's "first nsample in index
//      order" without any sorting.  The bitmap covers a window of bq_win(NS) ids (65536, 32768 with four
//      scales, so that eight warps' bitmaps fit shared memory); larger scenes are walked window by window in
//      increasing id order, carrying the hit count and the first hit, until every scale is full.
// Rigour: the cell index is a monotone function of the coordinate and c carries a 1 % margin, so every point
// whose fp32 d2 passes the strict `d2 < r^2` test lies in the 3 x 3 neighbourhood; the d2 expression and
// the compare are the reference's (common.cuh::sqdist3).
#include <stdlib.h>

#include "common.cuh"

namespace spsk {

constexpr int BG_MAXC = 11264;        // max cells per scene (44 KB of counters)
constexpr int BG_GMAX = 106;          // max cells per axis (106 * 106 <= BG_MAXC)
constexpr int BG_WARPS = 8;
constexpr int BG_WIN = 65536;        // point ids per build window (one counting sort, one cell_start array)
constexpr int BG_PREFIX_MIN = 1024;  // neighbourhoods with at least this many candidates start with an index-order prefix scan

struct GridParams {   // per scene, written by the build kernel
    float minx, miny, minz, inv_c, inv_cz;
    int gx, gy, gz;       // gz = 1 for LiDAR-shaped scenes (the xy grid uses the whole cell budget); > 1 splits the columns
};                        // into z slabs when the xy extent is small (feature-space queries of SPSNet's DenseEdgeConv)

// ids per query bitmap window: eight warps' bitmaps of NS * bq_win / 32 words stay within 200 KB of shared memory
__host__ __device__ constexpr int bq_win(int ns) { return ns <= 3 ? BG_WIN : BG_WIN / 2; }
static_assert(BG_WARPS * 3 * (bq_win(3) / 32) * 4 <= 200 * 1024 && BG_WARPS * 4 * (bq_win(4) / 32) * 4 <= 200 * 1024,
              "query bitmaps exceed the shared-memory budget");

static int build_windows(int n) { return max(1, (n + BG_WIN - 1) / BG_WIN); }

// workspace layout (bytes, 16-aligned): [GridParams b][sorted b*n float4][cell_start b*windows*(BG_MAXC+1) int]
static size_t grid_ws_bytes(int b, int n) {
    return sizeof(GridParams) * (size_t)b + sizeof(int) * (size_t)b * build_windows(n) * (BG_MAXC + 1) +
           sizeof(float4) * (size_t)b * n + 256;
}

__device__ __forceinline__ int cell_coord(float v, float vmin, float inv_c, int g) {
    const int c = (int)floorf((v - vmin) * inv_c);
    return min(max(c, 0), g - 1);
}

__global__ void __launch_bounds__(1024, 1)
bq_grid_build_kernel(int n, float rmax, const float *__restrict__ xyz, GridParams *__restrict__ params,
                     int *__restrict__ cell_start, float4 *__restrict__ sorted) {
    __shared__ int cnt[BG_MAXC];
    __shared__ float red[6][32];
    __shared__ int wsum[32];
    // every window's CTA reduces the whole scene's box (exact min / max: the same GridParams in every CTA)
    const int win = blockIdx.x, b = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float *pts = xyz + (size_t)b * n * 3;
    const int w0 = win * BG_WIN, nw = min(BG_WIN, n - w0);   // this CTA's ids [w0, w0 + nw)
    float x0 = 3.0e38f, x1 = -3.0e38f, y0 = 3.0e38f, y1 = -3.0e38f, z0 = 3.0e38f, z1 = -3.0e38f;
    for (int i = tid; i < n; i += 1024) {
        const float x = __ldg(pts + (size_t)i * 3), y = __ldg(pts + (size_t)i * 3 + 1), z = __ldg(pts + (size_t)i * 3 + 2);
        x0 = fminf(x0, x); x1 = fmaxf(x1, x); y0 = fminf(y0, y); y1 = fmaxf(y1, y); z0 = fminf(z0, z); z1 = fmaxf(z1, z);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        x0 = fminf(x0, __shfl_xor_sync(0xFFFFFFFFu, x0, o)); x1 = fmaxf(x1, __shfl_xor_sync(0xFFFFFFFFu, x1, o));
        y0 = fminf(y0, __shfl_xor_sync(0xFFFFFFFFu, y0, o)); y1 = fmaxf(y1, __shfl_xor_sync(0xFFFFFFFFu, y1, o));
        z0 = fminf(z0, __shfl_xor_sync(0xFFFFFFFFu, z0, o)); z1 = fmaxf(z1, __shfl_xor_sync(0xFFFFFFFFu, z1, o));
    }
    if (lane == 0) { red[0][warp] = x0; red[1][warp] = x1; red[2][warp] = y0; red[3][warp] = y1; red[4][warp] = z0; red[5][warp] = z1; }
    for (int i = tid; i < BG_MAXC; i += 1024) cnt[i] = 0;
    __syncthreads();
    x0 = red[0][0]; x1 = red[1][0]; y0 = red[2][0]; y1 = red[3][0]; z0 = red[4][0]; z1 = red[5][0];
    for (int w = 1; w < 32; ++w) {
        x0 = fminf(x0, red[0][w]); x1 = fmaxf(x1, red[1][w]); y0 = fminf(y0, red[2][w]); y1 = fmaxf(y1, red[3][w]);
        z0 = fminf(z0, red[4][w]); z1 = fmaxf(z1, red[5][w]);
    }
    const float ex = fmaxf(x1 - x0, 0.f), ey = fmaxf(y1 - y0, 0.f), ez = fmaxf(z1 - z0, 0.f);
    float c = fmaxf(rmax * 1.01f, 1e-6f);
    c = fmaxf(c, fmaxf(ex, ey) / (float)(BG_GMAX - 2));       // never more than BG_GMAX cells per axis
    const float inv_c = 1.0f / c;
    const int gx = min(BG_GMAX, (int)floorf(ex * inv_c) + 1), gy = min(BG_GMAX, (int)floorf(ey * inv_c) + 1);
    // z slabs with whatever cell budget the xy grid leaves (none for LiDAR scenes: 70 x 80 m at 0.8 m cells); slab height
    // >= the xy edge, stretched when the budget caps the count -- the cell index stays a monotone function of z with an
    // edge >= 1.01 r, so the 3 x 3 x 3 neighbourhood argument holds unchanged
    // ... and only when the scene is at least 4 slabs tall: splitting a LiDAR scene of 2-3 slabs (KITTI layer 1: 4 m at
    // 1.6 m cells) triples the number of cell rows a query walks for no fewer candidates (measured: +17 % on that query)
    const int gz_budget = max(1, BG_MAXC / (gx * gy));
    const int gz_wanted = (int)floorf(ez * inv_c) + 1;
    const int gz = gz_wanted >= 4 ? max(1, min(min(gz_budget, BG_GMAX), gz_wanted)) : 1;
    const float cz = fmaxf(c, ez / (float)max(gz - 1, 1) * (gz > 1 ? 1.0f : 0.0f));
    const float inv_cz = gz > 1 ? 1.0f / fmaxf(cz, c) : 0.0f;
    const int ncell = gx * gy * gz;
    if (tid == 0 && win == 0) {
        GridParams p;
        p.minx = x0; p.miny = y0; p.minz = z0; p.inv_c = inv_c; p.inv_cz = inv_cz; p.gx = gx; p.gy = gy; p.gz = gz;
        params[b] = p;
    }
    // histogram
    for (int i = w0 + tid; i < w0 + nw; i += 1024) {
        const int cx = cell_coord(__ldg(pts + (size_t)i * 3), x0, inv_c, gx);
        const int cy = cell_coord(__ldg(pts + (size_t)i * 3 + 1), y0, inv_c, gy);
        const int cz_i = gz > 1 ? cell_coord(__ldg(pts + (size_t)i * 3 + 2), z0, inv_cz, gz) : 0;
        atomicAdd(&cnt[(cz_i * gy + cy) * gx + cx], 1);
    }
    __syncthreads();
    // exclusive scan of cnt[0..ncell) -> cell_start ; cnt becomes the running cursor
    const int per = (ncell + 1023) / 1024;
    const int beg = tid * per, end = min(beg + per, ncell);
    int local = 0;
    for (int i = beg; i < end; ++i) local += cnt[i];
    int incl = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int v = wsum[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int u = __shfl_up_sync(0xFFFFFFFFu, v, o);
            if (lane >= o) v += u;
        }
        wsum[lane] = v;   // inclusive over warps
    }
    __syncthreads();
    int run = incl - local + (warp ? wsum[warp - 1] : 0);
    int *cs = cell_start + ((size_t)b * gridDim.x + win) * (BG_MAXC + 1);
    for (int i = beg; i < end; ++i) {
        const int c0 = cnt[i];
        cs[i] = run;
        cnt[i] = run;
        run += c0;
    }
    if (tid == 0) cs[ncell] = nw;
    __syncthreads();
    // scatter (order inside a cell is irrelevant: the query orders hits through its bitmap)
    float4 *out = sorted + (size_t)b * n + w0;
    for (int i = w0 + tid; i < w0 + nw; i += 1024) {
        const float x = __ldg(pts + (size_t)i * 3), y = __ldg(pts + (size_t)i * 3 + 1), z = __ldg(pts + (size_t)i * 3 + 2);
        const int cx = cell_coord(x, x0, inv_c, gx), cy = cell_coord(y, y0, inv_c, gy);
        const int cz_i = gz > 1 ? cell_coord(z, z0, inv_cz, gz) : 0;
        const int pos = atomicAdd(&cnt[(cz_i * gy + cy) * gx + cx], 1);
        out[pos] = make_float4(x, y, z, __int_as_float(i));
    }
}

struct BgScales {
    float r2[SPSK_MAX_SCALES];
    int nsample[SPSK_MAX_SCALES];
    int *idx[SPSK_MAX_SCALES];
};

// ONE: n <= bq_win(NS), a single window (one build window, bitmap of ceil(n / 32) words); else bq_win(NS) / 32 words
template <int NS, bool ONE>
__global__ void __launch_bounds__(BG_WARPS * 32)
bq_grid_query_kernel(int n, int m, int words, BgScales sc, const float *__restrict__ new_xyz,
                     const float *__restrict__ xyz, const GridParams *__restrict__ params,
                     const int *__restrict__ cell_start, const float4 *__restrict__ sorted, int prefix_min, int prefix_mul4) {
    extern __shared__ uint32_t bitmaps[];   // [BG_WARPS][NS][words]
    const int b = blockIdx.y;
    const int warp = threadIdx.x >> 5;
    const uint32_t lane = lane_id();
    uint32_t *bm = bitmaps + (size_t)warp * NS * words;
    // The bitmaps are zeroed ONCE per warp; afterwards every centre clears exactly the rows it touched while reading
    // them back, so the per-centre cost follows the number of hits, not n / 32.
    for (int i = lane; i < NS * words; i += 32) bm[i] = 0u;
    __syncwarp();
    const GridParams gp = params[b];
    constexpr int W = bq_win(NS);
    const int nwin = ONE ? 1 : (n + W - 1) / W;               // bitmap windows
    const int nbuild = ONE ? 1 : (n + BG_WIN - 1) / BG_WIN;   // build windows (cell_start arrays)
    const int *cs = cell_start + (size_t)b * nbuild * (BG_MAXC + 1);
    const float4 *pts = sorted + (size_t)b * n;
    const float *raw = xyz + (size_t)b * n * 3;
    for (int p = blockIdx.x * BG_WARPS + warp; p < m; p += gridDim.x * BG_WARPS) {
        const float *c = new_xyz + ((size_t)b * m + p) * 3;
        const float qx = __ldg(c), qy = __ldg(c + 1), qz = __ldg(c + 2);
        int pcnt[NS], pfirst[NS];
#pragma unroll
        for (int s = 0; s < NS; ++s) { pcnt[s] = 0; pfirst[s] = -1; }
        bool alldone = false;
        // the centre may lie outside the scene box (vote centres): unclamped cell coordinate, clamped ranges
        const int ccx = (int)floorf((qx - gp.minx) * gp.inv_c), ccy = (int)floorf((qy - gp.miny) * gp.inv_c);
        const int xlo = max(ccx - 1, 0), xhi = min(ccx + 1, gp.gx - 1);
        const int ylo = max(ccy - 1, 0), yhi = min(ccy + 1, gp.gy - 1);
        const int ccz = gp.gz > 1 ? (int)floorf((qz - gp.minz) * gp.inv_cz) : 0;
        const int zlo = gp.gz > 1 ? max(ccz - 1, 0) : 0, zhi = gp.gz > 1 ? min(ccz + 1, gp.gz - 1) : 0;
        const int ny = yhi - ylo + 1, nrows = ny > 0 && zhi >= zlo ? ny * (zhi - zlo + 1) : 0;   // <= 9 (y, z) rows of cells
        // Candidates the grid phase would have to test for this centre.  In a dense neighbourhood (SPSNet's DenseEdgeConv
        // queries 24-wide FEATURES, thousands of them inside one radius) the reference's index-order scan stops after a few
        // hundred points while the grid would test them all: scan the first `tn` points in index order first.  tn = the
        // candidate count itself, so the detour costs at most as much again as the grid phase it may save (and nothing for
        // the LiDAR-shaped neighbourhoods of the SA layers, which stay below BG_PREFIX_MIN).
        int cand = 0;
        if (xlo <= xhi && (int)lane < nrows) {
            const int dz = ((int)lane >= ny) + ((int)lane >= 2 * ny), dy = (int)lane - dz * ny;   // ny <= 3: no division
            const int row = ((zlo + dz) * gp.gy + ylo + dy) * gp.gx;
            for (int bw = 0; bw < nbuild; ++bw) {
                const int *cw = cs + (size_t)bw * (BG_MAXC + 1);
                cand += __ldg(cw + row + xhi + 1) - __ldg(cw + row + xlo);
            }
        }
        cand = __reduce_add_sync(0xFFFFFFFFu, cand);
        const int tn = cand >= prefix_min ? min(n, (((cand >> 2) * prefix_mul4) + 31) & ~31) : 0;
        // Prefix phase: exactly the reference's scan order, 32 points per step, hits appended in index order through a
        // ballot; stops as soon as every scale has its nsample indices (the reference's break).
        for (int k0 = 0; k0 < tn && !alldone; k0 += 32) {
            const int k = k0 + (int)lane;
            float d2 = 3.0e38f;
            if (k < tn) d2 = sqdist3(qx, qy, qz, __ldg(raw + (size_t)k * 3), __ldg(raw + (size_t)k * 3 + 1), __ldg(raw + (size_t)k * 3 + 2));
            alldone = true;
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                const int ns = sc.nsample[s];
                if (pcnt[s] < ns) {
                    const bool hit = d2 < sc.r2[s];
                    const uint32_t hm = __ballot_sync(0xFFFFFFFFu, hit);
                    if (hm) {
                        if (pfirst[s] < 0) pfirst[s] = k0 + __ffs(hm) - 1;
                        const int pos = pcnt[s] + __popc(hm & ((1u << lane) - 1u));
                        if (hit && pos < ns) sc.idx[s][((size_t)b * m + p) * ns + pos] = k;
                        pcnt[s] += __popc(hm);
                    }
                }
                alldone = alldone && pcnt[s] >= ns;
            }
        }
        // Grid phase, one bitmap window of ids [lo, lo + W) at a time; windows whose ids all lie below tn were covered by
        // the prefix phase.  pcnt / pfirst carry the hits written so far and the smallest hit across windows.
        for (int win = 0; win < nwin && !alldone; ++win) {
            const int lo = ONE ? 0 : win * W;
            const int *cw = cs + (size_t)(lo / BG_WIN) * (BG_MAXC + 1);   // the build window holding [lo, lo + W)
            const float4 *pw = pts + (lo / BG_WIN) * BG_WIN;
            // rows (32 words = 1024 ids of the window) that received a hit, per scale: 64 rows cover W <= 65536
            uint32_t tlo[NS], thi[NS];
#pragma unroll
            for (int s = 0; s < NS; ++s) { tlo[s] = 0u; thi[s] = 0u; }
            if (xlo <= xhi && tn < min(n, lo + W)) {
                for (int rw = 0, cy = ylo, cz = zlo; rw < nrows; ++rw) {
                    const int row = (cz * gp.gy + cy) * gp.gx;
                    if (++cy > yhi) { cy = ylo; ++cz; }
                    const int beg = __ldg(cw + row + xlo), end = __ldg(cw + row + xhi + 1);
                    for (int k0 = beg; k0 < end; k0 += 32) {
                        const int k = k0 + (int)lane;
                        float d2 = 3.0e38f;
                        uint32_t oi = 0u;
                        if (k < end) {
                            const float4 v = __ldg(pw + k);
                            d2 = sqdist3(qx, qy, qz, v.x, v.y, v.z);
                            oi = (uint32_t)__float_as_int(v.w);
                        }
                        const uint32_t li = oi - (uint32_t)lo;   // index inside the bitmap window
                        const bool inwin = ONE || li < (uint32_t)W;   // a build window holds two bitmap windows with 4 scales
                        const uint32_t row = li >> 10;
#pragma unroll
                        for (int s = 0; s < NS; ++s) {
                            // (points below tn were already handled, in order, by the prefix phase)
                            const bool hit = d2 < sc.r2[s] && inwin && (int)oi >= tn && pcnt[s] < sc.nsample[s];
                            if (hit) atomicOr(&bm[s * words + (li >> 5)], 1u << (li & 31u));
                            tlo[s] |= (hit && row < 32u) ? (1u << row) : 0u;
                            thi[s] |= (hit && row >= 32u) ? (1u << (row - 32u)) : 0u;
                        }
                    }
                }
            }
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                tlo[s] = __reduce_or_sync(0xFFFFFFFFu, tlo[s]);
                thi[s] = __reduce_or_sync(0xFFFFFFFFu, thi[s]);
            }
            __syncwarp();
            // Read the touched rows back in index order (lane = word: conflict-free shared memory reads), clearing them on
            // the way; all rows are cleared even after nsample indices are out.
            alldone = true;
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                const int ns = sc.nsample[s];
                int *out = sc.idx[s] + ((size_t)b * m + p) * ns;
                uint32_t *w = bm + s * words;
                int base = pcnt[s];      // hits written so far (warp-uniform)
                int first = pfirst[s];   // smallest hit index (warp-uniform once found)
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    uint32_t rows = half ? thi[s] : tlo[s];
                    while (rows) {
                        const int i = (__ffs(rows) - 1) + 32 * half;
                        rows &= rows - 1u;
                        const int wi = i * 32 + (int)lane;
                        uint32_t bits = 0u;
                        if (wi < words) { bits = w[wi]; w[wi] = 0u; }
                        if (base >= ns) continue;   // row only needed clearing
                        const uint32_t nz = __ballot_sync(0xFFFFFFFFu, bits != 0u);
                        if (nz == 0u) continue;
                        const int cnt = __popc(bits);
                        int incl = cnt;
#pragma unroll
                        for (int o = 1; o < 32; o <<= 1) {
                            const int v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                            if ((int)lane >= o) incl += v;
                        }
                        if (first < 0) {
                            const int l0 = __ffs(nz) - 1;
                            const uint32_t b0 = __shfl_sync(0xFFFFFFFFu, bits, l0);
                            first = lo + (i * 32 + l0) * 32 + (__ffs(b0) - 1);
                        }
                        int pos = base + incl - cnt;
                        while (bits && pos < ns) {
                            const int bit = __ffs(bits) - 1;
                            bits &= bits - 1u;
                            out[pos++] = lo + wi * 32 + bit;
                        }
                        base += __shfl_sync(0xFFFFFFFFu, incl, 31);
                    }
                }
                pcnt[s] = base;
                pfirst[s] = first;
                alldone = alldone && base >= ns;
            }
        }
#pragma unroll
        for (int s = 0; s < NS; ++s) {
            const int ns = sc.nsample[s];
            int *out = sc.idx[s] + ((size_t)b * m + p) * ns;
            if (pcnt[s] > 0) {
                for (int l = min(pcnt[s], ns) + (int)lane; l < ns; l += 32) out[l] = pfirst[s];   // first-hit padding
            } else {
                for (int l = (int)lane; l < ns; l += 32) out[l] = 0;
            }
        }
        __syncwarp();
    }
}

}  // namespace spsk

extern "C" long long spsk_ball_query_grid_workspace_bytes(int b, int n) {
    if (b < 0 || n < 0) return -1;
    return (long long)spsk::grid_ws_bytes(b, n);
}

extern "C" int spsk_ball_query_msg_grid(int b, int n, int m, int nscales, const float *radius, const int *nsample,
                                        const float *new_xyz, const float *xyz, int *const *idx, void *workspace,
                                        long long workspace_bytes, spsk_stream_t stream) {
    using namespace spsk;
    SPSK_REQUIRE(b >= 0 && n >= 1 && m >= 0 && b <= 65535, SPSK_ERR_INVALID_ARG, "ball_query_msg_grid: bad sizes b=%d n=%d m=%d", b, n, m);
    SPSK_REQUIRE(n <= SPSK_BQ_GRID_MAX_N, SPSK_ERR_UNSUPPORTED, "ball_query_msg_grid: n=%d > %d", n, SPSK_BQ_GRID_MAX_N);
    SPSK_REQUIRE(nscales >= 1 && nscales <= SPSK_MAX_SCALES && radius && nsample && idx && new_xyz && xyz, SPSK_ERR_INVALID_ARG,
                 "ball_query_msg_grid: nscales=%d / null pointer", nscales);
    if (b == 0 || m == 0) return SPSK_OK;
    SPSK_REQUIRE(workspace && workspace_bytes >= (long long)grid_ws_bytes(b, n), SPSK_ERR_WORKSPACE,
                 "ball_query_msg_grid: workspace %lld B < %lld B", workspace_bytes, (long long)grid_ws_bytes(b, n));
    BgScales sc{};
    float rmax = 0.f;
    for (int s = 0; s < nscales; ++s) {
        SPSK_REQUIRE(nsample[s] >= 1 && idx[s], SPSK_ERR_INVALID_ARG, "ball_query_msg_grid: scale %d nsample=%d / null idx", s, nsample[s]);
        sc.r2[s] = radius[s] * radius[s];
        sc.nsample[s] = nsample[s];
        sc.idx[s] = idx[s];
        rmax = fmaxf(rmax, fabsf(radius[s]));
    }
    const int nbuild = build_windows(n);
    uint8_t *ws = reinterpret_cast<uint8_t *>(workspace);
    ws = reinterpret_cast<uint8_t *>(((uintptr_t)ws + 15) & ~(uintptr_t)15);
    GridParams *params = reinterpret_cast<GridParams *>(ws);
    float4 *sorted = reinterpret_cast<float4 *>(ws + ((sizeof(GridParams) * (size_t)b + 15) & ~(size_t)15));
    int *cell_start = reinterpret_cast<int *>(reinterpret_cast<uint8_t *>(sorted) + sizeof(float4) * (size_t)b * n);
    cudaStream_t st = as_stream(stream);
    bq_grid_build_kernel<<<dim3(nbuild, b), 1024, 0, st>>>(n, rmax, xyz, params, cell_start, sorted);
    SPSK_LAUNCH_CHECK("bq_grid_build_kernel");
    // prefix-scan policy (see the kernel): start at BG_PREFIX_MIN candidates, scan `cand` points.  SPSK_BQ_PREFIX_MIN /
    // SPSK_BQ_PREFIX_MUL4 (length = cand * MUL4 / 4) are tuning knobs for A/B measurements.
    static const int prefix_min = [] { const char *e = getenv("SPSK_BQ_PREFIX_MIN"); return e ? max(32, atoi(e)) : BG_PREFIX_MIN; }();
    static const int prefix_mul4 = [] { const char *e = getenv("SPSK_BQ_PREFIX_MUL4"); return e ? max(1, atoi(e)) : 4; }();
    const int win = bq_win(nscales);
    const bool one = n <= win;
    const int words = one ? (n + 31) / 32 : win / 32;
    const size_t smem = sizeof(uint32_t) * (size_t)BG_WARPS * nscales * words;   // <= 192 KB (static_assert above)
    // each warp walks several centres (the bitmap is zeroed once per warp): ~4 waves of CTAs over the GPU
    const int want = (m + BG_WARPS - 1) / BG_WARPS;
    const int per_scene = max(1, min(want, (SPSK_NUM_SMS * 6 * 4 + b - 1) / b));
    dim3 grid(per_scene, b);
#define SPSK_BG_LAUNCH(NSV, ONEV)                                                                                    \
    do {                                                                                                             \
        if (smem > 48 * 1024) {                                                                                      \
            cudaError_t e = cudaFuncSetAttribute(bq_grid_query_kernel<NSV, ONEV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
            if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(bq_grid_query_kernel)");              \
        }                                                                                                            \
        bq_grid_query_kernel<NSV, ONEV><<<grid, BG_WARPS * 32, smem, st>>>(n, m, words, sc, new_xyz, xyz, params, cell_start, sorted, prefix_min, prefix_mul4); \
    } while (0)
#define SPSK_BG_LAUNCH_NS(NSV)                                  \
    do {                                                        \
        if (one) SPSK_BG_LAUNCH(NSV, true); else SPSK_BG_LAUNCH(NSV, false); \
    } while (0)
    switch (nscales) {
        case 1: SPSK_BG_LAUNCH_NS(1); break;
        case 2: SPSK_BG_LAUNCH_NS(2); break;
        case 3: SPSK_BG_LAUNCH_NS(3); break;
        default: SPSK_BG_LAUNCH_NS(4); break;
    }
#undef SPSK_BG_LAUNCH_NS
#undef SPSK_BG_LAUNCH
    SPSK_LAUNCH_CHECK("bq_grid_query_kernel");
    return SPSK_OK;
}
