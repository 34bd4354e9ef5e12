// interpolate.cu -- three_nn / three_interpolate (+ backward) for PointnetFPModule.
//
// Replaces three_nn_kernel_fast, three_interpolate_kernel_fast, three_interpolate_grad_kernel_fast
// (src/interpolate_gpu.cu:16-59, 84-104, 127-149).  three_nn: one thread per unknown point, the known
// points staged through shared memory tiles (the reference re-reads them from global per thread);
// the reference's `float d < double best` compares with bests initialised to 1e40 are equivalent to
// float compares against +inf (a float is either < every double above FLT_MAX or compared exactly),
// and (float)1e40 == +inf, so the never-updated outputs match too.  three_nn_cluster_kernel gives the same outputs from a
// per-cluster xy grid of the known points (large scenes: the all-pairs scan grows as n * m).
#include "common.cuh"
#include <math_constants.h>

namespace spsk {

constexpr int NN_THREADS = 256;
constexpr int NN_TILE = 1024;

__global__ void __launch_bounds__(NN_THREADS)
three_nn_kernel(int n, int m, const float *__restrict__ unknown, const float *__restrict__ known,
                float *__restrict__ dist2, int *__restrict__ idx) {
    __shared__ float sx[NN_TILE], sy[NN_TILE], sz[NN_TILE];
    const int b = blockIdx.y;
    const int p = blockIdx.x * NN_THREADS + threadIdx.x;
    const bool active = p < n;
    float ux = 0.f, uy = 0.f, uz = 0.f;
    if (active) {
        const float *u = unknown + ((size_t)b * n + p) * 3;
        ux = __ldg(u); uy = __ldg(u + 1); uz = __ldg(u + 2);
    }
    const float *kn = known + (size_t)b * m * 3;
    float best1 = CUDART_INF_F, best2 = CUDART_INF_F, best3 = CUDART_INF_F;
    int i1 = 0, i2 = 0, i3 = 0;
    for (int t0 = 0; t0 < m; t0 += NN_TILE) {
        const int tn = min(NN_TILE, m - t0);
        __syncthreads();
        for (int i = threadIdx.x; i < tn * 3; i += NN_THREADS) {
            const float v = __ldg(kn + (size_t)t0 * 3 + i);
            const int k = i / 3, c = i - 3 * k;
            (c == 0 ? sx : (c == 1 ? sy : sz))[k] = v;
        }
        __syncthreads();
        if (active) {
            for (int kl = 0; kl < tn; ++kl) {
                const float d = sqdist3(ux, uy, uz, sx[kl], sy[kl], sz[kl]);
                const int k = t0 + kl;
                if (d < best1) {
                    best3 = best2; i3 = i2;
                    best2 = best1; i2 = i1;
                    best1 = d; i1 = k;
                } else if (d < best2) {
                    best3 = best2; i3 = i2;
                    best2 = d; i2 = k;
                } else if (d < best3) {
                    best3 = d; i3 = k;
                }
            }
        }
    }
    if (!active) return;
    float *od = dist2 + ((size_t)b * n + p) * 3;
    int *oi = idx + ((size_t)b * n + p) * 3;
    od[0] = best1; od[1] = best2; od[2] = best3;
    oi[0] = i1; oi[1] = i2; oi[2] = i3;
}

// ---- three_nn on large scenes: the known points of a scene in the shared memory of one cluster ---------------------------
// Which three candidates the reference keeps: its strict-`<` cascade in index order inserts each d behind every equal one
// already held, so it keeps the three smallest (d, id) pairs in lexicographic order among those with d < +inf (NaN fails
// every compare), and +inf / id 0 in slots it never fills.  sqdist3 never returns -0, so for d >= +0 the float bits order
// like the values: the key (bits(d) << 32 | id) orders candidates exactly as (d, id), the key of +inf / id 0 is the empty
// slot and every candidate with d = +inf or NaN has a key >= it.  Keeping the three smallest keys, merged in any order,
// is therefore the brute-force kernel's result bit for bit.
//
// Layout: CTA r of a cluster of C CTAs holds the known ids [r * chunk, (r + 1) * chunk), chunk <= TN_CAP, counting-sorted
// into square xy cells (cell-major float4 (x, y, z, id) + cell starts in its own shared memory).  All CTAs derive the same
// cell geometry from the exact box of the scene's known points.  A warp answers one unknown point at a time: it tests the
// 3 x 3 cells around the point's cell, then ring after ring of cells further out, in every CTA's slice (DSMEM), until the
// lower bound on d of every point outside the visited square is strictly greater than the third-best d (or the square
// covers the grid).
constexpr int TN_THREADS = 1024;
constexpr int TN_WARPS = TN_THREADS / 32;
constexpr int TN_CAP = 8192;      // known points per CTA: 128 KB of float4
constexpr int TN_MAXC = 16384;    // max cells per scene (64 KB of cell starts per CTA)
constexpr int TN_GMAX = 128;      // max cells per axis (TN_GMAX * TN_GMAX <= TN_MAXC)
constexpr int TN_PPC = 2;         // known points per cell over the scene's box, before the caps
constexpr size_t TN_SMEM = sizeof(float4) * TN_CAP + sizeof(int) * (TN_MAXC + 1) + sizeof(float) * 4;
static_assert(TN_GMAX * TN_GMAX <= TN_MAXC, "cell budget");
static_assert(TN_CAP * 16 == SPSK_THREE_NN_GRID_MAX_M, "SPSK_THREE_NN_GRID_MAX_M is 16 CTAs of TN_CAP known points");
constexpr unsigned long long TN_EMPTY = 0x7F80000000000000ull;   // key of (+inf, id 0)

__device__ __forceinline__ int ld_cluster_s32(uint32_t a) {
    int v;
    asm volatile("ld.shared::cluster.s32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ float ld_cluster_f32(uint32_t a) {
    float v;
    asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ float4 ld_cluster_f4(uint32_t a) {
    float4 v;
    asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}

// In-place exclusive prefix sum of a[0, count) (shared memory) by the whole block (blockDim.x a multiple of 32); ends with
// a __syncthreads.  wsum: __shared__ int[32].
__device__ __forceinline__ void block_exclusive_scan(int *a, int count, int *wsum) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int per = (count + blockDim.x - 1) / blockDim.x;
    const int beg = tid * per, end = min(beg + per, count);
    int local = 0;
    for (int i = beg; i < end; ++i) local += a[i];
    int incl = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int v = lane < nwarps ? wsum[lane] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int u = __shfl_up_sync(0xFFFFFFFFu, v, o);
            if (lane >= o) v += u;
        }
        wsum[lane] = v;   // inclusive over warps
    }
    __syncthreads();
    int run = incl - local + (warp ? wsum[warp - 1] : 0);
    for (int i = beg; i < end; ++i) {
        const int c0 = a[i];
        a[i] = run;
        run += c0;
    }
    __syncthreads();
}

__device__ __forceinline__ void top3_insert(unsigned long long key, unsigned long long &k1, unsigned long long &k2,
                                            unsigned long long &k3) {
    if (key < k3) {
        if (key < k2) {
            k3 = k2;
            if (key < k1) { k2 = k1; k1 = key; } else { k2 = key; }
        } else {
            k3 = key;
        }
    }
}

// Lower bound on the fp32 d (sqdist3) of every known point outside the cells [cx - R, cx + R] x [cy - R, cy + R], for the
// query at cell coordinates (tx, ty) = ((qx - minx) * inv_c, (qy - miny) * inv_c), computed in fp32 like cell_coord.
// Why it holds: a point in a cell beyond the square on the right has s = (px - minx) * inv_c >= cx + R + 1 (cell_coord is
// floor(s), clamped; the clamp only lowers the top cell's index), so s - tx >= gap_right; on the left s < cx - R, so
// tx - s > gap_left; in y likewise.  Every point lies in the box, so |s - tx| >= bx, the distance from tx to [0, gx].  A
// point outside the square is beyond it in x (dx >= max(gap_x, bx), dy >= by) or in y (dx >= bx, dy >= max(gap_y, by)).
// The fp32 s and tx differ from their exact values by a few ulps of their magnitudes (<= gx + 1 and |tx|): the slack of
// 1e-4 * (gx + |tx| + 2) cells covers that with a wide margin.  Cell units become metres through c = 1 / inv_c, and sqdist3's
// three subtractions, three products and two sums round d down by less than 1e-6 relative: the factor 0.9995 on the
// linear gaps (0.999 on d), applied before squaring so that an overflow to +inf implies d = +inf too, covers both.  NaN
// gaps (non-finite query) compare false, so such a query never stops early.
__device__ __forceinline__ float tn_ring_bound(float tx, float ty, int cx, int cy, int R, int gx, int gy, float c_lin) {
    const float inf = CUDART_INF_F;
    const float gxm = fminf(cx - R > 0 ? tx - (float)(cx - R) : inf, cx + R < gx - 1 ? (float)(cx + R + 1) - tx : inf);
    const float gym = fminf(cy - R > 0 ? ty - (float)(cy - R) : inf, cy + R < gy - 1 ? (float)(cy + R + 1) - ty : inf);
    const float bx = fmaxf(fmaxf(-tx, tx - (float)gx), 0.f), by = fmaxf(fmaxf(-ty, ty - (float)gy), 0.f);
    const float sx = 1e-4f * ((float)gx + fabsf(tx) + 2.f), sy = 1e-4f * ((float)gy + fabsf(ty) + 2.f);
    const float ax = fmaxf(fmaxf(gxm, bx) - sx, 0.f) * c_lin, ay = fmaxf(fmaxf(gym, by) - sy, 0.f) * c_lin;
    const float lx = fmaxf(bx - sx, 0.f) * c_lin, ly = fmaxf(by - sy, 0.f) * c_lin;
    return fminf(ax * ax + ly * ly, lx * lx + ay * ay);
}

// grid: b * per_scene clusters of `csize` CTAs (csize = cluster size, a power of two <= 16); cluster `part` of scene b
// answers the unknown points [part * rows, (part + 1) * rows).
__global__ void __launch_bounds__(TN_THREADS, 1)
three_nn_cluster_kernel(int n, int m, int chunk, int per_scene, int rows, const float *__restrict__ unknown,
                        const float *__restrict__ known, float *__restrict__ dist2, int *__restrict__ idx) {
    extern __shared__ float4 tn_smem[];
    float4 *pts = tn_smem;                                // [TN_CAP] this CTA's known points, cell-major
    int *cs = reinterpret_cast<int *>(pts + TN_CAP);      // [ncell + 1]: cell k holds pts[cs[k], cs[k + 1])
    float *cbox = reinterpret_cast<float *>(cs + TN_MAXC + 1);   // this CTA's x0, x1, y0, y1
    __shared__ float red[6][32];
    __shared__ int wsum[32];
    const int tid = threadIdx.x, warp = tid >> 5;
    const uint32_t lane = lane_id();
    const uint32_t csize = cluster_nctarank(), rank = cluster_ctarank();
    const uint32_t lc = __ffs(csize) - 1;
    const int cl = blockIdx.x / csize, b = cl / per_scene, part = cl - b * per_scene;
    const float *kp = known + (size_t)b * m * 3;
    const int k0 = (int)rank * chunk, kn = max(0, min(chunk, m - k0));

    // 1. the scene's box: each CTA reduces its slice, then every warp combines all slices (the same order everywhere)
    float box[6];
    block_box3(kp, k0, k0 + kn, red, box);
    if (tid == 0) { cbox[0] = box[0]; cbox[1] = box[1]; cbox[2] = box[2]; cbox[3] = box[3]; }
    cluster_sync_all();
    const uint32_t cbox_sh = (uint32_t)__cvta_generic_to_shared(cbox);
    float x0 = 3.0e38f, x1 = -3.0e38f, y0 = 3.0e38f, y1 = -3.0e38f;
    if (lane < csize) {
        const uint32_t a = cluster_map_shared(cbox_sh, lane);
        x0 = ld_cluster_f32(a); x1 = ld_cluster_f32(a + 4); y0 = ld_cluster_f32(a + 8); y1 = ld_cluster_f32(a + 12);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        x0 = fminf(x0, __shfl_xor_sync(0xFFFFFFFFu, x0, o)); x1 = fmaxf(x1, __shfl_xor_sync(0xFFFFFFFFu, x1, o));
        y0 = fminf(y0, __shfl_xor_sync(0xFFFFFFFFu, y0, o)); y1 = fmaxf(y1, __shfl_xor_sync(0xFFFFFFFFu, y1, o));
    }
    // 2. cell geometry: square cells of ~TN_PPC points over the box, at most TN_GMAX per axis.  A box that is not finite
    // (an infinite coordinate, or no non-NaN one) makes the whole scene one cell: the search is then the full scan.
    const float ex = x1 - x0, ey = y1 - y0;
    float c = sqrtf(ex * ey / (float)max(1, min(TN_MAXC, m / TN_PPC)));
    c = fmaxf(c, fmaxf(ex, ey) / (float)(TN_GMAX - 2));
    int gx = 1, gy = 1;
    float inv_c = 0.f;
    if (isfinite(ex) && isfinite(ey) && ex >= 0.f && ey >= 0.f && c > 0.f && isfinite(1.0f / c)) {
        inv_c = 1.0f / c;
        gx = min(TN_GMAX, (int)floorf(ex * inv_c) + 1);
        gy = min(TN_GMAX, (int)floorf(ey * inv_c) + 1);
    } else {
        x0 = 0.f; y0 = 0.f;
    }
    const int ncell = gx * gy;
    // 3. counting sort of this CTA's slice: counts in cs[k + 1], exclusive scan, scatter with cs[k + 1] as the cursor
    for (int i = tid; i <= ncell; i += TN_THREADS) cs[i] = 0;
    __syncthreads();
    for (int i = tid; i < kn; i += TN_THREADS) {
        const float *p = kp + (size_t)(k0 + i) * 3;
        atomicAdd(&cs[1 + cell_coord(__ldg(p + 1), y0, inv_c, gy) * gx + cell_coord(__ldg(p), x0, inv_c, gx)], 1);
    }
    __syncthreads();
    block_exclusive_scan(cs + 1, ncell, wsum);
    for (int i = tid; i < kn; i += TN_THREADS) {
        const float *p = kp + (size_t)(k0 + i) * 3;
        const float x = __ldg(p), y = __ldg(p + 1), z = __ldg(p + 2);
        const int pos = atomicAdd(&cs[1 + cell_coord(y, y0, inv_c, gy) * gx + cell_coord(x, x0, inv_c, gx)], 1);
        pts[pos] = make_float4(x, y, z, __int_as_float(k0 + i));
    }
    cluster_sync_all();   // every slice is sorted and visible cluster-wide

    // 4. queries
    const uint32_t pts_sh = (uint32_t)__cvta_generic_to_shared(pts), cs_sh = (uint32_t)__cvta_generic_to_shared(cs);
    const float c_lin = (inv_c > 0.f ? 1.0f / inv_c : 0.f) * 0.9995f;
    const int q_end = min(n, (part + 1) * rows);
    for (int p = part * rows + (int)rank * TN_WARPS + warp; p < q_end; p += (int)csize * TN_WARPS) {
        const float *u = unknown + ((size_t)b * n + p) * 3;
        const float qx = __ldg(u), qy = __ldg(u + 1), qz = __ldg(u + 2);
        const float tx = (qx - x0) * inv_c, ty = (qy - y0) * inv_c;
        // the query may lie outside the box (or be NaN): start from the nearest cell
        const int cx = (int)fminf(fmaxf(floorf(tx), 0.f), (float)(gx - 1));
        const int cy = (int)fminf(fmaxf(floorf(ty), 0.f), (float)(gy - 1));
        const int rmax = max(max(cx, gx - 1 - cx), max(cy, gy - 1 - cy));
        unsigned long long k1 = TN_EMPTY, k2 = TN_EMPTY, k3 = TN_EMPTY;
        for (int R = 1;; ++R) {
            // segments of cells (one row, a run of x) new at this step: the 3 x 3 block first, then the ring at distance R
            const int nseg = R == 1 ? 3 : 4 * R;
            for (int q0 = 0; q0 < nseg << lc; q0 += 32) {
                // lane = one (segment, CTA) pair: its run of that CTA's cell-major points
                const int q = q0 + (int)lane, s = q >> lc;
                const uint32_t cta = (uint32_t)q & (csize - 1u);
                int y, xa, xb;
                if (R == 1) { y = cy - 1 + s; xa = cx - 1; xb = cx + 1; }
                else if (s < 2) { y = s ? cy + R : cy - R; xa = cx - R; xb = cx + R; }
                else { y = cy - R + 1 + ((s - 2) >> 1); xa = xb = (s & 1) ? cx + R : cx - R; }
                xa = max(xa, 0); xb = min(xb, gx - 1);
                int beg = 0, len = 0;
                if (s < nseg && y >= 0 && y < gy && xa <= xb) {
                    const uint32_t a = cluster_map_shared(cs_sh, cta) + 4u * (uint32_t)(y * gx);
                    beg = ld_cluster_s32(a + 4u * (uint32_t)xa);
                    len = ld_cluster_s32(a + 4u * (uint32_t)(xb + 1)) - beg;
                }
                int incl = len;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                    if ((int)lane >= o) incl += v;
                }
                const int total = __shfl_sync(0xFFFFFFFFu, incl, 31);
                const int base = beg - (incl - len);   // candidate k of this pair is point k + base of its CTA
                for (int j0 = 0; j0 < total; j0 += 32) {
                    const int k = j0 + (int)lane;
                    int L = 0;   // the pair holding candidate k: the first lane whose inclusive count exceeds k
#pragma unroll
                    for (int st = 16; st > 0; st >>= 1)
                        if (__shfl_sync(0xFFFFFFFFu, incl, L + st - 1) <= k) L += st;
                    const int kb = __shfl_sync(0xFFFFFFFFu, base, L);
                    if (k < total) {
                        const float4 v = ld_cluster_f4(cluster_map_shared(pts_sh, (uint32_t)L & (csize - 1u)) + 16u * (uint32_t)(k + kb));
                        const float d = sqdist3(qx, qy, qz, v.x, v.y, v.z);
                        top3_insert(((unsigned long long)__float_as_uint(d) << 32) | __float_as_uint(v.w), k1, k2, k3);
                    }
                }
            }
            // the warp's three smallest keys (ids are unique, so one lane pops each; empty keys pop harmlessly)
            unsigned long long g[3];
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                const uint32_t hi = (uint32_t)(k1 >> 32);
                const uint32_t mh = __reduce_min_sync(0xFFFFFFFFu, hi);
                const uint32_t ml = __reduce_min_sync(0xFFFFFFFFu, hi == mh ? (uint32_t)k1 : 0xFFFFFFFFu);
                g[r] = ((unsigned long long)mh << 32) | ml;
                if (k1 == g[r]) { k1 = k2; k2 = k3; k3 = TN_EMPTY; }
            }
            // lane 0 keeps them, the other lanes start empty
            k1 = lane ? TN_EMPTY : g[0]; k2 = lane ? TN_EMPTY : g[1]; k3 = lane ? TN_EMPTY : g[2];
            if (R >= rmax) break;
            if (tn_ring_bound(tx, ty, cx, cy, R, gx, gy, c_lin) > __uint_as_float((uint32_t)(g[2] >> 32))) break;
        }
        // lane r < 3 writes slot r of lane 0's list
        const unsigned long long s2 = __shfl_sync(0xFFFFFFFFu, k2, 0), s3 = __shfl_sync(0xFFFFFFFFu, k3, 0);
        const unsigned long long g = lane == 0 ? k1 : (lane == 1 ? s2 : s3);
        if (lane < 3) {
            dist2[((size_t)b * n + p) * 3 + lane] = __uint_as_float((uint32_t)(g >> 32));
            idx[((size_t)b * n + p) * 3 + lane] = (int)(uint32_t)g;
        }
    }
    cluster_sync_all();   // no CTA leaves while another may still read its shared memory
}

// out[b,c,j] = w0*p[i0] + w1*p[i1] + w2*p[i2]; the reference build contracts this into
// FMUL t = w1*p1 ; FFMA t = w0*p0 + t ; FFMA out = w2*p2 + t  (SASS of the rebuilt reference object).
__global__ void __launch_bounds__(256)
three_interpolate_kernel(int c, int m, int n, const float *__restrict__ points, const int *__restrict__ idx,
                         const float *__restrict__ weight, float *__restrict__ out) {
    const int b = blockIdx.z;
    const int j = blockIdx.x * 256 + threadIdx.x;
    if (j >= n) return;
    const int *ix = idx + ((size_t)b * n + j) * 3;
    const float *w = weight + ((size_t)b * n + j) * 3;
    const int i0 = __ldg(ix), i1 = __ldg(ix + 1), i2 = __ldg(ix + 2);
    const float w0 = __ldg(w), w1 = __ldg(w + 1), w2 = __ldg(w + 2);
    const int c0 = blockIdx.y * 8, c1 = min(c, c0 + 8);
    for (int ci = c0; ci < c1; ++ci) {
        const float *src = points + ((size_t)b * c + ci) * m;
        const float t = __fmaf_rn(w0, __ldg(src + i0), __fmul_rn(w1, __ldg(src + i1)));
        out[((size_t)b * c + ci) * n + j] = __fmaf_rn(w2, __ldg(src + i2), t);
    }
}

__global__ void __launch_bounds__(256)
three_interpolate_grad_kernel(int c, int n, int m, const float *__restrict__ grad_out, const int *__restrict__ idx,
                              const float *__restrict__ weight, float *__restrict__ grad_points) {
    const int b = blockIdx.z;
    const int j = blockIdx.x * 256 + threadIdx.x;
    if (j >= n) return;
    const int *ix = idx + ((size_t)b * n + j) * 3;
    const float *w = weight + ((size_t)b * n + j) * 3;
    const int i0 = __ldg(ix), i1 = __ldg(ix + 1), i2 = __ldg(ix + 2);
    const float w0 = __ldg(w), w1 = __ldg(w + 1), w2 = __ldg(w + 2);
    const int c0 = blockIdx.y * 8, c1 = min(c, c0 + 8);
    for (int ci = c0; ci < c1; ++ci) {
        const float g = __ldg(grad_out + ((size_t)b * c + ci) * n + j);
        float *dst = grad_points + ((size_t)b * c + ci) * m;
        atomicAdd(dst + i0, __fmul_rn(g, w0));
        atomicAdd(dst + i1, __fmul_rn(g, w1));
        atomicAdd(dst + i2, __fmul_rn(g, w2));
    }
}

}  // namespace spsk

extern "C" int spsk_three_nn(int b, int n, int m, const float *unknown, const float *known, float *dist2, int *idx,
                             spsk_stream_t stream) {
    using namespace spsk;
    SPSK_REQUIRE(b >= 0 && n >= 0 && m >= 0 && b <= 65535, SPSK_ERR_INVALID_ARG, "three_nn: bad sizes b=%d n=%d m=%d", b, n, m);
    if (b == 0 || n == 0) return SPSK_OK;
    SPSK_REQUIRE(unknown && known && dist2 && idx, SPSK_ERR_INVALID_ARG, "three_nn: null pointer");
    cudaStream_t st = as_stream(stream);
    if (n >= SPSK_THREE_NN_GRID_MIN_N && m >= SPSK_THREE_NN_GRID_MIN_M && m <= SPSK_THREE_NN_GRID_MAX_M) {
        int csize = 1;   // the smallest cluster in which a CTA holds at most TN_CAP known points
        while ((m + csize - 1) / csize > TN_CAP) csize *= 2;
        const int chunk = (m + csize - 1) / csize;
        // about two waves of one CTA per SM (each cluster rebuilds its scene's grid), at least one unknown point per warp
        const int per_scene = max(1, min((2 * SPSK_NUM_SMS) / (csize * b), (n + csize * TN_WARPS - 1) / (csize * TN_WARPS)));
        const int rows = (n + per_scene - 1) / per_scene;
        static ClusterKernelState state;
        const int rc = launch_cluster(state, three_nn_cluster_kernel, "three_nn_cluster_kernel", b * per_scene, csize,
                                      TN_THREADS, TN_SMEM, st, n, m, chunk, per_scene, rows, unknown, known, dist2, idx);
        if (rc != SPSK_CLUSTER_UNSCHEDULABLE) return rc;   // else: the brute-force kernel, same results
    }
    dim3 grid((n + NN_THREADS - 1) / NN_THREADS, b);
    three_nn_kernel<<<grid, NN_THREADS, 0, st>>>(n, m, unknown, known, dist2, idx);
    SPSK_LAUNCH_CHECK("three_nn_kernel");
    return SPSK_OK;
}

extern "C" int spsk_three_interpolate(int b, int c, int m, int n, const float *points, const int *idx,
                                      const float *weight, float *out, spsk_stream_t stream) {
    using namespace spsk;
    SPSK_REQUIRE(b >= 0 && c >= 0 && n >= 0 && m >= 0 && b <= 65535, SPSK_ERR_INVALID_ARG, "three_interpolate: bad sizes");
    if (b == 0 || c == 0 || n == 0) return SPSK_OK;
    SPSK_REQUIRE(points && idx && weight && out, SPSK_ERR_INVALID_ARG, "three_interpolate: null pointer");
    dim3 grid((n + 255) / 256, (c + 7) / 8, b);
    three_interpolate_kernel<<<grid, 256, 0, as_stream(stream)>>>(c, m, n, points, idx, weight, out);
    SPSK_LAUNCH_CHECK("three_interpolate_kernel");
    return SPSK_OK;
}

extern "C" int spsk_three_interpolate_grad(int b, int c, int n, int m, const float *grad_out, const int *idx,
                                           const float *weight, float *grad_points, spsk_stream_t stream) {
    using namespace spsk;
    SPSK_REQUIRE(b >= 0 && c >= 0 && n >= 0 && m >= 0 && b <= 65535, SPSK_ERR_INVALID_ARG, "three_interpolate_grad: bad sizes");
    if (b == 0 || c == 0 || n == 0) return SPSK_OK;
    SPSK_REQUIRE(grad_out && idx && weight && grad_points, SPSK_ERR_INVALID_ARG, "three_interpolate_grad: null pointer");
    dim3 grid((n + 255) / 256, (c + 7) / 8, b);
    three_interpolate_grad_kernel<<<grid, 256, 0, as_stream(stream)>>>(c, n, m, grad_out, idx, weight, grad_points);
    SPSK_LAUNCH_CHECK("three_interpolate_grad_kernel");
    return SPSK_OK;
}
