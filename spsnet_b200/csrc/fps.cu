// fps.cu -- farthest point sampling (D-FPS on xyz, F-FPS on a precomputed distance matrix).
//
// Replaces farthest_point_sampling_kernel / furthest_point_sampling_with_dist_kernel of the
// reference (src/sampling_gpu.cu:93-209, 256-371).  Same arithmetic, same winners (bit-exact,
// including the block-tree tie-break, see common.cuh::fps_rank), different machine mapping.
// FPS is latency bound: m-1 strictly sequential arg-max steps per scene.
//
//   D-FPS, 1024 <= n <= 16384        fps_pruned_kernel, one CTA per scene: only the sub-buckets of Morton-sorted points that
//                                    a new sample can change are updated; running minima in tensor or shared memory
//   D-FPS, 16384 < n <= 262144       fps_pruned_kernel on one 2/4/8/16-CTA cluster per scene, arg-max across the cluster
//                                    through distributed shared memory
//   n < 1024, F-FPS, SPSK_FPS=dense  fps_kernel_1024 / fps_kernel: every point every step, running minima in registers, xyz
//                                    staged once into shared memory, 1 __syncthreads per step (the reference takes 11)
//   larger scenes                    fps_generic_kernel: running minima in the caller's `temp`
#include "mma_ptx.cuh"
#include <stdlib.h>

namespace spsk {

// order-preserving float -> uint map (handles negatives; -0 is canonicalised by the caller)
__device__ __forceinline__ uint32_t ordered_bits(float f) {
    uint32_t u = __float_as_uint(f);
    return u ^ ((u >> 31) ? 0xFFFFFFFFu : 0x80000000u);
}

// Block-wide arg-max of (value, ~rank): returns the winning point index to every thread.
// slots: W uint2 entries for this iteration's parity.  One barrier.
__device__ __forceinline__ uint32_t block_argmax(uint32_t u, uint32_t inv_rank, uint2 *slots, int nwarps,
                                                 uint32_t s_mask, uint32_t s_log2) {
    const uint32_t lane = lane_id();
    const uint32_t warp = threadIdx.x >> 5;
    const uint32_t m = __reduce_max_sync(0xFFFFFFFFu, u);
    const uint32_t c = (u == m) ? inv_rank : 0u;
    const uint32_t r = __reduce_max_sync(0xFFFFFFFFu, c);
    if (lane == 0) slots[warp] = make_uint2(m, r);
    __syncthreads();
    uint2 v = make_uint2(0u, 0u);
    if ((int)lane < nwarps) v = slots[lane];
    const uint32_t m2 = __reduce_max_sync(0xFFFFFFFFu, v.x);
    const uint32_t c2 = (v.x == m2) ? v.y : 0u;
    const uint32_t r2 = __reduce_max_sync(0xFFFFFFFFu, c2);
    return fps_unrank(~r2, s_mask, s_log2);
}

// Main kernel, n >= 1024 (reference block size S = 1024 = T).  All points of one thread (k = tid + p*T)
// share k mod S and rank(k) grows with p, so "first strict maximum in p order" is exactly the
// reference's in-thread rule AND its tree tie-break restricted to this thread.  T is a compile-time
// constant and padding points carry tmp = -1 (fminf(d, -1) = -1 never beats best >= -1), so the
// unrolled body is branch-free straight-line code: 3 LDS (or registers) + 10 ALU per point.
template <int P, bool REGXYZ, bool DISTMAT>
__global__ void __launch_bounds__(1024, 1)
fps_kernel_1024(int n, int m, const float *__restrict__ src, float *__restrict__ temp, int *__restrict__ idx) {
    constexpr int T = 1024;
    constexpr uint32_t s_mask = 1023u, s_log2 = 10u;
    extern __shared__ float smem[];
    __shared__ uint2 slots[2][32];
    const int tid = threadIdx.x;
    const size_t scene = blockIdx.x;
    constexpr int NP = P * T;  // padded point count
    float *sx = smem, *sy = smem + NP, *sz = smem + 2 * NP;
    const float *base = DISTMAT ? src + scene * (size_t)n * n : src + scene * (size_t)n * 3;
    if (temp) temp += scene * (size_t)n;
    idx += scene * (size_t)m;

    if (!DISTMAT) {
        for (int i = tid; i < 3 * NP; i += T) smem[i] = 0.f;
        __syncthreads();
        for (int i = tid; i < 3 * n; i += T) {
            const float v = __ldg(base + i);
            const int k = i / 3, c = i - 3 * k;
            smem[c * NP + k] = v;
        }
        __syncthreads();
    }

    float tmp[P];
    float px[REGXYZ ? P : 1], py[REGXYZ ? P : 1], pz[REGXYZ ? P : 1];
#pragma unroll
    for (int p = 0; p < P; ++p) {
        const int k = tid + p * T;
        tmp[p] = (k < n) ? (temp ? temp[k] : 1e10f) : -1.f;
        if (REGXYZ) { px[p] = sx[k]; py[p] = sy[k]; pz[p] = sz[k]; }
    }

    int old = 0;
    int keep = 0;   // picks are flushed 32 at a time by warp 0 (see fps_pruned_kernel); idx[0] = 0 lives in lane 0

    for (int j = 1; j < m; ++j) {
        float x1 = 0.f, y1 = 0.f, z1 = 0.f;
        const float *drow = nullptr;
        if (DISTMAT) {
            drow = base + (size_t)old * n;
        } else {
            x1 = sx[old]; y1 = sy[old]; z1 = sz[old];
        }
        float best = -1.f;
        int bp = 0;
#pragma unroll
        for (int p = 0; p < P; ++p) {
            const int k = tid + p * T;
            float d;
            if (DISTMAT) d = (k < n) ? __ldg(drow + k) : 0.f;
            else if (REGXYZ) d = sqdist3(px[p], py[p], pz[p], x1, y1, z1);
            else d = sqdist3(sx[k], sy[k], sz[k], x1, y1, z1);
            const float t = fminf(d, tmp[p]);
            tmp[p] = t;
            const bool gt = t > best;
            best = gt ? t : best;
            bp = gt ? p : bp;
        }
        const uint32_t kb = (uint32_t)(tid + bp * T);
        const uint32_t u = ordered_bits(__fadd_rn(best, 0.f));
        const uint32_t inv_rank = ~fps_rank(kb, s_mask, s_log2);
        old = (int)block_argmax(u, inv_rank, slots[j & 1], T / 32, s_mask, s_log2);
        if (tid < 32) {
            if ((tid & 31) == (j & 31)) keep = old;
            if ((j & 31) == 31) idx[j - 31 + tid] = keep;
        }
    }
    if (tid < 32 && (m & 31) != 0 && tid < (m & 31)) idx[(m & ~31) + tid] = keep;   // the last partial line

    if (temp) {
#pragma unroll
        for (int p = 0; p < P; ++p) {
            const int k = tid + p * T;
            if (k < n) temp[k] = tmp[p];
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// Spatially pruned D-FPS (same winners, far less work per step).
//
// The update temp[k] = min(temp[k], |p_k - q|^2) cannot change temp[k] when |p_k - q|^2 >= temp[k].  Points
// are sorted once along a Morton curve (in-kernel counting sort by cell code) and cut
// into sub-buckets of 32 consecutive points (one per lane).  Each sub-bucket keeps its bounding box, the
// maximum of its running minima (bmax) and the rank of its best point.  Per step a lane evaluates the
// box-to-query lower bound lb of "its" sub-bucket with THE SAME fp32 expression as the distance itself
// (fl() is monotone, so lb <= every fl(|p_k - q|^2) in the box) and the warp skips the sub-bucket when
// lb >= bmax -- exactly the sub-buckets whose temps provably do not change.  Surviving sub-buckets are
// updated with the reference arithmetic, so temps, maxima and the (value, rank) arg-max are bit-identical
// to the unpruned kernel; only the amount of work differs (after a few hundred samples a new point touches
// a handful of the 512 sub-buckets).  The sort only decides HOW MUCH is skipped, never the result.
//
// 512 threads, P points per lane (P*512 >= n), sub-bucket s = p*16 + warp (round-robin over warps so that
// neighbouring sub-buckets are processed by different warps), sorted xyz in shared memory (SoA), original
// indices in registers, running minima in tensor or shared memory (see below), orig->sorted position map (u16)
// in shared memory.
// CL = true: a thread-block CLUSTER per scene (n > 16384, e.g. Waymo's 65536 points): CTA r of the cluster owns the
// contiguous index range [r*chunk, (r+1)*chunk), prunes and updates it exactly like the single-CTA kernel, and the
// per-iteration arg-max is completed across the cluster through distributed shared memory: each CTA reduces its 16 warp
// summaries locally, warp 0 sends ONE (value, ~rank, x, y, z) record to every CTA of the cluster with st.async -- the
// store itself completes transaction bytes on the receiver's mbarrier, so there is no cluster barrier and no fence on the
// chain -- and every warp picks the winner among the csize records.  The winner's coordinates travel with the record, so
// no CTA ever reads another CTA's points.
// st.async: the store itself completes `16` transaction bytes on the consumer CTA's mbarrier -- data and signal in one
// message, no fence and no cluster barrier on the per-iteration chain (measured: barrier.cluster arrive.release +
// wait.acquire costs 518 cycles at 4 x 512 threads and compiles to MEMBAR.ALL.GPU + CCTL.IVALL around it).
__device__ __forceinline__ void st_async_v4(const void *local_rec, const void *local_bar, uint32_t cta, uint4 v) {
    const uint32_t ra = cluster_map_shared((uint32_t)__cvta_generic_to_shared(local_rec), cta);
    const uint32_t rb = cluster_map_shared((uint32_t)__cvta_generic_to_shared(local_bar), cta);
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];"
                 ::"r"(ra), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "r"(rb) : "memory");
}
// Not mma_ptx.cuh's mbar_wait: its spin counter and trap would add instructions to the per-step chain.
__device__ __forceinline__ void xbar_wait(uint64_t *bar, uint32_t parity) {
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(bar);
    uint32_t done = 0;
#pragma unroll 1
    while (!done) {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(done) : "r"(a), "r"(parity) : "memory");
    }
}

// PROF: compile the phase counters in (spsk_fps_set_profile).  They are predicated instructions, but on this latency chain
// every issue slot counts: 16 warps x ~40 predicated-off instructions per iteration were ~10 % of the iteration.
//
// Running minima (and each point's tie-break key ~rank): the index of a visited sub-bucket is DYNAMIC, so a visit is one
// generic loop body (ffs over the ballot mask, load, distance, store, two REDUX).  In registers the index would have to be
// static: the round-1 kernel ran a 32-case ladder of warp-uniform branches around 32 statically indexed copies of the body,
// ~400-500 cycles per visited sub-bucket on the critical warp against ~160 for the generic body (phase counters, round 2).
//  - P >= 16 (more than 4096 points per CTA, and every cluster CTA): TENSOR MEMORY.  The minima of a lane are private to it,
//    which is exactly the access pattern tcgen05.ld/st offer (a warp reaches the 32 TMEM lanes of its quarter; column =
//    sub-bucket; 12-cycle load).  Shared memory cannot take them (xyz 192 KB + index map 32 KB already fill it at 16384
//    points); the 256 KB of TMEM are otherwise unused by this kernel.  Layout: warp w owns columns [(w / 4) * 2P, +2P) of lane
//    quarter w % 4; sub-bucket p = columns (2p, 2p + 1) = (running minimum bits, ~rank or 0 for padding).
//  - P <= 8: SHARED memory, next to xyz.  Such a small CTA must not hold TMEM columns: it shares its SM with sa_mma CTAs that
//    allocate all 512.
template <int P, bool CL, bool PROF>
__global__ void __launch_bounds__(512, 1)
fps_pruned_kernel(int n_scene, int m, const float *__restrict__ src, float *__restrict__ temp, int *__restrict__ idx,
                  unsigned long long *__restrict__ prof) {
    constexpr int T = 512, W = 16, NP = T * P;
    constexpr bool TM = P >= 16;
    static_assert(TM || !CL, "the shared-memory minima follow the index map, which only a single-CTA scene has");
    constexpr uint32_t s_mask = 1023u, s_log2 = 10u;   // reference block size is 1024 for n >= 1024
    extern __shared__ float smem[];
    __shared__ float red[6][W];
    float *sx = smem, *sy = smem + NP, *sz = smem + 2 * NP;
    unsigned short *pos_of = reinterpret_cast<unsigned short *>(smem + 3 * NP);
    float *stmp = smem + 3 * NP + NP / 2;                        // !TM: running minima by sorted position ...
    uint32_t *sir = reinterpret_cast<uint32_t *>(stmp + NP);    // ... and ~rank (0 = padding)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t crank = CL ? cluster_ctarank() : 0u, csize = CL ? cluster_nctarank() : 1u;
    const size_t scene = CL ? blockIdx.x / csize : blockIdx.x;
    const int chunk = CL ? (n_scene + (int)csize - 1) / (int)csize : n_scene;
    const int gbase = (int)crank * chunk;                       // first scene index owned by this CTA
    const int n = max(0, min(n_scene - gbase, chunk));          // points owned by this CTA (<= NP)
    const float *scene_base = src + scene * (size_t)n_scene * 3;
    const float *base = scene_base + (size_t)gbase * 3;
    if (temp) temp += scene * (size_t)n_scene;   // indexed with scene indices
    idx += scene * (size_t)m;
    constexpr uint32_t TM_COLS = 8 * P < 32 ? 32 : 8 * P;   // 4 warps per lane quarter x P sub-buckets x 2 columns (power of two)
    __shared__ uint32_t tm_slot;
    if (TM && warp == 0) tmem_alloc(smem_u32(&tm_slot), TM_COLS);

    // ---- bounding box of the owned points (only scales the Morton cells: any box gives the same samples)
    float lo[3] = {3.0e38f, 3.0e38f, 3.0e38f}, hi[3] = {-3.0e38f, -3.0e38f, -3.0e38f};
    for (int i = tid; i < n; i += T) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float v = __ldg(base + (size_t)i * 3 + c);
            lo[c] = fminf(lo[c], v);
            hi[c] = fmaxf(hi[c], v);
        }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[c] = fminf(lo[c], __shfl_xor_sync(0xFFFFFFFFu, lo[c], o));
            hi[c] = fmaxf(hi[c], __shfl_xor_sync(0xFFFFFFFFu, hi[c], o));
        }
        if (lane == 0) { red[c][warp] = lo[c]; red[3 + c][warp] = hi[c]; }
    }
    __syncthreads();
    float scl[3], org[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        float l = red[c][0], h = red[3 + c][0];
        for (int w = 1; w < W; ++w) { l = fminf(l, red[c][w]); h = fmaxf(h, red[3 + c][w]); }
        org[c] = l;
        const float cells = (c == 2) ? 16.f : 128.f;
        scl[c] = cells / fmaxf(h - l, 1e-20f);
    }
    // ---- spatial order of the owned points.  It only decides HOW MUCH is pruned, never the result, so it need not be a total
    // order: a counting sort by the top log2(NP) bits of the (7+7-bit xy Morton, 4-bit z) cell code -- as many cells as point
    // slots -- replaces the full bitonic sort of (code, index) keys, which cost ~8 % of the 16384 -> 4096 kernel (105 passes over
    // 16384 keys, a block barrier each).  Shared-memory atomics, one scan, one scatter; the order inside a cell is whatever the
    // atomics give (run to run the sub-buckets may differ, the samples cannot).
    auto cell_code = [&](int i) -> uint32_t {
        const float x = __ldg(base + (size_t)i * 3), y = __ldg(base + (size_t)i * 3 + 1), z = __ldg(base + (size_t)i * 3 + 2);
        uint32_t cx = min(127, max(0, (int)((x - org[0]) * scl[0])));
        uint32_t cy = min(127, max(0, (int)((y - org[1]) * scl[1])));
        const uint32_t cz = min(15, max(0, (int)((z - org[2]) * scl[2])));
        cx = (cx | (cx << 4)) & 0x0F0Fu; cx = (cx | (cx << 2)) & 0x3333u; cx = (cx | (cx << 1)) & 0x5555u;
        cy = (cy | (cy << 4)) & 0x0F0Fu; cy = (cy | (cy << 2)) & 0x3333u; cy = (cy | (cy << 1)) & 0x5555u;
        return (((cx | (cy << 1)) & 0x3FFFu) << 4) | cz;   // 18 bits
    };
    // [hist u32 x NP][codes u16 x NP][sorted u16 x NP] = 8 NP bytes of the 12 NP-byte xyz region
    uint32_t *hist = reinterpret_cast<uint32_t *>(smem);
    unsigned short *codes = reinterpret_cast<unsigned short *>(smem) + 2 * NP;
    unsigned short *sorted16 = reinterpret_cast<unsigned short *>(smem) + 3 * NP;   // point index by sorted position
    constexpr int CB = (P == 2 ? 10 : P == 4 ? 11 : P == 8 ? 12 : P == 16 ? 13 : 14);   // log2(NP) cells
    for (int i = tid; i < NP; i += T) { hist[i] = 0u; sorted16[i] = 0xFFFFu; }
    __syncthreads();
    for (int i = tid; i < n; i += T) {
        const uint32_t c = cell_code(i) >> (18 - CB);
        codes[i] = (unsigned short)c;
        atomicAdd(&hist[c], 1u);
    }
    __syncthreads();
    // exclusive scan over the NP counters: thread t owns counters [t P, (t + 1) P)
    uint32_t loc[P], run = 0u;
#pragma unroll
    for (int p = 0; p < P; ++p) { loc[p] = run; run += hist[tid * P + p]; }
    uint32_t inc = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t up = __shfl_up_sync(0xFFFFFFFFu, inc, o);
        if (lane >= o) inc += up;
    }
    uint32_t *wsum = reinterpret_cast<uint32_t *>(&red[0][0]);   // 16 warp totals (red is free again: the box is reduced)
    __syncthreads();
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    uint32_t wbase = 0u;
    for (int w = 0; w < warp; ++w) wbase += wsum[w];
    const uint32_t excl = wbase + inc - run;
#pragma unroll
    for (int p = 0; p < P; ++p) hist[tid * P + p] = excl + loc[p];
    __syncthreads();
    for (int i = tid; i < n; i += T) sorted16[atomicAdd(&hist[codes[i]], 1u)] = (unsigned short)i;
    __syncthreads();
    // ---- take ownership: slot p of this lane = sorted position ((p*W + warp)*32 + lane)
    uint32_t oidx[P];
#pragma unroll
    for (int p = 0; p < P; ++p) {
        const uint32_t v = sorted16[(p * W + warp) * 32 + lane];
        oidx[p] = v == 0xFFFFu ? 0xFFFFFFFFu : v;
    }
    if (TM) tc_fence_before();
    __syncthreads();   // sorted16 consumed; the region becomes sx/sy/sz
    uint32_t tbase = 0u;   // TM: this warp's first column in its lane quarter
    if (TM) {
        tc_fence_after();
        tbase = tm_slot + ((uint32_t)(warp & 3) << 21) + (uint32_t)(warp >> 2) * (2u * P);   // lane field = bits 31:16
    }
#pragma unroll
    for (int p = 0; p < P; ++p) {
        const int pos = (p * W + warp) * 32 + lane;
        const bool valid = oidx[p] != 0xFFFFFFFFu;
        const uint32_t oi = valid ? oidx[p] : 0u;                // index inside the owned range
        oidx[p] = valid ? oi + (uint32_t)gbase : 0xFFFFFFFFu;   // index inside the scene (decides the tie-break rank)
        sx[pos] = valid ? __ldg(base + (size_t)oi * 3) : 0.f;
        sy[pos] = valid ? __ldg(base + (size_t)oi * 3 + 1) : 0.f;
        sz[pos] = valid ? __ldg(base + (size_t)oi * 3 + 2) : 0.f;
        const float t0 = valid ? (temp ? temp[oidx[p]] : 1e10f) : -1.f;
        if (TM) tmem_st_x2(tbase + 2u * p, __float_as_uint(t0), valid ? ~fps_rank(oidx[p], s_mask, s_log2) : 0u);
        else { stmp[pos] = t0; sir[pos] = valid ? ~fps_rank(oidx[p], s_mask, s_log2) : 0u; }
        if (!CL && valid) pos_of[oi] = (unsigned short)pos;
    }
    if (TM) tmem_wait_st();
    __syncthreads();
    // ---- sub-bucket boxes: lane p keeps the box / bmax / best-rank of slot p of this warp
    float bx0 = 3.0e38f, bx1 = -3.0e38f, by0 = 3.0e38f, by1 = -3.0e38f, bz0 = 3.0e38f, bz1 = -3.0e38f;
    uint32_t bmax_bits = 0u, brank = 0u;
#pragma unroll
    for (int p = 0; p < P; ++p) {
        const int pos = (p * W + warp) * 32 + lane;
        const bool valid = oidx[p] != 0xFFFFFFFFu;
        float a0 = valid ? sx[pos] : 3.0e38f, a1 = valid ? sx[pos] : -3.0e38f;
        float c0 = valid ? sy[pos] : 3.0e38f, c1 = valid ? sy[pos] : -3.0e38f;
        float e0 = valid ? sz[pos] : 3.0e38f, e1 = valid ? sz[pos] : -3.0e38f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            a0 = fminf(a0, __shfl_xor_sync(0xFFFFFFFFu, a0, o)); a1 = fmaxf(a1, __shfl_xor_sync(0xFFFFFFFFu, a1, o));
            c0 = fminf(c0, __shfl_xor_sync(0xFFFFFFFFu, c0, o)); c1 = fmaxf(c1, __shfl_xor_sync(0xFFFFFFFFu, c1, o));
            e0 = fminf(e0, __shfl_xor_sync(0xFFFFFFFFu, e0, o)); e1 = fmaxf(e1, __shfl_xor_sync(0xFFFFFFFFu, e1, o));
        }
        const bool any_valid = __any_sync(0xFFFFFFFFu, valid);
        if (lane == p) {
            bx0 = a0; bx1 = a1; by0 = c0; by1 = c1; bz0 = e0; bz1 = e1;
            bmax_bits = any_valid ? 0x7F800000u : 0u;   // +inf: the first step visits every populated sub-bucket
        }
    }

    // Per iteration (the m-1 iterations are strictly sequential, so this loop is a latency chain):
    //   1. every lane p < P bounds "its" sub-bucket against the new sample and the warp ballots the buckets to visit;
    //   2. visited buckets only (a handful out of n/32 after the first few hundred samples) are updated, one generic
    //      body per set bit of the ballot, their running minima loaded and stored at a dynamic TMEM column (or shared
    //      memory slot);
    //   3. warp arg-max over the P bucket summaries, one 16-byte slot per warp (value, ~rank, sorted position of the
    //      bucket's best point), one barrier, arg-max over the 16 slots.  The winner's SORTED POSITION travels with the
    //      slot, so the next iteration reads its coordinates directly (no index -> position lookup on the chain).
    // Ties are rare: each arg-max first reduces the value alone and only falls back to the second (rank) reduction
    // when the maximum is not unique.
    __shared__ uint2 slots2[2][32];           // single CTA: one (value, ~rank) slot per warp; entries >= W stay zero so the
                                              // read-back needs no lane guard (a divergent load costs a BSSY/BSYNC pair)
    __shared__ uint4 crec[CL ? 2 : 1][CL ? 16 : 1][2];   // cluster: [parity][cta] = {value, ~rank, x, y | z, -, -, -}, one record per CTA
    __shared__ uint4 cslot[CL ? 2 : 1][CL ? 32 : 1];       // cluster: per-warp {value, ~rank, sorted position, -}; entries >= W stay zero
    __shared__ uint64_t xbar[2];                         // cluster: transaction barriers of the two record tables
    if (tid < 64) slots2[tid >> 5][tid & 31] = make_uint2(0u, 0u);
    if (CL) {
        if (tid < 64) cslot[tid >> 5][tid & 31] = make_uint4(0u, 0u, 0u, 0u);
        if (tid == 0) {
            mbar_init(smem_u32(&xbar[0]), 1);
            mbar_init(smem_u32(&xbar[1]), 1);
            mbar_init_fence();
            // the one local arrival + the bytes a phase receives: one 32-byte record from every CTA of the cluster
            mbar_expect_tx(smem_u32(&xbar[0]), csize * 32u);
            mbar_expect_tx(smem_u32(&xbar[1]), csize * 32u);
        }
    }
    __syncthreads();
    uint32_t bpos = 0u;   // lane p: sorted position of sub-bucket p's best point
    // The picks are written 32 at a time: lane (j & 31) of warp 0 keeps pick j in a register and the warp stores one
    // coalesced 128-byte line every 32 iterations.  A store per iteration sits on the latency chain: the CTA barrier of the
    // next iteration orders memory, so it waits for the store's acknowledgement from L2.
    int keep = 0;   // idx[0] = 0 (reference :113-115) lives in lane 0 until the first flush
    int qpos = CL ? 0 : pos_of[0];   // first sample is point 0 (reference :113-115)
    float qx = __ldg(scene_base), qy = __ldg(scene_base + 1), qz = __ldg(scene_base + 2);
    if (CL) cluster_sync_all();      // every CTA of the cluster is resident before the first remote store
    // optional profiling (spsk_fps_set_profile): cycles of warp 0 per phase + sub-buckets visited by all warps
    const bool pf = PROF && prof != nullptr && tid == 0 && !CL;
    unsigned long long pc[6] = {0, 0, 0, 0, 0, 0};
    unsigned long long visited = 0;
    uint32_t wm = 0u, wr = 0u, wpos = 0u;   // this warp's best (value, ~rank, position): recomputed only after a visit

    for (int j = 1; j < m; ++j) {
        long long t0 = (PROF && pf) ? clock64() : 0;
        const float x1 = CL ? qx : sx[qpos], y1 = CL ? qy : sy[qpos], z1 = CL ? qz : sz[qpos];
        // box lower bound with the distance's own expression (monotone => rigorous in fp32)
        const float lx = fmaxf(fmaxf(__fsub_rn(bx0, x1), __fsub_rn(x1, bx1)), 0.f);
        const float ly = fmaxf(fmaxf(__fsub_rn(by0, y1), __fsub_rn(y1, by1)), 0.f);
        const float lz = fmaxf(fmaxf(__fsub_rn(bz0, z1), __fsub_rn(z1, bz1)), 0.f);
        const float lb = __fmaf_rn(lz, lz, __fmaf_rn(lx, lx, __fmul_rn(ly, ly)));
        const bool act = (lane < P) && (lb < __uint_as_float(bmax_bits));
        const uint32_t mask = __ballot_sync(0xFFFFFFFFu, act);
        if (PROF && pf) { const long long t1 = clock64(); pc[0] += t1 - t0; t0 = t1; }
        if (PROF && prof != nullptr && lane == 0) visited += __popc(mask);
        // visit: the running minimum and the point's tie-break key come from TMEM (or shared memory)
        uint32_t mk = mask;
        while (mk) {
            const int pb = __ffs(mk) - 1;
            mk &= mk - 1u;
            const int pos = (pb * W + warp) * 32 + lane;
            uint32_t tb, ir;
            if (TM) tmem_ld_x2(tbase + 2u * (uint32_t)pb, tb, ir);
            else { tb = __float_as_uint(stmp[pos]); ir = sir[pos]; }
            const float d = sqdist3(sx[pos], sy[pos], sz[pos], x1, y1, z1);
            const float t = fminf(d, __uint_as_float(tb));
            if (TM) tmem_st_x1(tbase + 2u * (uint32_t)pb, __float_as_uint(t));
            else stmp[pos] = t;
            const uint32_t u = (t > 0.f) ? __float_as_uint(t) : 0u;   // padding keeps t = -1, ir = 0
            const uint32_t mx = __reduce_max_sync(0xFFFFFFFFu, u);
            const uint32_t cand = (u == mx) ? ir : 0u;
            const uint32_t rr = __reduce_max_sync(0xFFFFFFFFu, cand);
            uint32_t bp = 0u;   // cluster mode only: the best point's position travels with the summary
            if (CL) bp = __reduce_max_sync(0xFFFFFFFFu, (ir != 0u && cand == rr) ? (uint32_t)pos : 0u);
            if (lane == pb) { bmax_bits = mx; brank = rr; bpos = bp; }
        }
        // (the tcgen05.wait::st that orders these stores before the next load of the same columns -- a later iteration -- is
        // taken after the block barrier below, off the critical warp's path to it)
        if (PROF && pf) { const long long t1 = clock64(); pc[1] += t1 - t0; t0 = t1; }
        // warp best over its P sub-buckets: unchanged (cached) when this warp visited nothing -- most warps, most iterations;
        // their REDUX would only compete with the critical warp's for the same unit
        if (mask) {
            const uint32_t wv = (lane < P) ? bmax_bits : 0u;
            wm = __reduce_max_sync(0xFFFFFFFFu, wv);
            const uint32_t wc = (lane < P && bmax_bits == wm) ? brank : 0u;
            wr = __reduce_max_sync(0xFFFFFFFFu, wc);
            // (value, ~rank) identifies one point, so exactly one lane matches: a max-reduction moves its position
            if (CL) wpos = __reduce_max_sync(0xFFFFFFFFu, (lane < P && bmax_bits == wm && brank == wr) ? bpos : 0u);
        }
        if (!CL) {
            uint2 *sl = slots2[j & 1];
            if (lane == 0) {
                sl[warp] = make_uint2(wm, wr);
            }
            if (PROF && pf) { const long long t1 = clock64(); pc[2] += t1 - t0; t0 = t1; }
            __syncthreads();
            if (TM && mask) tmem_wait_st();
            if (PROF && pf) { const long long t1 = clock64(); pc[3] += t1 - t0; t0 = t1; }
            // block best over the W warp slots
            const uint2 v = sl[lane];
            // (tried in round 2 and dropped: the block maximum of the value through a native shared-memory atomicMax + ballot /
            // shuffle for the rank instead of the two REDUX below -- 1086 vs 895 cycles per iteration: the atomic sits in front of
            // the barrier on every warp and VOTE + SHFL are no faster than one REDUX)
            const uint32_t m2 = __reduce_max_sync(0xFFFFFFFFu, v.x);
            const uint32_t r2 = __reduce_max_sync(0xFFFFFFFFu, (v.x == m2) ? v.y : 0u);
            // the sample's original index; its sorted position through the map
            const int old = (int)fps_unrank(~r2, s_mask, s_log2);
            qpos = pos_of[old];
            if (warp == 0) {
                if (lane == (j & 31)) keep = old;
                if ((j & 31) == 31) idx[j - 31 + lane] = keep;
            }
            if (PROF && pf) { const long long t1 = clock64(); pc[4] += t1 - t0; t0 = t1; }
        } else {
            // 1. CTA-local arg-max over the W warp slots (same as the single-CTA kernel, the winner's sorted position rides along)
            uint4 *cs_ = cslot[j & 1];
            if (lane == 0) cs_[warp] = make_uint4(wm, wr, wpos, 0u);
            __syncthreads();
            if (TM && mask) tmem_wait_st();
            const uint4 sv = cs_[lane];
            const uint32_t cm = __reduce_max_sync(0xFFFFFFFFu, sv.x);
            const uint32_t cr = __reduce_max_sync(0xFFFFFFFFu, (sv.x == cm) ? sv.y : 0u);
            uint4(*tab)[2] = crec[j & 1];
            uint64_t *xb = &xbar[j & 1];
            // 2. warp 0 sends this CTA's record {value, ~rank, x, y | z} to every CTA of the cluster; the stores themselves
            //    complete the transaction bytes the receivers' barriers were armed with (2 x 16 bytes per sender)
            if (warp == 0) {
                const int wl = __ffs(__ballot_sync(0xFFFFFFFFu, sv.x == cm && sv.y == cr)) - 1;
                const uint32_t rp = __shfl_sync(0xFFFFFFFFu, sv.z, wl);
                if (lane < csize) {
                    const float rx = sx[rp], ry = sy[rp], rz = sz[rp];
                    st_async_v4(&tab[crank][0], xb, lane, make_uint4(cm, cr, __float_as_uint(rx), __float_as_uint(ry)));
                    st_async_v4(&tab[crank][1], xb, lane, make_uint4(__float_as_uint(rz), 0u, 0u, 0u));
                }
            }
            // 3. wait for the csize records of this iteration: table (j & 1) is in its ((j - 1) / 2)-th phase
            xbar_wait(xb, (uint32_t)((j - 1) >> 1) & 1u);
            uint32_t bv = 0u, br = 0u;
            if (lane < csize) { const uint4 a0 = tab[lane][0]; bv = a0.x; br = a0.y; }
            const uint32_t m2 = __reduce_max_sync(0xFFFFFFFFu, bv);
            const uint32_t r2 = __reduce_max_sync(0xFFFFFFFFu, (lane < csize && bv == m2) ? br : 0u);
            const int wi = __ffs(__ballot_sync(0xFFFFFFFFu, lane < csize && bv == m2 && br == r2)) - 1;
            const uint4 w0 = tab[wi][0], w1 = tab[wi][1];
            qx = __uint_as_float(w0.z); qy = __uint_as_float(w0.w); qz = __uint_as_float(w1.x);
            // 4. re-arm this table's barrier for its next phase (iteration j + 2).  Safe to do as soon as this thread has passed
            //    the wait: no CTA can send iteration j + 2 before it has received OUR record of iteration j + 1, which is sent
            //    after this point; a slower warp of this CTA still waiting on the old parity sees it as completed.
            if (tid == 0) mbar_expect_tx(smem_u32(xb), csize * 32u);
            if (crank == 0 && warp == 0) {
                if (lane == (j & 31)) keep = (int)fps_unrank(~w0.y, s_mask, s_log2);
                if ((j & 31) == 31) idx[j - 31 + lane] = keep;
            }
        }
    }
    if (crank == 0 && warp == 0 && (m & 31) != 0 && lane < (m & 31)) idx[(m & ~31) + lane] = keep;   // the last partial line
    if (PROF && prof != nullptr) {
        if (pf) for (int i = 0; i < 5; ++i) atomicAdd(prof + i, pc[i]);
        if (lane == 0) atomicAdd(prof + 5, visited);
    }
    if (temp) {
#pragma unroll
        for (int p = 0; p < P; ++p) {
            uint32_t tb, ir;
            if (TM) tmem_ld_x2(tbase + 2u * p, tb, ir);
            else { const int pos = (p * W + warp) * 32 + lane; tb = __float_as_uint(stmp[pos]); ir = sir[pos]; }
            if (ir != 0u) temp[fps_unrank(~ir, s_mask, s_log2)] = __uint_as_float(tb);   // ~rank gives back the scene index
        }
    }
    if (TM) {
        tc_fence_before();
        __syncthreads();
        if (warp == 0) { tc_fence_after(); tmem_dealloc(tm_slot, TM_COLS); }
    }
}

static unsigned long long *g_fps_prof = nullptr;

// csize: CTAs per scene (CL only).  Returns SPSK_CLUSTER_UNSCHEDULABLE when the device cannot co-schedule such a cluster.
template <int P, bool CL>
static int launch_fps_pruned(int b, int n, int m, int csize, const float *src, float *temp, int *idx, cudaStream_t st) {
    const size_t smem = sizeof(float) * 3 * 512 * P + (CL ? 0 : sizeof(unsigned short) * 512 * P)   // xyz (+ index -> position map)
                        + (P >= 16 ? 0 : 8 * 512 * P);                                               // (+ minima and ~rank)
    const bool prof = g_fps_prof != nullptr;
    auto kern = prof ? fps_pruned_kernel<P, CL, true> : fps_pruned_kernel<P, CL, false>;
    if constexpr (CL) {
        static ClusterKernelState state[2];   // one per kernel: [prof]
        return launch_cluster(state[prof], kern, "fps_pruned_kernel", b, csize, 512, smem, st, n, m, src, temp, idx, g_fps_prof);
    }
    if (smem + 8192 > 48 * 1024) {
        static SmemAttrOnce attr[2];   // one per kernel: [prof]
        if (int rc = attr[prof].ensure(reinterpret_cast<const void *>(kern), (int)smem, "cudaFuncSetAttribute(fps_pruned_kernel)")) return rc;
    }
    kern<<<b, 512, smem, st>>>(n, m, src, temp, idx, g_fps_prof);
    SPSK_LAUNCH_CHECK("fps_pruned_kernel");
    return SPSK_OK;
}

// Small scenes, n < 1024: the reference block has S = 2^floor(log2 n) < 1024 threads; T = blockDim.x =
// max(S, 32) is a runtime multiple of S and every thread owns at most P = 2 points (same in-thread rule).
template <int P, bool REGXYZ, bool DISTMAT>
__global__ void __launch_bounds__(1024, 1)
fps_kernel(int n, int m, uint32_t s_mask, uint32_t s_log2, const float *__restrict__ src,
           float *__restrict__ temp, int *__restrict__ idx) {
    extern __shared__ float smem[];
    __shared__ uint2 slots[2][32];

    const int T = blockDim.x;
    const int tid = threadIdx.x;
    const int nwarps = T >> 5;
    const size_t scene = blockIdx.x;
    float *sx = smem, *sy = smem + n, *sz = smem + 2 * (size_t)n;
    const float *base = DISTMAT ? src + scene * (size_t)n * n : src + scene * (size_t)n * 3;
    if (temp) temp += scene * (size_t)n;
    idx += scene * (size_t)m;

    if (!DISTMAT) {
        for (int i = tid; i < 3 * n; i += T) {
            const float v = base[i];
            const int k = i / 3, c = i - 3 * k;
            smem[c * n + k] = v;
        }
        __syncthreads();
    }

    float tmp[P];
    float px[REGXYZ ? P : 1], py[REGXYZ ? P : 1], pz[REGXYZ ? P : 1];
#pragma unroll
    for (int p = 0; p < P; ++p) {
        const int k = tid + p * T;
        tmp[p] = (k < n) ? (temp ? temp[k] : 1e10f) : 0.f;
        if (REGXYZ) {
            px[p] = (k < n) ? sx[k] : 0.f;
            py[p] = (k < n) ? sy[k] : 0.f;
            pz[p] = (k < n) ? sz[k] : 0.f;
        }
    }

    int old = 0;
    int keep = 0;   // picks are flushed 32 at a time by warp 0 (see fps_pruned_kernel); idx[0] = 0 lives in lane 0
    const bool has_point = tid < n;

    for (int j = 1; j < m; ++j) {
        float x1 = 0.f, y1 = 0.f, z1 = 0.f;
        const float *drow = nullptr;
        if (DISTMAT) {
            drow = base + (size_t)old * n;
        } else {
            x1 = sx[old]; y1 = sy[old]; z1 = sz[old];
        }
        float best = -1.f;
        int bp = 0;
#pragma unroll
        for (int p = 0; p < P; ++p) {
            const int k = tid + p * T;
            if (k < n) {
                float d;
                if (DISTMAT) d = __ldg(drow + k);
                else if (REGXYZ) d = sqdist3(px[p], py[p], pz[p], x1, y1, z1);
                else d = sqdist3(sx[k], sy[k], sz[k], x1, y1, z1);
                const float t = fminf(d, tmp[p]);
                tmp[p] = t;
                if (t > best) { best = t; bp = p; }
            }
        }
        const uint32_t kb = (uint32_t)(tid + bp * T);
        const uint32_t u = has_point ? ordered_bits(__fadd_rn(best, 0.f)) : 0u;
        const uint32_t inv_rank = has_point ? ~fps_rank(kb, s_mask, s_log2) : 0u;
        old = (int)block_argmax(u, inv_rank, slots[j & 1], nwarps, s_mask, s_log2);
        if (tid < 32) {
            if ((tid & 31) == (j & 31)) keep = old;
            if ((j & 31) == 31) idx[j - 31 + tid] = keep;
        }
    }
    if (tid < 32 && (m & 31) != 0 && tid < (m & 31)) idx[(m & ~31) + tid] = keep;   // the last partial line

    if (temp) {
#pragma unroll
        for (int p = 0; p < P; ++p) {
            const int k = tid + p * T;
            if (k < n) temp[k] = tmp[p];
        }
    }
}

// Any-n fallback: running minima in the caller's `temp` (global/L2), xyz from global.  Same winners.
template <bool DISTMAT>
__global__ void __launch_bounds__(1024, 1)
fps_generic_kernel(int n, int m, uint32_t s_mask, uint32_t s_log2, const float *__restrict__ src,
                   float *__restrict__ temp, int *__restrict__ idx) {
    __shared__ uint2 slots[2][32];
    const int T = blockDim.x;
    const int tid = threadIdx.x;
    const size_t scene = blockIdx.x;
    const float *base = DISTMAT ? src + scene * (size_t)n * n : src + scene * (size_t)n * 3;
    temp += scene * (size_t)n;
    idx += scene * (size_t)m;
    int old = 0;
    int keep = 0;   // picks are flushed 32 at a time by warp 0 (see fps_pruned_kernel); idx[0] = 0 lives in lane 0
    const bool has_point = tid < n;
    for (int j = 1; j < m; ++j) {
        float x1 = 0.f, y1 = 0.f, z1 = 0.f;
        const float *drow = nullptr;
        if (DISTMAT) drow = base + (size_t)old * n;
        else { x1 = __ldg(base + old * 3); y1 = __ldg(base + old * 3 + 1); z1 = __ldg(base + old * 3 + 2); }
        float best = -1.f;
        int bk = tid;
        for (int k = tid; k < n; k += T) {
            float d;
            if (DISTMAT) d = __ldg(drow + k);
            else d = sqdist3(__ldg(base + k * 3), __ldg(base + k * 3 + 1), __ldg(base + k * 3 + 2), x1, y1, z1);
            const float t = fminf(d, temp[k]);
            temp[k] = t;
            if (t > best) { best = t; bk = k; }
        }
        const uint32_t u = has_point ? ordered_bits(__fadd_rn(best, 0.f)) : 0u;
        const uint32_t inv_rank = has_point ? ~fps_rank((uint32_t)bk, s_mask, s_log2) : 0u;
        old = (int)block_argmax(u, inv_rank, slots[j & 1], T >> 5, s_mask, s_log2);
        if (tid < 32) {
            if ((tid & 31) == (j & 31)) keep = old;
            if ((j & 31) == 31) idx[j - 31 + tid] = keep;
        }
    }
    if (tid < 32 && (m & 31) != 0 && tid < (m & 31)) idx[(m & ~31) + tid] = keep;   // the last partial line
}

template <int P, bool REGXYZ, bool DISTMAT>
static int launch_fps(int b, int n, int m, int threads, uint32_t s_mask, uint32_t s_log2, const float *src,
                      float *temp, int *idx, cudaStream_t st) {
    const size_t smem = DISTMAT ? 0 : sizeof(float) * 3 * (size_t)n;
    auto kern = fps_kernel<P, REGXYZ, DISTMAT>;
    if (smem + 2048 > 48 * 1024) {  // dynamic + the kernel's static smem must stay under the 48 KB default
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(fps_kernel)");
    }
    kern<<<b, threads, smem, st>>>(n, m, s_mask, s_log2, src, temp, idx);
    SPSK_LAUNCH_CHECK("fps_kernel");
    return SPSK_OK;
}

template <int P, bool REGXYZ, bool DISTMAT>
static int launch_fps_1024(int b, int n, int m, const float *src, float *temp, int *idx, cudaStream_t st) {
    const size_t smem = DISTMAT ? 0 : sizeof(float) * 3 * (size_t)P * 1024;
    auto kern = fps_kernel_1024<P, REGXYZ, DISTMAT>;
    if (smem + 2048 > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(fps_kernel_1024)");
    }
    kern<<<b, 1024, smem, st>>>(n, m, src, temp, idx);
    SPSK_LAUNCH_CHECK("fps_kernel_1024");
    return SPSK_OK;
}


// SPSK_FPS=dense selects the unpruned kernels (same results; used by the tests to cross-check both)
static bool fps_dense_forced() {
    const char *e = getenv("SPSK_FPS");
    return e && e[0] == 'd';
}

template <bool DISTMAT>
static int fps_dispatch(int b, int n, int m, const float *src, float *temp, int *idx, cudaStream_t st) {
    SPSK_REQUIRE(b >= 0 && n >= 1 && m >= 0, SPSK_ERR_INVALID_ARG, "fps: bad sizes b=%d n=%d m=%d", b, n, m);
    SPSK_REQUIRE(src && idx, SPSK_ERR_INVALID_ARG, "fps: null pointer");
    if (b == 0 || m == 0) return SPSK_OK;
    const int S = ref_block_threads(n);
    uint32_t s_log2 = 0;
    while ((1 << s_log2) < S) ++s_log2;
    const uint32_t s_mask = (uint32_t)S - 1u;
    const int threads = S < 32 ? 32 : S;  // multiple of S, >= one warp; 1024 for n >= 1024
    const int per_thread = (n + threads - 1) / threads;
    const bool fits = per_thread <= 16;  // 16 x 1024 padded points of SoA xyz = 192 KB of shared memory
    // n > 16384 (Waymo-shaped scenes): one cluster per scene, each CTA prunes its own slice, DSMEM arg-max.  Cluster size: the
    // fewest CTAs that hold the scene -- least SM-time per scene, which is what a pipelined serving loop pays.  n <= 16384 * cl,
    // so a CTA owns at most 16384 points: the P = 32 kernel holds them.  131072 < n <= 262144 takes a 16-CTA cluster
    // (non-portable size; falls through to the streaming kernel if the device cannot co-schedule it).
    if (!DISTMAT && threads == 1024 && n > 16384 && n <= 16 * 16384 && !fps_dense_forced()) {
        const int cl = n <= 2 * 16384 ? 2 : (n <= 4 * 16384 ? 4 : (n <= 8 * 16384 ? 8 : 16));
        const int rc = launch_fps_pruned<32, true>(b, n, m, cl, src, temp, idx, st);
        if (rc != SPSK_CLUSTER_UNSCHEDULABLE) return rc;
    }
    if (!fits) {
        SPSK_REQUIRE(temp != nullptr, SPSK_ERR_UNSUPPORTED,
                     "fps: n=%d exceeds the on-chip variants (<=131072, or <=262144 where 16-CTA clusters can run); pass a (b,n) `temp` scratch filled with 1e10", n);
        fps_generic_kernel<DISTMAT><<<b, threads, 0, st>>>(n, m, s_mask, s_log2, src, temp, idx);
        SPSK_LAUNCH_CHECK("fps_generic_kernel");
        return SPSK_OK;
    }
    if (!DISTMAT && threads == 1024 && n <= 16384 && !fps_dense_forced()) {
        if (n <= 1024) return launch_fps_pruned<2, false>(b, n, m, 1, src, temp, idx, st);
        if (n <= 2048) return launch_fps_pruned<4, false>(b, n, m, 1, src, temp, idx, st);
        if (n <= 4096) return launch_fps_pruned<8, false>(b, n, m, 1, src, temp, idx, st);
        if (n <= 8192) return launch_fps_pruned<16, false>(b, n, m, 1, src, temp, idx, st);
        return launch_fps_pruned<32, false>(b, n, m, 1, src, temp, idx, st);
    }
    if (threads == 1024) {
        if (per_thread <= 1) return launch_fps_1024<1, !DISTMAT, DISTMAT>(b, n, m, src, temp, idx, st);
        if (per_thread <= 2) return launch_fps_1024<2, !DISTMAT, DISTMAT>(b, n, m, src, temp, idx, st);
        if (per_thread <= 4) return launch_fps_1024<4, !DISTMAT, DISTMAT>(b, n, m, src, temp, idx, st);
        if (per_thread <= 8) return launch_fps_1024<8, !DISTMAT, DISTMAT>(b, n, m, src, temp, idx, st);
        return launch_fps_1024<16, false, DISTMAT>(b, n, m, src, temp, idx, st);
    }
    if (per_thread <= 1) return launch_fps<1, !DISTMAT, DISTMAT>(b, n, m, threads, s_mask, s_log2, src, temp, idx, st);
    return launch_fps<2, !DISTMAT, DISTMAT>(b, n, m, threads, s_mask, s_log2, src, temp, idx, st);
}

}  // namespace spsk

extern "C" int spsk_fps_set_profile(unsigned long long *counters) {
    spsk::g_fps_prof = counters;
    return SPSK_OK;
}

extern "C" int spsk_farthest_point_sampling(int b, int n, int m, const float *xyz, float *temp, int *idx,
                                            spsk_stream_t stream) {
    return spsk::fps_dispatch<false>(b, n, m, xyz, temp, idx, spsk::as_stream(stream));
}

extern "C" int spsk_furthest_point_sampling_with_dist(int b, int n, int m, const float *dist, float *temp,
                                                      int *idx, spsk_stream_t stream) {
    return spsk::fps_dispatch<true>(b, n, m, dist, temp, idx, spsk::as_stream(stream));
}
