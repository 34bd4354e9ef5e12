// common.cuh -- shared helpers for the sm_100a kernels behind include/spsk.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/spsk.h"

#ifndef SPSK_NUM_SMS
#define SPSK_NUM_SMS 148  // B200
#endif

namespace spsk {

// ---- error plumbing (thread-local message, C-ABI returns the code) --------------------------------
void set_error(const char *fmt, ...);
int cuda_fail(cudaError_t e, const char *what);
void count_launch();
unsigned int *fp16_overflow_word();   // device address of this device's fp16 range-guard word (api.cu), or nullptr
constexpr float FP16_MAX = 65504.f;

#define SPSK_REQUIRE(cond, code, ...)            \
    do {                                         \
        if (!(cond)) {                           \
            ::spsk::set_error(__VA_ARGS__);      \
            return (code);                       \
        }                                        \
    } while (0)

// every kernel launch of the library goes through this check and is counted (spsk_launch_count)
#define SPSK_LAUNCH_CHECK(what)                                   \
    do {                                                          \
        cudaError_t e__ = cudaGetLastError();                     \
        if (e__ != cudaSuccess) return ::spsk::cuda_fail(e__, what); \
        ::spsk::count_launch();                                   \
    } while (0)

static inline cudaStream_t as_stream(spsk_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

// index of the current device into the per-device tables below
static inline int device_slot() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
    return dev;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device attribute: set it once per (kernel, device).
struct SmemAttrOnce {
    bool done[64] = {};
    int ensure(const void *func, int bytes, const char *what) {
        const int dev = device_slot();
        if (done[dev]) return 0;
        cudaError_t e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        if (e != cudaSuccess) return cuda_fail(e, what);
        done[dev] = true;
        return 0;
    }
};

// reference: src/cuda_utils.h:10-14 opt_n_threads -- the block size the REFERENCE would launch the FPS
// kernels with; it decides the arg-max tie-break (see fps_rank below), not our launch shape.
static inline int ref_block_threads(int n) {
    int p = 1;
    while (p * 2 <= n && p < 1024) p *= 2;
    return p;
}

// ---- numerics that decide bit-exactness ---------------------------------------------------------
// The reference's nvcc build contracts  dx*dx + dy*dy + dz*dz  into
//     FMUL t = dy*dy ; FFMA t = dx*dx + t ; FFMA d = dz*dz + t
// in all four distance kernels (sampling_gpu.cu:133, ball_query_gpu.cu:33,95, interpolate_gpu.cu:43;
// verified on the SASS of the objects rebuilt for sm_100a).  Spelled with explicit intrinsics so no
// compiler flag can change it.  (a - b) per component, a = first argument.
__device__ __forceinline__ float sqdist3(float ax, float ay, float az, float bx, float by, float bz) {
    const float dx = __fsub_rn(ax, bx);
    const float dy = __fsub_rn(ay, by);
    const float dz = __fsub_rn(az, bz);
    return __fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy)));
}

// FPS arg-max tie-break.  The reference block (S = ref_block_threads(n) threads) lets thread t scan
// k = t, t+S, ... keeping the FIRST strict maximum and then merges (t, t+h), h = S/2..1, keeping the
// left entry unless the right is strictly greater (sampling_gpu.cu:86-91,119-207).  Among points
// that tie on the maximum the winner therefore minimises (bit_reverse_{log2 S}(k mod S), k), a pure
// function of k:  rank(k) = brev(k & (S-1)) | (k >> log2 S)   (brev puts the reversed low bits on top).
__device__ __forceinline__ uint32_t fps_rank(uint32_t k, uint32_t s_mask, uint32_t s_log2) {
    return __brev(k & s_mask) | (k >> s_log2);
}
// The inverse of fps_rank: the point index k whose rank is `rank`.  s_log2 == 0 (S = 1) keeps every bit of the rank; the
// general mask would shift by 32, which is undefined.
__device__ __forceinline__ uint32_t fps_unrank(uint32_t rank, uint32_t s_mask, uint32_t s_log2) {
    const uint32_t low_mask = s_log2 ? ((1u << (32u - s_log2)) - 1u) : 0xFFFFFFFFu;
    return (__brev(rank) & s_mask) | ((rank & low_mask) << s_log2);
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

// ---- thread-block clusters (fps.cu, topk.cu) ------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t cluster_nctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// the shared::cluster address of the variable at shared::cta address `local_addr` in CTA `cta` of this cluster
__device__ __forceinline__ uint32_t cluster_map_shared(uint32_t local_addr, uint32_t cta) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(cta));
    return r;
}

// What launch_cluster has set up or learned for one kernel, per device.  Each cluster kernel owns one, as a static beside
// its launch: two kernels of the same function type (e.g. a kernel with and without its profiling counters) must not share
// it, or the second would never get its shared-memory attribute.
struct ClusterKernelState {
    SmemAttrOnce smem;
    signed char schedulable[64] = {};   // csize > 8: 0 = not asked yet, 1 = yes, -1 = no
};
// launch_cluster's result when the device cannot co-schedule a cluster of that size of that kernel.  It is no CUDA error
// and sets no message: each caller decides what to do instead.  Distinct from SPSK_OK and every SPSK_ERR_* code.
constexpr int SPSK_CLUSTER_UNSCHEDULABLE = 1;

// Launches `kern` on nclusters clusters of csize CTAs (along x) with `smem` bytes of dynamic shared memory each.  Clusters of
// more than 8 CTAs are a non-portable size: the kernel opts in and the device is asked once whether it can co-schedule one.
// The answer cannot change for a (kernel, device, cluster shape), and both callers use a single size above 8 (16), so it is
// cached per (kernel, device) and never asked again, e.g. inside a CUDA-graph capture.
template <typename... KArgs, typename... Args>
static int launch_cluster(ClusterKernelState &state, void (*kern)(KArgs...), const char *name, int nclusters, int csize,
                          int threads, size_t smem, cudaStream_t st, Args... args) {
    if (int rc = state.smem.ensure(reinterpret_cast<const void *>(kern), (int)smem, name)) return rc;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(nclusters * csize));
    cfg.blockDim = dim3((unsigned)threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)csize;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (csize > 8) {
        signed char &ok = state.schedulable[device_slot()];
        if (ok == 0) {
            int clusters = 0;
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
            if (e == cudaSuccess) e = cudaOccupancyMaxActiveClusters(&clusters, kern, &cfg);
            if (e != cudaSuccess) (void)cudaGetLastError();
            ok = e == cudaSuccess && clusters >= 1 ? 1 : -1;
        }
        if (ok < 0) return SPSK_CLUSTER_UNSCHEDULABLE;
    }
    cudaError_t e = cudaLaunchKernelEx(&cfg, kern, args...);
    if (e != cudaSuccess) return cuda_fail(e, name);
    SPSK_LAUNCH_CHECK(name);
    return SPSK_OK;
}

}  // namespace spsk
