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

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device attribute: set it once per (kernel, device).
struct SmemAttrOnce {
    bool done[64] = {};
    int ensure(const void *func, int bytes, const char *what) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
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

}  // namespace spsk
