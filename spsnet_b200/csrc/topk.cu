// topk.cu -- score-based down-sampling (IA-SSD ctr/cls-aware, SPSNet stability-aware) in one launch.
//
// Replaces the torch-op chains of PointnetSAModuleMSG_WithSampling.forward:
//   ctr/cls-aware (pointnet2_modules.py:287-291):  max(dim=-1) -> sigmoid -> topk(npoint) -> .int()
//   'ss'/'sss'   (pointnet2_modules.py:293-303):   sigmoid(max cls) * (1 - sigmoid(stds/8 - 3)) -> topk -> .int()
// (4 resp. ~8 tiny kernels + a radix-select/sort in torch.topk).  Scores are computed with the same fp32
// op sequence torch uses (each torch op rounds once: mul by 1/8 is exact, sub, sigmoid = 1/(1+expf(-x))
// with IEEE add/div, rsub, mul), packed as (score_bits, ~index) 64-bit keys and sorted descending by a
// bitonic network in shared memory; the first npoint keys are the answer.  Order: descending score, ties
// by ascending point index (torch.topk leaves tie order unspecified; see DESIGN.md "top-k parity").
//
// n <= 16384: one CTA per scene sorts the whole scene in its shared memory (score_topk_kernel).
// 16384 < n <= 262144: one thread-block cluster of n_pad / 16384 = 2, 4, 8 or 16 CTAs per scene runs the
// same network over the cluster's distributed shared memory (score_topk_cluster_kernel).
#include "common.cuh"

namespace spsk {

constexpr int TOPK_THREADS = 1024;
constexpr int TOPK_CTA_KEYS = 16384;   // keys per CTA of the cluster kernel: 128 KB of shared memory

__device__ __forceinline__ float sigmoid_like_torch(float x) {
    // ATen sigmoid (CUDA): one / (one + std::exp(-a)) in fp32
    return __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-x)));
}

// Sort key of point i of a scene (cb: its cls rows, sb: its stds or nullptr): score bits above ~i, so that a
// descending sort orders by score, then by ascending index.  The low word of a real key is never 0, so the
// padding key 0 sorts last.  Both kernels use this function: their results cannot drift apart.
__device__ __forceinline__ unsigned long long score_key(const float *__restrict__ cb, const float *__restrict__ sb,
                                                        int num_class, int i) {
    float mx = __ldg(cb + (size_t)i * num_class);
    for (int c = 1; c < num_class; ++c) {   // torch.max propagates NaN (fmaxf would drop it); a NaN score sorts first, as in torch.topk
        const float v = __ldg(cb + (size_t)i * num_class + c);
        mx = (v != v || v > mx) ? v : mx;
    }
    float score = sigmoid_like_torch(mx);
    if (sb) {
        const float t = __fsub_rn(__fmul_rn(__ldg(sb + i), 0.125f), 3.0f);
        const float sta = __fsub_rn(1.0f, sigmoid_like_torch(t));
        score = __fmul_rn(score, sta);
    }
    return ((unsigned long long)__float_as_uint(score) << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)i);
}

__device__ __forceinline__ void write_pick(unsigned long long key, int *idx, float *scores, size_t at) {
    idx[at] = (int)(0xFFFFFFFFu - (uint32_t)(key & 0xFFFFFFFFull));
    if (scores) scores[at] = __uint_as_float((uint32_t)(key >> 32));
}

__global__ void __launch_bounds__(TOPK_THREADS, 1)
score_topk_kernel(int n, int n_pad, int num_class, int npoint, const float *__restrict__ cls,
                  const float *__restrict__ stds, int *__restrict__ idx, float *__restrict__ scores) {
    extern __shared__ unsigned long long keys[];
    const int b = blockIdx.x;
    const float *cb = cls + (size_t)b * n * num_class;
    const float *sb = stds ? stds + (size_t)b * n : nullptr;
    for (int i = threadIdx.x; i < n_pad; i += TOPK_THREADS) keys[i] = i < n ? score_key(cb, sb, num_class, i) : 0ull;
    __syncthreads();
    for (int k = 2; k <= n_pad; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n_pad; i += TOPK_THREADS) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const unsigned long long a = keys[i], c = keys[ixj];
                    const bool desc = (i & k) == 0;
                    if (desc ? (a < c) : (a > c)) { keys[i] = c; keys[ixj] = a; }
                }
            }
            __syncthreads();
        }
    }
    for (int j = threadIdx.x; j < npoint; j += TOPK_THREADS) write_pick(keys[j], idx, scores, (size_t)b * npoint + j);
}

// One cluster of csize = n_pad / TOPK_CTA_KEYS CTAs per scene.  The bitonic network runs over the sort positions
// 0..n_pad-1; CTA r holds positions [r * TOPK_CTA_KEYS, (r + 1) * TOPK_CTA_KEYS) in its shared memory.
//  - steps with j < TOPK_CTA_KEYS pair positions of the same CTA: a local compare-exchange, as in score_topk_kernel;
//  - steps with j >= TOPK_CTA_KEYS pair CTA r with CTA r ^ (j / TOPK_CTA_KEYS), slot for slot: every thread reads the
//    partner's key over distributed shared memory and keeps the max or the min for its own slot.  All reads of the
//    cluster happen between two cluster barriers, and every CTA writes only its own keys after the second one.
// At n_pad = 262144 that is 10 cluster steps of 171.
__global__ void __launch_bounds__(TOPK_THREADS, 1)
score_topk_cluster_kernel(int n, int n_pad, int num_class, int npoint, const float *__restrict__ cls,
                          const float *__restrict__ stds, int *__restrict__ idx, float *__restrict__ scores) {
    constexpr int PER_THREAD = TOPK_CTA_KEYS / TOPK_THREADS;
    extern __shared__ unsigned long long keys[];
    const uint32_t crank = cluster_ctarank();
    const int b = blockIdx.x / (int)cluster_nctarank();
    const int base = (int)crank * TOPK_CTA_KEYS;   // sort position of keys[0]
    const float *cb = cls + (size_t)b * n * num_class;
    const float *sb = stds ? stds + (size_t)b * n : nullptr;
    for (int i = threadIdx.x; i < TOPK_CTA_KEYS; i += TOPK_THREADS)
        keys[i] = base + i < n ? score_key(cb, sb, num_class, base + i) : 0ull;
    __syncthreads();
    const uint32_t keys_addr = (uint32_t)__cvta_generic_to_shared(keys);
    for (int k = 2; k <= n_pad; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            if (j >= TOPK_CTA_KEYS) {
                const uint32_t remote = cluster_map_shared(keys_addr, crank ^ (uint32_t)(j / TOPK_CTA_KEYS));
                // k > j: the whole CTA merges in one direction; the lower CTA of the pair keeps the max in a descending merge
                const bool keep_max = ((base & j) == 0) == ((base & k) == 0);
                unsigned long long v[PER_THREAD];
                cluster_sync_all();   // the partner has finished (and published) the previous step
#pragma unroll
                for (int s = 0; s < PER_THREAD; ++s) {
                    const int i = threadIdx.x + s * TOPK_THREADS;
                    unsigned long long c;
                    asm volatile("ld.shared::cluster.u64 %0, [%1];" : "=l"(c) : "r"(remote + 8u * (uint32_t)i));
                    const unsigned long long a = keys[i];
                    v[s] = keep_max ? (a > c ? a : c) : (a < c ? a : c);
                }
                cluster_sync_all();   // no CTA overwrites a key before every CTA has read it
#pragma unroll
                for (int s = 0; s < PER_THREAD; ++s) keys[threadIdx.x + s * TOPK_THREADS] = v[s];
            } else {
                // pair p -> positions (i, i + j) with bit j of i clear: every thread has work on every step
                for (int p = threadIdx.x; p < TOPK_CTA_KEYS / 2; p += TOPK_THREADS) {
                    const int i = ((p & ~(j - 1)) << 1) | (p & (j - 1));
                    const unsigned long long a = keys[i], c = keys[i + j];
                    const bool desc = ((base + i) & k) == 0;
                    if (desc ? (a < c) : (a > c)) { keys[i] = c; keys[i + j] = a; }
                }
            }
            __syncthreads();
        }
    }
    // no DSMEM access follows the last cluster step's second barrier, so a CTA may leave without a final cluster barrier
    for (int i = threadIdx.x; i < TOPK_CTA_KEYS && base + i < npoint; i += TOPK_THREADS)
        write_pick(keys[i], idx, scores, (size_t)b * npoint + base + i);
}

static int launch_score_topk_cluster(int b, int n, int n_pad, int num_class, int npoint, const float *cls, const float *stds,
                                     int *idx, float *scores, cudaStream_t st) {
    const int csize = n_pad / TOPK_CTA_KEYS;
    const size_t smem = sizeof(unsigned long long) * TOPK_CTA_KEYS;
    auto kern = score_topk_cluster_kernel;
    static SmemAttrOnce attr;
    if (int rc = attr.ensure(reinterpret_cast<const void *>(kern), (int)smem, "cudaFuncSetAttribute(score_topk_cluster_kernel)")) return rc;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(b * csize));
    cfg.blockDim = dim3(TOPK_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute cl[1];
    cl[0].id = cudaLaunchAttributeClusterDimension;
    cl[0].val.clusterDim.x = (unsigned)csize;
    cl[0].val.clusterDim.y = 1;
    cl[0].val.clusterDim.z = 1;
    cfg.attrs = cl;
    cfg.numAttrs = 1;
    if (csize > 8) {
        // 16-CTA clusters are a non-portable size: opt in, and make sure this device can co-schedule one.  The answer cannot
        // change for a (kernel, device), so it is asked once per device (and never again inside a CUDA-graph capture).
        static signed char schedulable[64] = {};   // 0 = not asked yet, 1 = yes, -1 = no
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
        if (schedulable[dev] == 0) {
            int nclusters = 0;
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
            if (e == cudaSuccess) e = cudaOccupancyMaxActiveClusters(&nclusters, kern, &cfg);
            if (e != cudaSuccess) (void)cudaGetLastError();
            schedulable[dev] = e == cudaSuccess && nclusters >= 1 ? 1 : -1;
        }
        if (schedulable[dev] < 0) {
            set_error("score_topk: n=%d needs a 16-CTA cluster of %zu-byte CTAs, which this device cannot schedule", n, smem);
            return SPSK_ERR_UNSUPPORTED;
        }
    }
    cudaError_t e = cudaLaunchKernelEx(&cfg, kern, n, n_pad, num_class, npoint, cls, stds, idx, scores);
    if (e != cudaSuccess) return cuda_fail(e, "cudaLaunchKernelEx(score_topk_cluster_kernel)");
    SPSK_LAUNCH_CHECK("score_topk_cluster_kernel");
    return SPSK_OK;
}

}  // namespace spsk

extern "C" int spsk_score_topk(int b, int n, int num_class, int npoint, const float *cls, const float *stds,
                               int *idx, float *scores, spsk_stream_t stream) {
    using namespace spsk;
    SPSK_REQUIRE(b >= 0 && n >= 1 && num_class >= 1 && npoint >= 0, SPSK_ERR_INVALID_ARG,
                 "score_topk: bad sizes b=%d n=%d num_class=%d npoint=%d", b, n, num_class, npoint);
    SPSK_REQUIRE(npoint <= n, SPSK_ERR_INVALID_ARG, "score_topk: npoint=%d > n=%d", npoint, n);
    SPSK_REQUIRE(n <= SPSK_TOPK_MAX_N, SPSK_ERR_UNSUPPORTED, "score_topk: n=%d > %d", n, SPSK_TOPK_MAX_N);
    if (b == 0 || npoint == 0) return SPSK_OK;
    SPSK_REQUIRE(cls && idx, SPSK_ERR_INVALID_ARG, "score_topk: null pointer");
    int n_pad = 2;
    while (n_pad < n) n_pad <<= 1;
    if (n_pad > TOPK_CTA_KEYS) return launch_score_topk_cluster(b, n, n_pad, num_class, npoint, cls, stds, idx, scores, as_stream(stream));
    const size_t smem = sizeof(unsigned long long) * (size_t)n_pad;
    if (smem + 2048 > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(score_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(score_topk_kernel)");
    }
    score_topk_kernel<<<b, TOPK_THREADS, smem, as_stream(stream)>>>(n, n_pad, num_class, npoint, cls, stds, idx, scores);
    SPSK_LAUNCH_CHECK("score_topk_kernel");
    return SPSK_OK;
}
