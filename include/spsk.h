/*
 * spsk.h -- C-ABI of the B200-native point-sampling + set-abstraction kernels (libspsk.so).
 *
 * This is the drop-in boundary for the hot path of AlanLiangC/SPSNet's
 * pcdet/ops/pointnet2/pointnet2_batch.  Every entry point is `extern "C"`, takes raw DEVICE
 * pointers, plain ints/floats and an explicit stream (a `cudaStream_t` passed as `void*`; NULL =
 * legacy default stream), returns 0 on success or a negative spsk_status, never allocates, never
 * synchronises and never calls exit().  No torch types appear in any signature.
 *
 * Section 1 mirrors, one to one, the 11 functions the reference binds through pybind11
 * (src/pointnet2_api.cpp:10-26): same argument order and meaning, tensors replaced by their
 * data pointers, plus the trailing stream.  INTEGRATION.md shows the ctypes / pybind stubs a
 * maintainer of the reference adds to route `pointnet2_utils.py` through these symbols.
 *
 * Section 2 holds the fused entry points that replace chains of torch ops of
 * `pointnet2_modules.py` (top-k samplers, MSG ball query, grouped shared-MLP + max-pool).
 *
 * Layouts (identical to the reference): xyz (B,N,3) f32, features (B,C,N) f32, indices int32,
 * everything contiguous.  All file:line citations are relative to the reference repository.
 */
#ifndef SPSK_H_
#define SPSK_H_

#ifdef __cplusplus
extern "C" {
#endif

typedef void *spsk_stream_t; /* cudaStream_t */

#if defined(__GNUC__)
#define SPSK_API __attribute__((visibility("default")))
#else
#define SPSK_API
#endif

typedef enum spsk_status {
    SPSK_OK = 0,
    SPSK_ERR_INVALID_ARG = -1, /* null pointer, negative size, nsample/npoint out of range */
    SPSK_ERR_UNSUPPORTED = -2, /* shape outside what the kernels are built for (see message) */
    SPSK_ERR_CUDA = -3,        /* launch failed; spsk_last_error() has cudaGetErrorString */
    SPSK_ERR_WORKSPACE = -4    /* caller-provided workspace too small */
} spsk_status;

/* Human-readable description of the last error raised on the calling thread. */
SPSK_API const char *spsk_last_error(void);
/* ABI version of this header (bumped on any signature change or added entry point; currently 5). */
SPSK_API int spsk_abi_version(void);
/* Number of CUDA kernels this library has launched in this process (all threads). */
SPSK_API unsigned long long spsk_launch_count(void);
/* Compute capability the library was compiled for (100 => sm_100a). */
SPSK_API int spsk_built_for_sm(void);

/* ------------------------------------------------------------------------------------------------
 * Section 1 -- the reference's 11 native ops
 * ---------------------------------------------------------------------------------------------- */

/* D-FPS.  Replaces farthest_point_sampling_wrapper (src/sampling.cpp:34-43 ->
 * src/sampling_gpu.cu:93-253).  xyz (b,n,3); idx (b,m) out; idx[:,0] = 0.
 * temp (b,n): the reference's running-min scratch, pre-filled by the caller (1e10,
 * pointnet2_utils.py:26).  If non-NULL its contents are honoured on input and the final minima are
 * written back, exactly like the reference.  NULL means "all 1e10" and nothing is written (the
 * running minima live in registers).  Bit-exact indices incl. the block-tree tie-break. */
SPSK_API int spsk_farthest_point_sampling(int b, int n, int m, const float *xyz, float *temp, int *idx,
                                 spsk_stream_t stream);

/* Tuning aid: with a non-NULL `counters` (6 x u64 device words, zeroed by the caller) the pruned D-FPS kernel adds, summed
 * over scenes, warp 0's cycles in [query + bound, sub-bucket updates, warp arg-max, barrier wait, block arg-max] and the
 * number of 32-point sub-buckets visited by all warps. */
SPSK_API int spsk_fps_set_profile(unsigned long long *counters);

/* F-FPS over a precomputed (b,n,n) distance matrix.  Replaces
 * furthest_point_sampling_with_dist_wrapper (src/sampling.cpp:46-56 -> src/sampling_gpu.cu:256-416).
 * Offsets are 64-bit here (the reference overflows int32 for b*n*n >= 2^31). */
SPSK_API int spsk_furthest_point_sampling_with_dist(int b, int n, int m, const float *dist, float *temp,
                                           int *idx, spsk_stream_t stream);

/* out[b,c,j] = points[b,c,idx[b,j]].  Replaces gather_points_wrapper (src/sampling.cpp:11-20 ->
 * src/sampling_gpu.cu:8-44).  points (b,c,n), idx (b,npoints), out (b,c,npoints). */
SPSK_API int spsk_gather_points(int b, int c, int n, int npoints, const float *points, const int *idx,
                       float *out, spsk_stream_t stream);

/* grad_points[b,c,idx[b,j]] += grad_out[b,c,j] (grad_points pre-zeroed by the caller).  Replaces
 * gather_points_grad_wrapper (src/sampling.cpp:22-32 -> src/sampling_gpu.cu:46-84). */
SPSK_API int spsk_gather_points_grad(int b, int c, int n, int npoints, const float *grad_out, const int *idx,
                            float *grad_points, spsk_stream_t stream);

/* First `nsample` neighbours (index order) with d2 < radius^2; first-hit padding; rows of centres
 * with no neighbour are left untouched (caller pre-zeroes, pointnet2_utils.py:246).  Replaces
 * ball_query_wrapper (src/ball_query.cpp:32-42 -> src/ball_query_gpu.cu:9-67).
 * new_xyz (b,m,3), xyz (b,n,3), idx (b,m,nsample). */
SPSK_API int spsk_ball_query(int b, int n, int m, float radius, int nsample, const float *new_xyz,
                    const float *xyz, int *idx, spsk_stream_t stream);

/* Shell query min_radius^2 <= d2 < max_radius^2 plus the d2 == 0 clause (a coincident point is
 * inserted twice when min_radius == 0, as in the reference).  Replaces ball_query_dilated_wrapper
 * (src/ball_query.cpp:45-56 -> src/ball_query_gpu.cu:70-137). */
SPSK_API int spsk_ball_query_dilated(int b, int n, int m, float max_radius, float min_radius, int nsample,
                            const float *new_xyz, const float *xyz, int *idx, spsk_stream_t stream);

/* out[b,c,p,s] = points[b,c,idx[b,p,s]].  Replaces group_points_wrapper (src/group_points.cpp:30-40
 * -> src/group_points_gpu.cu:53-92). */
SPSK_API int spsk_group_points(int b, int c, int n, int npoints, int nsample, const float *points,
                      const int *idx, float *out, spsk_stream_t stream);

/* Scatter-add backward of group_points.  Replaces group_points_grad_wrapper
 * (src/group_points.cpp:18-28 -> src/group_points_gpu.cu:14-50). */
SPSK_API int spsk_group_points_grad(int b, int c, int n, int npoints, int nsample, const float *grad_out,
                           const int *idx, float *grad_points, spsk_stream_t stream);

/* Three nearest known points of every unknown point: squared distances (the python layer takes the
 * sqrt) and indices, first index wins ties.  Replaces three_nn_wrapper (src/interpolate.cpp:21-30
 * -> src/interpolate_gpu.cu:16-81).  unknown (b,n,3), known (b,m,3), dist2/idx (b,n,3). */
SPSK_API int spsk_three_nn(int b, int n, int m, const float *unknown, const float *known, float *dist2,
                  int *idx, spsk_stream_t stream);

/* out[b,c,j] = sum_i weight[b,j,i] * points[b,c,idx[b,j,i]] with the reference build's rounding
 * order.  Replaces three_interpolate_wrapper (src/interpolate.cpp:32-44 ->
 * src/interpolate_gpu.cu:84-124).  points (b,c,m), idx/weight (b,n,3), out (b,c,n). */
SPSK_API int spsk_three_interpolate(int b, int c, int m, int n, const float *points, const int *idx,
                           const float *weight, float *out, spsk_stream_t stream);

/* Backward of three_interpolate (grad_points pre-zeroed).  Replaces three_interpolate_grad_wrapper
 * (src/interpolate.cpp:46-58 -> src/interpolate_gpu.cu:127-169). */
SPSK_API int spsk_three_interpolate_grad(int b, int c, int n, int m, const float *grad_out, const int *idx,
                                const float *weight, float *grad_points, spsk_stream_t stream);

/* Atomic-free, bit-reproducible form of the three backward scatters above (SURVEY.md 8f rank 4): a stable sort of the
 * (scene, target) keys followed by a segment reduction in ascending entry order (csrc/scatter_grad.cu).
 *   grad_points[b, ch, idx[b, l]] += weight[b, l] * grad_out[b, ch, l / div]      l = 0 .. l_per_scene-1
 * gather: l_per_scene = npoints, div = 1, weight = NULL; group: l_per_scene = npoints * nsample, div = 1, weight = NULL;
 * three_interpolate: l_per_scene = 3 n, div = 3, weight = the (b, n, 3) weights.  grad_out (b, c, cols) with
 * cols >= ceil(l_per_scene / div); grad_points (b, c, n) is fully written (no pre-zeroing needed). */
SPSK_API long long spsk_scatter_grad_workspace_bytes(int b, int n, long long l_per_scene);
SPSK_API int spsk_scatter_grad(int b, int c, int n, long long l_per_scene, int cols, int div, const float *grad_out,
                               const int *idx, const float *weight, float *grad_points, void *workspace,
                               long long workspace_bytes, spsk_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Section 2 -- fused replacements for torch-op chains in pointnet2_modules.py
 * ---------------------------------------------------------------------------------------------- */

/* Score-based down-sampling: one launch replaces max -> sigmoid -> topk -> int() (IA-SSD ctr/cls-aware,
 * pointnet2_modules.py:287-291) and, when stds != NULL, SPSNet's stability-weighted variant
 * score = sigmoid(max_c cls) * (1 - sigmoid(stds/8 - 3)) (pointnet2_modules.py:293-303).
 * cls (b,n,num_class) f32; stds (b,n) f32 or NULL; idx (b,npoint) out, ordered by descending score,
 * ties broken by ascending point index; scores (b,npoint) out or NULL (the picked scores).
 * n <= SPSK_TOPK_MAX_N, in one launch and without workspace: n <= 16384 sorts each scene in one CTA's shared
 * memory; 16384 < n <= 262144 sorts it across a thread-block cluster of ceil_pow2(n) / 16384 CTAs (2, 4, 8 or
 * 16; 128 KB of shared memory each).  A 16-CTA cluster (n > 131072) is a non-portable size: a device that
 * cannot schedule one returns SPSK_ERR_UNSUPPORTED. */
#define SPSK_TOPK_MAX_N 262144
SPSK_API int spsk_score_topk(int b, int n, int num_class, int npoint, const float *cls, const float *stds,
                    int *idx, float *scores, spsk_stream_t stream);

/* Point-major row gather: out[b,j,:] = in[b,idx[b,j],:], in (b,n,c), out (b,m,c).  With c = 3 this is
 * new_xyz = xyz[sample_idx], replacing transpose -> gather_operation -> transpose -> contiguous
 * (pointnet2_modules.py:261,424). */
SPSK_API int spsk_gather_rows(int b, int n, int m, int c, const float *in, const int *idx, float *out,
                     spsk_stream_t stream);

/* Multi-scale ball query: ONE scan of xyz per centre answers up to SPSK_MAX_SCALES radii
 * (replaces the per-scale ball_query calls of QueryAndGroup.forward, pointnet2_utils.py:307, inside
 * the MSG loop pointnet2_modules.py:429-431).  idx[s] is (b,m,nsample[s]); unlike spsk_ball_query
 * empty rows ARE written (zeros), so no memset is needed.  Results identical to nscales separate
 * spsk_ball_query calls on zero-filled outputs. */
#define SPSK_MAX_SCALES 4
SPSK_API int spsk_ball_query_msg(int b, int n, int m, int nscales, const float *radius, const int *nsample,
                        const float *new_xyz, const float *xyz, int *const *idx, spsk_stream_t stream);

/* Same contract and results as spsk_ball_query_msg, computed through a per-scene uniform xy grid (cells of
 * edge >= 1.01 * max radius, 3 x 3 neighbourhood per centre, hits ordered through a per-warp index bitmap):
 * the work drops from n to a few dozen pair tests per centre when the radius is small against the scene.
 * `workspace` is caller-owned device scratch of at least spsk_ball_query_grid_workspace_bytes(b, n) bytes.
 * n <= SPSK_BQ_GRID_MAX_N (SPSK_ERR_UNSUPPORTED above): the grid is built per window of 65536 point ids and the
 * query walks windows of 65536 ids (32768 with four scales) in increasing id order until every scale is full. */
#define SPSK_BQ_GRID_MAX_N 262144
SPSK_API long long spsk_ball_query_grid_workspace_bytes(int b, int n);
SPSK_API int spsk_ball_query_msg_grid(int b, int n, int m, int nscales, const float *radius, const int *nsample,
                             const float *new_xyz, const float *xyz, int *const *idx, void *workspace,
                             long long workspace_bytes, spsk_stream_t stream);

/* One shared-MLP layer over grouped rows, the unit the SA layer is built from (replaces
 * grouping_operation x2 + subtract + cat + Conv2d1x1 + BatchNorm2d(eval) + ReLU [+ max_pool2d],
 * pointnet2_utils.py:307-315 and pointnet2_modules.py:204-211,431-436).
 *
 *   rows r = (b, p, s), p < m centres, s < nsample.
 *   input row  (gather != 0): [xyz[b,idx]-new_xyz[b,p] (3, if use_xyz), features[b,:,idx] (c_feat)]
 *   input row  (gather == 0): in_rows[r, 0:c_in]                    (row-major workspace)
 *   y[r, co] = relu?( bias[co] + sum_k in[r,k] * wt[k, co] )         wt is (c_in, c_out) = W^T, BN folded
 *   pool == 0: out_rows[r, 0:c_out]                                  (row-major workspace)
 *   pool == 1: out_pooled[b, co_off + co, p] = max_s y  (relu must be on; out_pooled pre-zeroed,
 *              (b, c_total, m) layout = the reference's new_features)
 *   pool == 2: avg over s (pool_method 'avg_pool'), out_pooled pre-zeroed.
 */
typedef struct spsk_group_desc {
    int b, n, m, nsample;  /* scenes, source points, centres, neighbours per centre            */
    int c_feat;            /* feature channels gathered per neighbour (0 if features == NULL)  */
    int use_xyz;           /* prepend the 3 relative coordinates                               */
    const float *xyz;      /* (b,n,3)                                                          */
    const float *new_xyz;  /* (b,m,3)                                                          */
    const float *features; /* (b,c_feat,n) or NULL                                             */
    const int *idx;        /* (b,m,nsample)                                                    */
} spsk_group_desc;

SPSK_API int spsk_grouped_linear(const spsk_group_desc *g, int gather, const float *in_rows, int c_in,
                        const float *wt, const float *bias, int c_out, int relu, int pool,
                        float *out_rows, float *out_pooled, int c_total, int co_off,
                        spsk_stream_t stream);

/* Point-wise (1x1 Conv1d) layer on channel-major tensors, used for the aggregation / confidence /
 * vote MLPs (pointnet2_modules.py:216-243,449-455,485-500):
 *   out[b, co, p] = relu?( bias[co] + sum_k in[b, k, p] * wt[k, co] ),  in (b,c_in,m), out (b,c_out,m). */
SPSK_API int spsk_pointwise_linear(int b, int m, const float *in, int c_in, const float *wt, const float *bias,
                          int c_out, int relu, float *out, spsk_stream_t stream);

/* ---- tensor-core path (tcgen05 + TMEM) -------------------------------------------------------------
 * Point-major fp16 "twin" of a channel-major feature tensor: twin[b, i, 0:c] = (half)features[b, 0:c, i],
 * zero padded to cpad8 (multiple of 8) channels, so that gathering one neighbour is a run of 16-byte loads. */
SPSK_API int spsk_make_twin(int b, int c, int n, int cpad8, const float *features, void *twin, spsk_stream_t stream);

/* One MSG scale, fully fused on the tensor cores: gather (idx) -> [features | xyz - centre] -> nlayers x
 * (1x1 conv + folded BN + ReLU) -> max over nsample   (replaces QueryAndGroup.forward's grouping + cat and the
 * shared MLP + max_pool2d, pointnet2_utils.py:307-315, pointnet2_modules.py:204-211,431-436).
 * fp16 operands / fp32 accumulation; `split` selects hi+lo fp16 operands (3 products, fp32-grade) for narrow chains.
 *
 *   layer l   : input width kpad[l] (multiple of 16), output width cpad[l] (multiple of 16; last layer: multiple
 *               of 128), cpad[l] == kpad[l+1].  Plain mode: kpad[0] >= ceil8(c_feat) + 8*use_xyz with k order
 *               [features (ceil8(c_feat)), x, y, z, 0...].  Split mode: kpad[0] == 16, k order [f0..f7, x, y, z, 0...]
 *               (c_feat <= 8; xyz first when c_feat == 0), every width <= 64.
 *   wtiles    : per layer (layers concatenated) the matrix W'[wk, cpad] (wk = kpad, or 2*kpad = [Wh; Wl] rows in
 *               split mode -- the kernel runs 3*kpad of K per tile, Xh.Wh + Xl.Wh + Xh.Wl, reading the Wh rows twice)
 *               cut into tiles of (<=128 couts) x (<=64 k), ordered cout-chunk major then k, each tile
 *               `ncols x kw` fp16 in the canonical K-major no-swizzle UMMA layout
 *               byte(r, k) = (r/8)*(kw*16) + (k/8)*128 + (r%8)*16 + (k%8)*2;  zero padded
 *   bias      : folded BN shift, layers concatenated, cpad[l] floats each (zero padded)
 *   outputs   : out_cm[b, co_off + c, p] fp32 (the reference's new_features layout, (b, c_total, m)) and / or
 *               out16[(b*m + p) * ld16 + co16 + c] fp16 point-major for c < n16 (columns cout_last..n16 get zeros)
 *   nsample must be a power of two <= 128. */
typedef struct spsk_sa_mma_desc {
    int b, n, m, nsample;
    const float *xyz;       /* (b,n,3) */
    const float *new_xyz;   /* (b,m,3) */
    const int *idx;         /* (b,m,nsample) */
    int use_xyz;
    int c_feat;
    const void *twin;       /* (b,n,ldtwin) fp16 point-major features (plain mode), NULL if c_feat == 0 */
    int ldtwin;             /* multiple of 8, >= ceil8(c_feat) */
    const float *features;  /* (b,c_feat,n) fp32 (split mode) */
    int split;
    int nlayers;
    int kpad[4], cpad[4];
    const void *wtiles;
    const float *bias;
    int cout_last;
    float *out_cm; int c_total, co_off;
    void *out16; int ld16, co16, n16;
    int o16lo;              /* > 0: out16 also receives the residuals fp16(y - fp16(y)) at column o16lo + co16 + c */
    int l0_fused;           /* 1 (split chains, >= 2 layers, cpad[0] <= 32): layer 0 is evaluated in fp32 by the gather threads;
                               wtiles then carries, after the last layer's tiles, W0 as [16][cpad[0]] fp32 (same row order as
                               the split k order) followed by cpad[0] fp32 biases */
    int pair;               /* 1: CTA-pair kernel (tcgen05 cta_group::2, 256-row tiles) for wide chains: plain mode only, last cpad a
                               multiple of 256, and wtiles in the PAIR packing: per layer, 256-wide cout chunks; inside a chunk
                               the rows of pair rank 0 then rank 1 (hidden layers: half of the chunk each; last layer: 128
                               couts each), each as tiles of <= 64 k in the canonical layout */
    int ovf_tag;            /* fp16 range guard: bit (ovf_tag & 31) of the per-device overflow word is set when a hidden activation or
                               an fp16 output of this call exceeds 65504 (see spsk_fp16_overflow_poll); appended in ABI 3 */
    double *stats;          /* non-NULL: BATCH-STATISTICS pass of training-mode BatchNorm (reference pointnet2_modules.py:203-211 with
                               the module in train()): the chain is evaluated as usual, but the last layer's epilogue, instead of bias
                               + ReLU + max-pool, adds the raw accumulators z[row, c] of every real row into per-CTA partial sums
                               stats[(part * cpad_last + c) * 2 + {0, 1}] += {sum z, sum z*z}   (fp32 inside a 128-row tile, fp64
                               across tiles; each (part, c) cell is owned by ONE thread: no atomics, bit-reproducible).  The call
                               zeroes the slices it accumulates into (stream-ordered memset); the caller sums them over `part` and
                               divides by b*m*nsample; out_cm / out16 are not written
                               and may be NULL.  Plain launch shapes only (pair == 0).  Appended in ABI 4 */
    int stats_parts;        /* capacity of `stats` in parts; must be >= spsk_sa_mma_stats_parts() of this descriptor */
} spsk_sa_mma_desc;

/* Launch shape the library picks for a chain (only nlayers / kpad / cpad / split are read): dynamic shared memory,
 * co-resident CTAs per SM, weight-ring depth, and whether the packed chain stays resident in shared memory.
 * SPSK_ERR_UNSUPPORTED when the chain does not fit. */
SPSK_API int spsk_sa_mma_config(const spsk_sa_mma_desc *d, int *smem_bytes, int *ctas_per_sm, int *nstages, int *resident);
SPSK_API int spsk_sa_mma_forward(const spsk_sa_mma_desc *d, spsk_stream_t stream);
/* Host-only test / documentation aid: the static per-tile schedule (weight-tile groups, ring slots, barriers, phase parities) a
 * streaming chain runs with; 8 uint32 per entry into `words` (capacity 8 * SPSK_SA_SCHED_MAX), layout in csrc/sa_mma.cu.
 * info[6] = {hidden-ring stages, overlay-ring stages, resident, smem offset of the hidden ring, of the overlay ring, packed weight
 * bytes}.  *n = 0 when the chain does not use the table (resident, split or pair chains). */
#define SPSK_SA_SCHED_MAX 104
SPSK_API int spsk_sa_mma_schedule(const spsk_sa_mma_desc *d, int *n, unsigned int *words, int *info);
/* Number of partial-sum slices a statistics pass of this descriptor (sizes and chain filled in) writes: CTAs x epilogue groups. */
SPSK_API int spsk_sa_mma_stats_parts(const spsk_sa_mma_desc *d, int *nparts);
/* Tuning aid: when `counters` (device memory, SPSK_SA_PROF_COUNTERS x u64, zeroed by the caller) is non-NULL every
 * following spsk_sa_mma_forward adds the SM cycles its warp roles spent per wait / work category (order: mma total,
 * mma wait acc-empty, mma wait weights, mma wait activations, producer wait stage, producer wait hidden-done, epilogue
 * total, gather, wait hidden acc, hidden epilogue, wait pool acc, pool epilogue, mma issue, mma commit; summed over CTAs,
 * epilogue = thread 0). */
#define SPSK_SA_PROF_COUNTERS 14
SPSK_API int spsk_sa_mma_set_profile(unsigned long long *counters);

/* ---- training-mode BatchNorm around the statistics passes (spsk_sa_mma_desc.stats), reference pointnet2_modules.py:203-211 with
 * the module in train().  One training forward of an L-layer chain is, per layer l:
 *   spsk_sa_pack_layer(raw conv l as the LAST layer of the truncated chain) -> spsk_sa_mma_forward(stats) -> spsk_bn_stats_reduce
 *   [-> all-reduce of the 2c+1 doubles across ranks: SyncBatchNorm] -> spsk_bn_stats_finalize -> spsk_sa_pack_layer(conv l x scale)
 * and then one ordinary spsk_sa_mma_forward on the chain folded with the batch statistics. */

/* Pack one layer's weights for spsk_sa_mma_forward: w (cout, cin) fp32 row-major, the layout of Conv2d(1x1).weight; `scale`
 * (cout floats or NULL) multiplies row c (the BN fold); output = the layer's tiles of W'[wk, cpad] exactly as `wtiles` describes
 * them above (wk = kpad, or 2*kpad = [Wh; Wl] with split), zero padded, written at `wtiles` (the caller adds the layer's offset
 * wk * cpad * 2 bytes per preceding layer).  first != 0: layer 0, whose reference input order [x y z | features]
 * (pointnet2_utils.py:315) is permuted to the kernel's [features | x y z | 0] order; cin must equal c_feat + 3*use_xyz. */
SPSK_API int spsk_sa_pack_layer(const float *w, int cout, int cin, const float *scale, int first, int c_feat, int use_xyz, int kpad, int cpad,
                                int split, void *wtiles, spsk_stream_t stream);
/* parts (nparts, cpad, 2) fp64 of a statistics pass -> sums[2*ch + {0,1}] = {sum z, sum z*z} for ch < c, sums[2*c] = count
 * (2c + 1 doubles; summed in a fixed order: reproducible). */
SPSK_API int spsk_bn_stats_reduce(const double *parts, int nparts, int cpad, int c, double count, double *sums, spsk_stream_t stream);
/* sums (2c + 1 doubles, see above) -> mean, biased variance -> scale[ch] = gamma / sqrt(var + eps), bias[ch] = beta - mean * scale
 * (the BN fold for the following passes); running_mean / running_var (both or neither) get torch's update with `momentum`
 * (unbiased variance) unless momentum < 0; `moments` (c, 2) fp64 receives (mean, var) when non-NULL. */
SPSK_API int spsk_bn_stats_finalize(const double *sums, int c, const float *gamma, const float *beta, float eps, float momentum,
                                    float *running_mean, float *running_var, float *scale, float *bias, double *moments, spsk_stream_t stream);
/* Both steps in ONE launch, for statistics that stay on this rank (plain BatchNorm2d): parts -> (scale, bias), running statistics
 * updated (momentum < 0: not), *num_batches_tracked += 1 when non-NULL (torch's int64 counter), sums (2c + 1 doubles) written
 * when non-NULL. */
SPSK_API int spsk_bn_stats_reduce_finalize(const double *parts, int nparts, int cpad, int c, double count, const float *gamma, const float *beta,
                                           float eps, float momentum, float *running_mean, float *running_var, long long *num_batches_tracked,
                                           float *scale, float *bias, double *sums, spsk_stream_t stream);

/* Point-wise layer on the tensor cores:  y[row, c] = relu?( bias[c] + sum_k x[row, k] * W[c, k] )  over point-major
 * fp16 rows (replaces the aggregation / confidence / vote Conv1d + BN + ReLU stacks, pointnet2_modules.py:216-243,
 * 447-458, 485-500).
 *   x       : (rows, ldx) fp16, first k columns used (k multiple of 16; columns >= the true width must hold zeros)
 *   wtiles  : W (n x k) cut into 128-cout x 64-k tiles, cout-chunk major then k, each tile a full 16 KB block in the
 *             canonical K-major no-swizzle layout byte(r, kk) = (r/8)*1024 + (kk/8)*128 + (r%8)*16 + (kk%8)*2, zero
 *             padded; tiles must cover ceil128(max(n, n16)) couts
 *   bias    : ceil128(max(n, n16)) floats, zero padded
 *   outputs (any subset): out_cm[(row/m) , co_off + c, row%m] fp32 channel-major (b, c_total, m);
 *             out16[row*ld16 + c] fp16 for c < n16 (zeros above n); out_pm[row*ldpm + c] fp32 for c < n. */
typedef struct spsk_pw_desc {
    int rows, k, ldx, n, relu;
    int split;  /* 1: fp32-grade arithmetic on hi + lo fp16 halves: x rows hold hi in columns [0, k) and lo = fp16(v - hi) in
                   [xlo, xlo + k); wtiles hold, per (cout chunk, 64-wide k chunk), the Wh tile immediately followed by the Wl tile
                   (32 KB); y = xh.Wh + xl.Wh + xh.Wl */
    int xlo;
    const void *x;
    const void *wtiles;
    const float *bias;
    float *out_cm; int m, c_total, co_off;
    void *out16; int ld16, n16;
    int o16lo;  /* > 0: out16 also receives the residuals fp16(y - fp16(y)) at columns [o16lo, o16lo + n16) */
    float *out_pm; int ldpm;
    int ovf_tag;  /* fp16 range guard tag of this call (see spsk_sa_mma_desc.ovf_tag) */
} spsk_pw_desc;
SPSK_API int spsk_pw_mma_forward(const spsk_pw_desc *d, spsk_stream_t stream);

/* fp16 range guard.  The tensor-core path stores inter-layer activations as fp16 (largest finite value 65504) where the
 * reference's TF32 convolutions keep the fp32 exponent range (pointnet2_modules.py:203-211).  Every kernel that stores fp16
 * (spsk_sa_mma_forward, spsk_pw_mma_forward, spsk_make_twin) ORs bit (ovf_tag & 31) into a per-device word when a value it
 * stores exceeds that range.  This call SYNCHRONISES the device, returns the word and optionally clears it; the python
 * modules poll it after an eager forward and re-run the tagged modules on the exact-fp32 kernels (spsk_grouped_linear /
 * spsk_pointwise_linear), which have no range limit. */
SPSK_API int spsk_fp16_overflow_poll(unsigned int *mask, int clear);

/* ------------------------------------------------------------------------------------------------
 * Section 3 -- the consumer of the path (SURVEY.md §8f rank 3): rotated IoU / NMS and the fused
 * IA-SSD head post-processing.  Boxes are (N,7) f32 [x, y, z, dx, dy, dz, heading], contiguous.
 * ---------------------------------------------------------------------------------------------- */

/* ans_overlap[i,j] = area of the BEV intersection of boxes_a[i] and boxes_b[j].  Replaces boxes_overlap_bev_gpu
 * (pcdet/ops/iou3d_nms/src/iou3d_nms.cpp:48-67 -> src/iou3d_nms_kernel.cu:236-250). */
SPSK_API int spsk_boxes_overlap_bev(int num_a, const float *boxes_a, int num_b, const float *boxes_b,
                                    float *ans_overlap, spsk_stream_t stream);
/* ans_iou[i,j] = rotated BEV IoU.  Replaces boxes_iou_bev_gpu (src/iou3d_nms.cpp:69-88 ->
 * src/iou3d_nms_kernel.cu:251-265). */
SPSK_API int spsk_boxes_iou_bev(int num_a, const float *boxes_a, int num_b, const float *boxes_b, float *ans_iou,
                                spsk_stream_t stream);
/* ans_iou[i,j] = 3-D IoU (BEV overlap x height overlap over the union volume): one launch for the kernel + ~14
 * torch ops of boxes_iou3d_gpu (pcdet/ops/iou3d_nms/iou3d_nms_utils.py:48-81), same per-op fp32 rounding. */
SPSK_API int spsk_boxes_iou3d(int num_a, const float *boxes_a, int num_b, const float *boxes_b, float *ans_iou,
                              spsk_stream_t stream);

/* Greedy NMS over boxes already sorted by descending score, `batch` independent scenes per call.  Replaces nms_gpu
 * (normal = 0: rotated BEV IoU) and nms_normal_gpu (normal = 1: axis-aligned BEV IoU), src/iou3d_nms.cpp:90-188 ->
 * src/iou3d_nms_kernel.cu:267-365, INCLUDING the host-side suppression loop, which runs on the device here: the
 * call never allocates, never copies to the host and never synchronises.
 *   boxes (batch,n,7); counts (batch) device ints = boxes actually present per scene (NULL: all n);
 *   keep (batch,n) int64 out: positions (into the sorted order) of the surviving boxes, ascending;
 *   num_keep (batch) int32 out; workspace >= spsk_nms_workspace_bytes(batch,n) (the suppression bit mask). */
#define SPSK_NMS_MAX_N 32768
SPSK_API long long spsk_nms_workspace_bytes(int batch, int n);
SPSK_API int spsk_nms(int batch, int n, const float *boxes, const int *counts, float thresh, int normal,
                      long long *keep, int *num_keep, void *workspace, long long workspace_bytes,
                      spsk_stream_t stream);

/* IA-SSD head post-processing for a whole batch in 3 launches: per centre label = argmax class logit, score =
 * sigmoid(max logit), box = PointResidual_BinOri_Coder.decode_torch (pcdet/utils/box_coder_utils.py:279-319,
 * called from point_head_template.py:193-207); per scene score >= score_thresh -> top pre_max by score ->
 * rotated NMS -> first post_max survivors (detector3d_template.py:207-290 non-multi-class branch,
 * model_nms_utils.py:6-27).  Replaces ~40 torch ops + cudaMalloc + D2H mask copy + host loop PER SCENE.
 *   cls (batch*m, ld_cls) logits; reg (batch*m, ld_reg) box encodings (6 + 2*bin_size used);
 *   centers (batch*m, ld_centers): xyz of each centre (pass centers + 1 with ld 4 for [bs,x,y,z] rows);
 *   mean_size (num_class,3) device floats or NULL (use_mean_size = False);
 *   decoded, every row: box_preds (batch*m,7), scores (batch*m), labels (batch*m) int32 in 1..num_class;
 *   padded detections: out_boxes (batch,post_max,7), out_scores (batch,post_max), out_labels (batch,post_max)
 *   int64, out_index (batch,post_max) int64 = centre index within the scene (-1 padding), out_count (batch).
 * Optional parts: reg = NULL -> box_preds is an INPUT (already decoded boxes); cls = NULL -> labels is an input
 * (decode with given classes, = box_coder.decode_torch(enc, points, pred_classes)); out_boxes = NULL -> decode only
 * (one launch, no workspace needed). */
#define SPSK_DETECT_MAX_M 4096
typedef struct spsk_detect_desc {
    int batch, m, num_class, bin_size;
    const float *cls; int ld_cls;
    const float *reg; int ld_reg;
    const float *centers; int ld_centers;
    const float *mean_size;
    float score_thresh, nms_thresh;
    int nms_normal, pre_max, post_max;
    float *box_preds; float *scores; int *labels;
    float *out_boxes; float *out_scores; long long *out_labels; long long *out_index; int *out_count;
    void *workspace; long long workspace_bytes;
} spsk_detect_desc;
SPSK_API long long spsk_detect_workspace_bytes(int batch, int m);
SPSK_API int spsk_detect_postprocess(const spsk_detect_desc *d, spsk_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Section 4 -- SPSNet's surface-feature extractor (SURVEY.md §8f rank 4; USE_SURFACE: True in SPSNet.yaml:48):
 * one unit of FeatureExtraction = FCLayer transform + DenseEdgeConv with 3 FC layers, growth 12, max aggregation
 * (pcdet/ops/pointnet2/pointnet2_batch/surface_feature.py:45-115,118-187) in two launches.  The neighbour lists come
 * from spsk_ball_query (the reference calls QueryAndGroup(radius, knn, use_xyz=False), :54,79).
 * Weight blocks are HOST structs passed by value into the launch (constant-bank operands); [k][o] = input-major.
 * ---------------------------------------------------------------------------------------------- */
#define SPSK_EDGE_CH 24      /* conv_channels */
#define SPSK_EDGE_GROW 12    /* conv_growth_rate */
#define SPSK_EDGE_MAX_CIN 64
typedef struct spsk_edge_point_weights {
    int cin, relu;                                   /* transform FC: cin -> 24, optional ReLU (units 1..3) */
    float wt[SPSK_EDGE_MAX_CIN * SPSK_EDGE_CH];       /* wt[k*24 + o] = W_trans[o][k] */
    float bt[SPSK_EDGE_CH];
    float m[SPSK_EDGE_CH * 4 * SPSK_EDGE_GROW];       /* m[k*48 + o]: rows of [P | Q | R2 | R3] (see csrc/edge_conv.cu) */
    float c[4 * SPSK_EDGE_GROW];                      /* [b1 | 0 | b2 | b3] */
} spsk_edge_point_weights;
typedef struct spsk_edge_aggr_weights {
    float w2a[SPSK_EDGE_GROW * SPSK_EDGE_GROW];       /* [i*12 + o]: middle layer, columns that multiply l1 */
    float w3a[SPSK_EDGE_GROW * SPSK_EDGE_GROW];       /* last layer, columns that multiply l2 */
    float w3b[SPSK_EDGE_GROW * SPSK_EDGE_GROW];       /* last layer, columns that multiply l1 */
} spsk_edge_aggr_weights;
/* Per point: t = act(W_trans x + b) (rows, 24) and u = M t + c (rows, 48) = [P | Q | R2 | R3].  x (rows, ldx) f32. */
SPSK_API int spsk_edge_conv_point(const spsk_edge_point_weights *w, int rows, const float *x, int ldx, float *t,
                                  float *u, spsk_stream_t stream);
/* Per point i of scene s: out[i] = [max_j l3 | max_j l2 | max_j l1 | t_i] (60 floats, row stride ldo) over the k
 * neighbours j = idx[s, i, :] (indices within the scene), l1 = relu(P_i + Q_j), l2 = relu(W2a l1 + R2_i),
 * l3 = W3a l2 + W3b l1 + R3_i.  idx (b, n, k) int32; t (b*n, 24); u (b*n, 48). */
SPSK_API int spsk_edge_conv_aggregate(const spsk_edge_aggr_weights *w, int b, int n, int k, const int *idx,
                                      const float *t, const float *u, float *out, int ldo, spsk_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* SPSK_H_ */
