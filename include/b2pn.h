/*
 * b2pn -- C ABI of the B200-native PointNet++ set-abstraction path (libb2pn.so).
 *
 * The reference (cczls1991/DL_Biomass) is pure Python and has no FFI of its own; the native
 * boundary it crosses for this path is the torch.ops surface of torch_cluster / torch_scatter
 * / ATen that torch_geometric dispatches to.  Each entry point below names the reference call
 * site (file:line under /root/reference) and the upstream op it replaces.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the comment says "host"; the caller owns all
 *     buffers (inputs, outputs, workspaces); the library never allocates or synchronises, it
 *     only enqueues work on `stream` (a cudaStream_t passed as void*).
 *   - `ptr` arrays are CSR-style cloud offsets (int64, B+1 entries), as torch_cluster takes.
 *   - return value: 0 = ok, <0 = B2PN_E* argument error (nothing enqueued), >0 = cudaError_t
 *     reported by the launch.  b2pn_error_string() renders either.
 *   - re-entrant: there is NO process-wide setting.  Every option that shapes a launch (SM cap, deterministic
 *     reductions, kernel variant, random-number state) is a field of the call's argument struct, so the reference's
 *     thread-per-GPU callers (torch_geometric.nn.DataParallel, /root/reference/main.py:140) can drive several
 *     devices from several host threads.  The only static data are per-device caches of immutable facts (SM count,
 *     "dynamic shared memory attribute already raised") and the launch counter below (atomic).
 */
#ifndef B2PN_H_
#define B2PN_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2PN_ABI_VERSION 7
#define B2PN_OK 0
#define B2PN_EINVAL (-1)   /* null pointer / negative size / bad flag            */
#define B2PN_ENOTSUP (-2)  /* shape outside what the sm_100a kernels are built for */

typedef void *b2pn_stream_t;

int b2pn_abi_version(void);
const char *b2pn_error_string(int code);
/* kernels enqueued by this library so far in this process (bench.py's gpu_launches) */
int64_t b2pn_launch_count(void);

/* samples per cloud: ceil(float32(n) * float32(ratio)) -- torch_cluster.fps sizing
 * (reached from /root/reference/pointnet2_regressor.py:13).  Host-side helper. */
int64_t b2pn_fps_num_samples(int64_t n, float ratio);

/*
 * Farthest-point sampling.  Replaces torch.ops.torch_cluster.fps(src, ptr, ratio, random_start)
 * called at /root/reference/pointnet2_regressor.py:13 (SAModule.forward: idx = fps(pos, batch, ratio)).
 *   pos      [N,3] f32 row-major, clouds concatenated
 *   ptr      [B+1] i64 cloud offsets into pos
 *   out_ptr  [B+1] i64 offsets into out_idx (caller computes them with b2pn_fps_num_samples)
 *   start    [B]   i64 cloud-local start index, or NULL for 0 (random_start is drawn by the caller)
 *   max_n    host scalar: largest cloud in the batch (selects the kernel variant)
 *   out_idx  [M]   i64 GLOBAL point indices, per cloud in selection order (first = start)
 *   out_pos  [M,3] f32 pos[out_idx]   (optional, may be NULL; fuses pointnet2_regressor.py:19)
 *   out_batch[M]   i64 cloud id       (optional, may be NULL; fuses batch[idx] of :19)
 *   opts     host struct or NULL (defaults): kernel variant and the in-kernel random start (below)
 * Distances are ((dx*dx+dy*dy)+dz*dz) in separately rounded fp32; ties -> lowest index.
 */
typedef struct b2pn_fps_options {
    int32_t cluster;             /* CTAs per cloud: 0 = auto, 1/2/4/8/16; -1 / -2 = the pruned / Morton-sorted variants */
    int32_t threads;             /* threads per CTA: 0 = auto, 256/512/1024 (640/768 for the sorted variant)           */
    uint64_t seed;               /* random_start=True of torch_cluster.fps (the PyG default the reference runs with,    */
    int64_t *rng_state;          /* SURVEY.md A.1): with start == NULL and rng_state != NULL (DEVICE, 2 x i64, zeroed   */
                                 /* once by the caller) cloud b starts at b2pn_fps_random_start(seed, rng_state[0], b,  */
                                 /* n_b); the kernel advances rng_state[0] by one per call (graph replays included)     */
} b2pn_fps_options;
int b2pn_fps_f32(const float *pos, const int64_t *ptr, const int64_t *out_ptr, const int64_t *start,
                 int32_t B, int64_t max_n, int64_t *out_idx, float *out_pos, int64_t *out_batch,
                 const b2pn_fps_options *opts, b2pn_stream_t stream);
/* host-side restatement of the kernel's start draw: floor(u * n), u in [0,1) a hash of (seed, call, cloud) */
int64_t b2pn_fps_random_start(uint64_t seed, int64_t call, int32_t cloud, int64_t n);

/*
 * Farthest-point sampling in float64: the offline resampler that prepares the training clouds.  Replaces the numpy
 * farthest_point_sampling(coords, k) of /root/reference/downsampling_point_clouds.py:55-92 (called at :153), bit for
 * bit: float64 distances ((cx-x)^2+(cy-y)^2)+(cz-z)^2, first arg-max, start 0 unless `start` says otherwise, selected
 * points never compete again.  m <= n samples per cloud (out_ptr), no duplicates in the output.
 *   pos [N,3] f64, ptr / out_ptr [B+1] i64, start [B] i64 or NULL, out_idx [M] i64 GLOBAL indices,
 *   dist_workspace [N] f64 scratch.  One CTA per cloud: batch the plots.
 */
int b2pn_fps_f64(const double *pos, const int64_t *ptr, const int64_t *out_ptr, const int64_t *start, int32_t B,
                 int64_t *out_idx, double *dist_workspace, b2pn_stream_t stream);

/*
 * Segmented radius ball query with a neighbour cap.  Replaces
 * torch.ops.torch_cluster.radius(x, y, ptr_x, ptr_y, r, max_num_neighbors, num_workers) called at
 * /root/reference/pointnet2_regressor.py:14-15.  Instead of the compacted [2,E] edge list it
 * writes fixed-width slots (no data-dependent shape, no host sync):
 *   nbr [M,K] i32  GLOBAL source indices, ascending, first K with d2 < r*r (strict); pad = -1
 *   cnt [M]   i32  number of valid slots
 * edge_index of pointnet2_regressor.py:16 is (col = nbr[m,k], row = m) for k < cnt[m].
 * max_src / max_qry: host scalars, largest number of sources / queries in one cloud.
 */
int b2pn_ball_query_f32(const float *src_pos, const float *qry_pos, const int64_t *src_ptr,
                        const int64_t *qry_ptr, int32_t B, int64_t max_src, int64_t max_qry, double r,
                        int32_t K, int32_t *nbr, int32_t *cnt, b2pn_stream_t stream);

/*
 * The same query through a uniform grid, for large clouds (level 1: ~24 neighbours among 10 000 points make the
 * full scan above 99 % waste).  Identical results: cells of edge >= 1.0001 r, the same fp32 distance test on the
 * 27 cells around the query, hits sorted by source index.  workspace >= b2pn_ball_query_workspace_bytes().
 * n_src_total: number of source points over all clouds (src_ptr[B]).
 */
int64_t b2pn_ball_query_workspace_bytes(int32_t B, int64_t n_src_total);
int b2pn_ball_query_grid_f32(const float *src_pos, const float *qry_pos, const int64_t *src_ptr,
                             const int64_t *qry_ptr, int32_t B, int64_t n_src_total, int64_t max_qry, double r,
                             int32_t K, int32_t *nbr, int32_t *cnt, void *workspace, int64_t workspace_bytes,
                             b2pn_stream_t stream);

/*
 * Edge compaction (tensor-core path).  torch_cluster.radius returns a compact [2,E] edge list
 * (/root/reference/pointnet2_regressor.py:14-16); b2pn_ball_query_f32 writes fixed-width slots instead, and
 * this call packs the FILLED slots into rows for the bf16 set-abstraction kernels -- on the device, without
 * the masked_select host round trip: the row count stays in device memory (*num_rows).
 *   cnt [n_dst], nbr [n_dst,K]    output of b2pn_ball_query_f32, K <= 64
 *   rgrp    [capacity/8] u32      one descriptor per 8-row group: bits 0..23 centroid (0xFFFFFF none),
 *                                 24..26 first slot/8, 27..30 valid rows, 31 last group of the centroid
 *   row_src [capacity]   i32      gathered source point of the row, -1 = padding
 *   row_valid [capacity] fp16     1.0 for valid rows, 0 elsewhere (optional, may be NULL): the "ones" operand
 *                                 line that yields the bias gradients in the dW GEMMs
 *   num_rows [2]         i64      [0] rows in use (multiple of 64), [1] valid rows = edges (sum of cnt)
 * Centroid m owns max(8, round_up(cnt[m], 8)) consecutive rows that never cross a 64-row boundary.
 * capacity = b2pn_pack_rows_capacity(n_dst, K) rows (host-side upper bound used to size every buffer).
 */
int64_t b2pn_pack_rows_capacity(int64_t n_dst, int32_t K);
int64_t b2pn_pack_rows_workspace_bytes(int64_t n_dst);
int b2pn_pack_rows(const int32_t *cnt, const int32_t *nbr, int64_t n_dst, int32_t K, uint32_t *rgrp,
                   int32_t *row_src, void *row_valid, int64_t *num_rows, void *workspace,
                   int64_t workspace_bytes, b2pn_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Set-abstraction levels: fused gather + relative-position concat + shared MLP + max aggregation.
 *
 * One b2pn_sa_args describes one SAModule / GlobalSAModule call of
 * /root/reference/pointnet2_regressor.py:12-20 (PointConv(nn) == PointNetConv: message
 * nn([x_j || pos_j - pos_i]), aggr max) or :28-33 (nn(cat[x,pos]) + global_max_pool), i.e. the ATen /
 * cuBLAS / torch_scatter kernels K3..K8 of SURVEY.md 2.2.  `nn` is the PyG MLP of three Linear
 * layers with BatchNorm1d + activation after the first two (SURVEY.md A.4).
 * ---------------------------------------------------------------------------------------------- */
#define B2PN_PREC_F32 0   /* fp32 FMA on CUDA cores: the 1e-4 parity mode                      */
#define B2PN_PREC_BF16 1  /* 16-bit tcgen05 tensor-core tiles, fp32 accumulation in TMEM: forward-domain operands
                             (weights, normalised activations) in fp16, gradients in bf16 -- see DESIGN.md section 3 */
#define B2PN_SEG_SLOTS 0  /* SAModule: targets own K fixed-width neighbour slots (nbr/cnt)      */
#define B2PN_SEG_CLOUDS 1 /* GlobalSAModule: every source row belongs to cloud batch[row]       */
#define B2PN_X_F32 0
#define B2PN_X_BF16 1     /* 16-bit features (fp16: the out_bf16 side output of the previous level)            */
#define B2PN_ACT_NONE 0
#define B2PN_ACT_RELU 1

typedef struct b2pn_mlp3 {
    int32_t c[4];                /* channel list [c0, c1, c2, c3]; c0 = c_in + 3                     */
    int32_t act;                 /* B2PN_ACT_*                                                        */
    float eps, momentum;         /* BatchNorm1d eps (1e-5) and momentum (0.1)                         */
    const float *w[3];           /* Linear weight [c_{l+1}, c_l] row-major (torch layout)             */
    const float *b[3];           /* Linear bias   [c_{l+1}]                                           */
    const float *gamma[2];       /* BN weight [c_{l+1}] for l = 0,1                                   */
    const float *beta[2];        /* BN bias                                                           */
    float *running_mean[2];      /* updated in place when training                                    */
    float *running_var[2];
    int64_t *num_batches_tracked[2];
} b2pn_mlp3;

typedef struct b2pn_sa_args {
    int32_t precision;           /* B2PN_PREC_*                                                       */
    int32_t training;            /* 1: batch statistics + running-stat update, 0: running statistics  */
    int32_t seg_mode;            /* B2PN_SEG_*                                                        */
    int32_t K;                   /* slots per target (SLOTS); PREC_BF16: K <= 64                      */
    int64_t n_src, n_dst;        /* source points; targets (centroids or clouds)                      */
    int32_t c_in;                /* feature channels of x (0: no features, pointnet2_regressor.py:17) */
    int32_t x_dtype;             /* B2PN_X_F32 / B2PN_X_BF16 (16-bit = fp16, only with B2PN_PREC_BF16) */
    const void *x;               /* [n_src, c_in] row-major or NULL                                   */
    const float *pos_src;        /* [n_src, 3]                                                        */
    const float *pos_dst;        /* [n_dst, 3] (SLOTS) / NULL (CLOUDS: centre is the origin)          */
    const int32_t *nbr;          /* [n_dst, K] (SLOTS)                                                */
    const int32_t *cnt;          /* [n_dst]    (SLOTS); cnt[m] = 0 is allowed: an empty neighbourhood gives
                                    out[m] = 0 (and arg -1) on every path -- fp32, multi-pass 16-bit and the
                                    single-launch evaluation kernel -- as PyG's max aggregation of no messages */
    const int64_t *batch;        /* [n_src] sorted cloud id per row (CLOUDS)                          */
    b2pn_mlp3 mlp;
    float *out;                  /* [n_dst, c3]                                                       */
    int32_t *arg;                /* [n_dst, c3] arg-max slot (SLOTS) or source row (CLOUDS); -1 none  */
    void *h1, *h2;               /* saved activations of the two hidden layers.
                                    PREC_F32: pre-BN values, f32 row-major [rows, c], rows = n_dst*K (SLOTS) or
                                    n_src (CLOUDS).  PREC_BF16: normalised values (h-mean)*rstd, fp16
                                    FEATURE-major [c, ld], ld = row_capacity (SLOTS) or n_src rounded up to a
                                    multiple of 128 (CLOUDS)                                            */
    float *bn;                   /* [2][4][cmax] per BN layer: mean, rstd, scale, shift; cmax=max(c1,c2) */
    void *workspace;             /* b2pn_sa_workspace_bytes() bytes, scratch                          */
    int64_t workspace_bytes;
    /* PREC_BF16 + SEG_SLOTS: compacted rows from b2pn_pack_rows (ignored otherwise)                    */
    const uint32_t *rgrp;
    const int32_t *row_src;
    const int64_t *num_rows;
    int64_t row_capacity;        /* b2pn_pack_rows_capacity(n_dst, K)                                   */
    const void *row_valid;       /* fp16 [row_capacity] from b2pn_pack_rows, or NULL                    */
    /* PREC_BF16: activations of the two hidden layers AFTER BatchNorm affine + activation, fp16 feature-major
     * [c, ld] like h1/h2, invalid rows zero.  Written by forward, read by backward: stored next to the
     * normalised values so that every later consumer is a plain tensor-map (TMA) copy.  Required whenever
     * h1 != NULL.                                                                                        */
    void *a1, *a2;
    /* PREC_BF16 + SEG_SLOTS, optional (NULL = gather in the loader warps): the gathered + concatenated layer-1
     * operand, fp16 feature-major [c_img + 1, ld] with c_img = (x fp32 ? 2 : 1) * c_in + 6 image columns
     * [x | x_lo | dpos_hi | dpos_lo] and a last line of ones on valid rows.  Written by forward (or ahead of it by
     * b2pn_sa_gather_rows: set g1_ready = 1 and forward skips the gather), read by backward.                    */
    void *g1;
    int32_t g1_ready;
    /* per-call launch options (there is no process-wide state)                                              */
    int32_t sm_limit;            /* > 0: the persistent tensor-core kernels of THIS call take at most this many CTAs
                                    (0 = one per SM).  Used while the grouping kernels of the next batch run on a second
                                    stream: farthest-point sampling holds one SM per cloud for its whole latency-bound
                                    duration and a persistent kernel must not wait for those SMs                      */
    int32_t deterministic;       /* PREC_BF16 backward.  0: the row splits of a dW GEMM add their partial sums into one
                                    buffer with fp32 atomics (red.global.add.v4.f32): fastest, last bits vary from run to
                                    run (as in the reference's scatter / cuBLAS kernels).  1: per-split partials summed
                                    in a fixed order and the grad_x scatter of SLOTS levels accumulated in 64-bit fixed
                                    point: bit-reproducible gradients.
                                    Range of that accumulator: unit 2^-40, every fp32 addend rounded to it (absolute
                                    error <= 2^-41 ~ 4.5e-13 per addend; addends below that vanish) and every partial
                                    sum of one grad_x element held in |sum| < 2^23 ~ 8.4e6.  For the result to stay
                                    within 16-bit accuracy (~4e-3 relative) the typical addend must exceed ~1e-10;
                                    the level-2 addends of a bf16 training step (3 x 640 points) span 8e-10 .. 8e-2,
                                    median 1.6e-3; tests/test_sa_pinned_gpu.py sweeps grad_out over 2^-24 .. 2^12   */
    void *out_bf16;              /* PREC_BF16, optional: a 16-bit (fp16) copy of `out` [n_dst, c3] written by the same epilogue --
                                    the next level's gather reads it (half the bytes, no separate cast kernel)         */
} b2pn_sa_args;

typedef struct b2pn_sa_grads {
    const float *grad_out;       /* [n_dst, c3]                                                       */
    float *grad_w[3], *grad_b[3];/* overwritten                                                       */
    float *grad_gamma[2], *grad_beta[2];
    float *grad_x;               /* [n_src, c_in], overwritten (PREC_BF16: the library clears it before its scatter-add;
                                    PREC_F32: the caller passes it ZERO-INITIALISED); NULL = skip */
} b2pn_sa_grads;

/* scratch bytes needed by forward (backward=0) or backward (backward=1) for these shapes */
int64_t b2pn_sa_workspace_bytes(const b2pn_sa_args *args, int32_t backward);
int b2pn_sa_forward(const b2pn_sa_args *args, b2pn_stream_t stream);
/* 1 if b2pn_sa_forward would run these arguments (shapes, precision, training flag) through the single-launch evaluation
 * kernel, which stores no hidden activation.  The caller opts in by passing h1 == NULL (then h2, a1, a2, bn, g1 and arg
 * are not touched either -- arg may be NULL -- and no backward pass can follow); with h1 != NULL the multi-pass kernels run
 * and fill them.  0 otherwise. */
int b2pn_sa_eval_fused(const b2pn_sa_args *args);
/* PREC_BF16 + SEG_SLOTS: only the gather + concat of /root/reference/pointnet2_regressor.py:17-18's message inputs
 * ([x_j | pos_j - pos_i]) into args->g1.  Needs x, pos_src, pos_dst, the compacted rows and c_in / mlp.c[0..1]; no
 * weights, no workspace: a caller may run it ahead of the forward pass (e.g. for the next batch on another stream).
 * B2PN_ENOTSUP when the level does not take a materialised operand (b2pn_sa_forward then gathers in its loaders). */
int b2pn_sa_gather_rows(const b2pn_sa_args *args, b2pn_stream_t stream);
int b2pn_sa_backward(const b2pn_sa_args *args, const b2pn_sa_grads *grads, b2pn_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Regression head: the MLP([c0, c1, c2, c3], act=None, dropout=p) of /root/reference/pointnet2_regressor.py:50,58
 * (torch_geometric.nn.MLP: Lin -> BatchNorm1d -> dropout -> Lin -> BatchNorm1d -> dropout -> Lin) on B <= 32 rows,
 * one forward and one backward kernel instead of ~60 ATen launches.  fp32.  c1, c2 <= 256, c3 <= 8.
 * Training needs B >= 2 (B2PN_EINVAL otherwise): like torch's BatchNorm1d, the head does not normalise one row by
 * its own zero variance.
 * Dropout noise is counter based: (seed, *rng_counter, layer, element); forward bumps *rng_counter when training,
 * which keeps the op replayable from a CUDA graph.
 * ---------------------------------------------------------------------------------------------- */
typedef struct b2pn_head_args {
    int32_t B;                   /* rows (tree clouds)                                                */
    int32_t c[4];                /* channel list                                                      */
    int32_t training;            /* 1: batch statistics, running-stat update, dropout; 0: eval        */
    float p, eps, momentum;      /* dropout probability; BatchNorm eps, momentum                      */
    const float *x;              /* [B, c0]                                                           */
    const float *w[3];           /* Linear weights [c_{l+1}, c_l]                                     */
    const float *b[3];
    const float *gamma[2];
    const float *beta[2];
    float *running_mean[2];
    float *running_var[2];
    int64_t *num_batches_tracked[2];
    uint64_t seed;
    int64_t *rng_counter;        /* device scalar, may be NULL when p == 0 or not training            */
    float *out;                  /* [B, c3]                                                           */
    float *xhat[2];              /* saved for backward: normalised hidden values [B, c_{l+1}]         */
    uint8_t *mask[2];            /* saved dropout keep-masks [B, c_{l+1}] (may be NULL when p == 0)   */
    float *rstd[2];              /* saved 1/sqrt(var + eps) [c_{l+1}]                                 */
} b2pn_head_args;

typedef struct b2pn_head_grads {
    const float *grad_out;       /* [B, c3]                                                           */
    float *grad_x;               /* [B, c0] or NULL                                                   */
    float *grad_w[3], *grad_b[3];
    float *grad_gamma[2], *grad_beta[2];
} b2pn_head_grads;

int b2pn_head_forward(const b2pn_head_args *args, b2pn_stream_t stream);
int b2pn_head_backward(const b2pn_head_args *args, const b2pn_head_grads *grads, b2pn_stream_t stream);

/* The training loss of /root/reference/main.py:157-169: loss = sum_c w[c] * mean_b (y[b,c] - pred[b,c])^2 over
 * pred, y [B, C] row-major (C <= 32; the reference has C = 4 with w = 1/11, 1/12, 1/5, 1/72), and in the same launch
 * its gradient grad[b,c] = 2 w[c] (pred - y) / B (grad may be NULL).  fp32, fixed summation order. */
int b2pn_weighted_mse(const float *pred, const float *y, const float *w, int32_t B, int32_t C, float *loss,
                      float *grad, b2pn_stream_t stream);

/* The optimiser step of /root/reference/main.py:84,172 -- torch.optim.Adam(params, lr, weight_decay): L2 penalty added
 * to the gradient, bias-corrected first / second moments, no amsgrad -- as ONE launch over a flat arena holding every
 * parameter (dl_biomass_b200/optim.py): param, grad, exp_avg, exp_avg_sq are parallel fp32 buffers of n elements
 * (n % 4 == 0, 16-byte aligned).  grad is multiplied by grad_scale first (1/world_size after a SUM all-reduce).
 * state: DEVICE, 2 x i64 zero-initialised: [0] steps taken so far (the kernel uses state[0] + 1 in the bias corrections
 * and advances it, so a CUDA-graph replay is a real optimiser step), [1] scratch. */
int b2pn_adam_step(float *param, const float *grad, float *exp_avg, float *exp_avg_sq, int64_t n, float lr, float beta1,
                   float beta2, float eps, float weight_decay, float grad_scale, int64_t *state, b2pn_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Training-time augmentation on the device (SURVEY.md 8(f) row f2): point_removal -> random_noise -> rotate_points of
 * /root/reference/augmentation.py:54-122 as applied by AugmentPointCloudsInFiles.__getitem__ (:287-289), for B clouds
 * of a resident cloud cache, written straight into the concatenated batch layout (pos, x, batch) the model takes.
 * The caller draws the per-cloud scalars (they fix the layout); per-point randomness is counter based:
 * b2pn_augment_draw(seed, uid, stream, counter) is the 64-bit draw the kernel uses (stream 0: order key of source
 * point `counter`, top 32 bits; stream 1: duplication key of kept position `counter`; stream 2: deviate number
 * `counter` = kept position * (3 + F) + component, Box-Muller on bits 63..40 and 39..16).
 * ---------------------------------------------------------------------------------------------- */
#define B2PN_AUG_MAX_POINTS 16384   /* per source cloud (one CTA sorts a cloud in shared memory)                */
typedef struct b2pn_augment_cloud {
    int64_t src_off;             /* first point of the cloud in the cache                                      */
    int64_t out_off;             /* first output point of the cloud in the batch                               */
    uint64_t uid;                /* generator stream of this sample (e.g. epoch * dataset size + cloud id)     */
    int32_t n_src;               /* points of the cached cloud                                                 */
    int32_t n_keep;              /* points kept by point_removal: round(0.9 n_src) .. n_src                    */
    int32_t n_dup;               /* jittered copies appended by random_noise: 0 .. round(0.1 n_keep)           */
    float noise_sd;              /* jitter sd 0.01 .. 0.025, NEGATIVE when the deviates are subtracted         */
    float cos_a, sin_a;          /* rotation about z by a in (-180, 180] degrees                               */
} b2pn_augment_cloud;

/* clouds: HOST array of B records (copied into the launch parameters; nothing is read after return).
 * out_pos [sum(n_keep + n_dup), 3], out_x [.., F] (F > 0), optional out_batch (int64 cloud number 0..B-1 per point) and
 * out_src (int32 index of the source point inside its cached cloud, for carrying further attributes). */
int b2pn_augment_batch(const float *pos, const float *x, int32_t F, const b2pn_augment_cloud *clouds, int32_t B,
                       uint64_t seed, float *out_pos, float *out_x, int64_t *out_batch, int32_t *out_src,
                       b2pn_stream_t stream);
uint64_t b2pn_augment_draw(uint64_t seed, uint64_t uid, uint32_t stream, uint64_t counter);
int32_t b2pn_augment_max_points(void);

/*
 * Hardware self-test of the tcgen05 GEMM pipeline (debug aid used by tests/test_tc_gpu.py; not part of
 * the reference's surface).  out[m][row] (fp32, leading dimension ld_out) = sum_k w[m][k] * b(row, k) with
 * b in fp16, row-major [rows][k] (mode 0: K-major B tiles) or feature-major [k][ld] (mode 1: MN-major B
 * tiles; mode 2: the same operand fetched by TMA tensor-map copies).  zeros3: [rows,3] fp32 zeros.  workspace >= packed weight image + 1 KB.
 */
int b2pn_tc_gemm_selftest(const float *w, int32_t m_out, int32_t k, const void *b_bf16, int32_t mode, int64_t rows,
                          int64_t ld, const float *zeros3, float *out, int64_t ld_out, void *workspace,
                          int64_t workspace_bytes, b2pn_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* B2PN_H_ */
