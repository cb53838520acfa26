/*
 * pointrcnn_b200.h -- C ABI of libpointrcnn_b200.so: B200 (sm_100a) kernels for PointRCNN's
 * per-scene point-cloud operator path.
 *
 * This is the drop-in boundary.  Every entry point takes plain device pointers, sizes and a
 * CUDA stream (as void*; NULL = legacy default stream); no torch types.  Each one replaces
 * one native entry point of the reference's three extension modules (paths relative to the
 * reference tree); the extension-module shims in pointrcnn_b200/ext/{pointnet2_cuda,
 * iou3d_cuda,roipool3d_cuda}.py bind them under the reference's exact Python names.
 *
 * Conventions
 *   - all tensors contiguous; float = fp32, int = int32, long long = int64
 *   - the CALLER allocates every output (and zero-/1e10-fills where the reference's Python
 *     wrappers do: ball-query idx, grad buffers, pooled/empty, FPS temp)
 *   - scratch memory is caller-provided too (prb_*_workspace_bytes tells how much); nothing
 *     in this library calls cudaMalloc/cudaFree or synchronises the device, except
 *     prb_nms*_host which must fill a host buffer before returning (the reference signature)
 *   - return value: 0 on success, otherwise a cudaError_t (or -1 for bad arguments);
 *     prb_last_error() gives the message.  Nothing exit()s the process.
 *   - kernels launch on the given stream, on the current device (callers set the device).
 */
#ifndef POINTRCNN_B200_H_
#define POINTRCNN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PRB_ABI_VERSION 5   /* 3: prb_options (per-thread tuning block; no per-call environment reads); 4: mlp_tune, prb_mlp_rows2;
                             * 5: ordered FPS, input pipeline / KITTI output group, prb_options.roipool_fused */
#if defined(__GNUC__)
#define PRB_API __attribute__((visibility("default")))
#else
#define PRB_API
#endif

PRB_API int prb_abi_version(void);
PRB_API const char *prb_last_error(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
PRB_API unsigned long long prb_launch_count(void);

/* Per-thread tuning block.  Every heuristic the kernels' launchers apply can be overridden here; 0 / the value
 * prb_options_init() fills in means "library default".  The block is THREAD-LOCAL (each nn.DataParallel worker
 * thread owns one), nothing is process-global, and no entry point reads the environment per call: PRB_*
 * environment variables only seed the values prb_options_init() returns, once, when first used. */
typedef struct prb_options {
    int fps_cluster;   /* CTAs per scene of the cluster FPS kernel (1,2,4,8); 0 = heuristic */
    int fps_prune;     /* 0: never use the pruned single-CTA kernel; 1: for 4097..16384 points; 2: also 2049..4096 */
    int fps_threads;   /* threads per CTA of the rank kernel; 0 = heuristic */
    int fps_generic;   /* 1: force the generic (reference-shaped) kernel */
    int mlp_gather;    /* layer-0 row gather of the chain kernel: 0 registers (+tf32 rounding), 1 cp.async.cg, 2 cp.async.ca */
    int mlp_ng;        /* row groups per CTA (legacy kernel); 0 = heuristic */
    int mlp_occ;       /* 1: one CTA per SM; 3: the three-CTA build where it applies (narrow SA chains); 0 = plan rule / measured */
    int mlp_sms;       /* size the persistent grid for this many SMs; 0 = all */
    int mlp_atmem;     /* 1: layers >= 1 take their A operand from tensor memory (legacy kernel) */
    int mlp_sleepy;    /* bit 0: MMA issuer waits with a suspend hint, bit 1: weight producer does */
    int mlp_trace;     /* 1: record the phase trace read by prb_debug_mlp_trace */
    int mlp_pipeline;  /* 1: role-specialised pipelined chain kernel (gather of tile i+1 overlaps tile i); 0: legacy */
    int mlp_ne, mlp_ngw;   /* pipelined kernel: epilogue (1, 2) / gather (1, 2, 3) warp groups per CTA; 0 = plan rule */
    int mlp_zs, mlp_nbuf;  /* pipelined kernel: last-layer slice width (multiple of 32) / slice buffers (1 or 2); 0 = plan rule */
    int mlp_brows;     /* pipelined kernel: rows per weight stage / MMA N (32..256); 0 = 64 */
    int mlp_pool;      /* SA max-pool over 16..128 samples: 0 = quad tensor-memory layout (2 rows x 4 columns per thread, 3 exchange
                        * stages), 1 = shuffle butterfly, 2 = CREDUX (warp-wide max per channel), 3 = staged tile for 64/128 samples */
    int mlp_resident;  /* 1 (default): chains whose weight stages all fit in shared memory load them once per CTA instead of per tile */
    int mlp_lazy_ns;   /* poll interval (ns) of the run-ahead roles (gather warps, weight producers) in the narrow builds; 0 = 400 */
    int mlp_fill;      /* 1 (default): single-layer launches with fewer tiles than SMs are dealt to more column groups until every
                        * SM has one (lower latency, each group re-gathers its rows); 0: only as many groups as tensor memory needs */
    int mlp_tune;      /* 1 (default): the first eager launch of a chain shape times the two-CTA and the one-CTA build and
                        * caches the faster one per device and shape; 0: rule-based plan only */
    int roipool_exhaustive;  /* 1: roipool3d pass A tests every point against every box (no x-z binning) */
    int roipool_parts;     /* roipool3d pass B: CTAs per box (1..8); 0 = 1 */
    int roipool_stage_kb;  /* roipool3d pass B: shared staging area per CTA in KB (8..160); 0 = 48 */
    int roipool_direct;    /* 1: roipool3d pass B takes boxes with many rows through scalar L1 gathers (first version) instead of chunked staging */
    int nn_walk;           /* three_nn on the grid: 0 = 27 unrolled cell walks (default), 1 = one convergent cursor loop per lane (slower) */
    int nn_sort_queries;   /* 1: three_nn groups the queries by grid cell before the search; measured: the sort costs what the locality saves */
    int grid_csr;      /* 1: hash grid as CSR runs (counting sort per scene) instead of linked lists; slower at the RPN shapes */
    int grid_debug;    /* 1: print (and synchronise for) the 3-NN grid's fallback counts */
    float nn_cell;     /* 3-NN grid cell edge in units of the mean point spacing (default 1.6) */
    int roipool_fused;     /* 1: the binned assign pass of a box runs inside the copy kernel's CTA (no index list in HBM); 0 (default): two kernels --
                            * measured: fused 0.167 ms, two kernels 0.156 ms at the configs[3] shape */
} prb_options;
PRB_API void prb_options_init(prb_options *o);                 /* library defaults */
PRB_API int prb_set_thread_options(const prb_options *o);      /* NULL: back to the defaults */
PRB_API void prb_get_thread_options(prb_options *o);

/* ------------------------------------------------------------------ pointnet2_cuda ------
 * replaces pointnet2_lib/pointnet2/src/pointnet2_api.cpp:10-23 */

/* furthest_point_sampling_wrapper, sampling.cpp:36-46 -> sampling_gpu.cu:93-253.
 * xyz (b,n,3); temp (b,n) in/out running min distance (caller prefills 1e10); idx (b,m) int32.
 * Index-exact with the reference incl. its tie rule.  new_xyz (b,m,3) may be NULL; when given,
 * the sampled coordinates are emitted too (replaces the gather_operation that follows FPS in
 * pointnet2_modules.py:32-35). */
PRB_API int prb_furthest_point_sampling(int b, int n, int m, const float *xyz, float *temp, int *idx,
                                float *new_xyz, void *stream);
/* same, with caller scratch (device, prb_fps_workspace_bytes; 0 = none needed).  With scratch, scenes of
 * 4097..16384 points run the pruned single-CTA kernel (same indices and temp, bit for bit). */
PRB_API size_t prb_fps_workspace_bytes(int b, int n);
PRB_API int prb_furthest_point_sampling_ws(int b, int n, int m, const float *xyz, float *temp, int *idx,
                                   float *new_xyz, void *workspace, size_t workspace_bytes, void *stream);
/* same result, for inputs that are LIKELY already in sampling order (the output of a previous
 * furthest_point_sampling from point 0: SA level l+1 samples level l's output, pointnet2_msg.py:57-61, where the
 * answer is 0..m-1 unless two points tie for a maximum).  Per scene the library PROVES idx = (0..m-1) with n*m
 * independent distance evaluations (every pick the maximum, exact ties settled by the reference's rank rule; nothing is assumed about the input) and
 * writes idx / new_xyz / temp exactly as the sampling kernels would; scenes where the proof fails (ties, duplicates,
 * NaN, unordered input) are sampled by the ordinary kernels in the same call.  No host synchronisation.
 * todo_out (b) int32, optional: 0 = scene answered by the proof, 1 = sampled.  Scratch: prb_fps_ordered_workspace_bytes. */
PRB_API size_t prb_fps_ordered_workspace_bytes(int b, int n, int m);
PRB_API int prb_furthest_point_sampling_ordered_ws(int b, int n, int m, const float *xyz, float *temp, int *idx,
                                           float *new_xyz, int *todo_out, void *workspace, size_t workspace_bytes,
                                           void *stream);

/* gather_points_wrapper_fast / gather_points_grad_wrapper_fast, sampling.cpp:11-33 */
PRB_API int prb_gather_points(int b, int c, int n, int npoints, const float *points, const int *idx,
                      float *out, void *stream);
PRB_API int prb_gather_points_grad(int b, int c, int n, int npoints, const float *grad_out, const int *idx,
                           float *grad_points, void *stream);

/* ball_query_wrapper_fast, ball_query.cpp:14-25 -> ball_query_gpu.cu:9-67.
 * argument order is the reference's positional order (b,n,m,radius,nsample,new_xyz,xyz,idx). */
PRB_API int prb_ball_query(int b, int n, int m, float radius, int nsample, const float *new_xyz,
                   const float *xyz, int *idx, void *stream);
/* two radii over the same centres in one scan (the MSG case, pointnet2_modules.py:37-38);
 * each idx_k has the semantics of prb_ball_query(radius_k, nsample_k) */
PRB_API int prb_ball_query_msg2(int b, int n, int m, float radius0, int nsample0, float radius1, int nsample1,
                        const float *new_xyz, const float *xyz, int *idx0, int *idx1, void *stream);

/* group_points_wrapper_fast / group_points_grad_wrapper_fast, group_points.cpp:11-36 */
PRB_API int prb_group_points(int b, int c, int n, int npoints, int nsample, const float *points,
                     const int *idx, float *out, void *stream);
PRB_API int prb_group_points_grad(int b, int c, int n, int npoints, int nsample, const float *grad_out,
                          const int *idx, float *grad_points, void *stream);

/* three_nn_wrapper_fast, interpolate.cpp:14-23 (n unknown, m known; outputs d^2 and idx).
 * weight (b,n,3) may be NULL; when given, the inverse-distance weights of
 * pointnet2_modules.py:140-142 are emitted as well. */
PRB_API int prb_three_nn(int b, int n, int m, const float *unknown, const float *known, float *dist2,
                 int *idx, float *weight, void *stream);

/* three_interpolate_wrapper_fast (b,c,m,n) / three_interpolate_grad_wrapper_fast (b,c,n,m),
 * interpolate.cpp:26-54 -- note the different n/m order of the two, kept as in the reference */
PRB_API int prb_three_interpolate(int b, int c, int m, int n, const float *points, const int *idx,
                          const float *weight, float *out, void *stream);
PRB_API int prb_three_interpolate_grad(int b, int c, int n, int m, const float *grad_out, const int *idx,
                               const float *weight, float *grad_points, void *stream);

/* (B,C,N) <-> (B,N,C) layout change used in front of the fused kernels */
PRB_API int prb_transpose_bcn_to_bnc(int b, int c, int n, const float *in, float *out, void *stream);

/* ------------------------------------------------------------------ fused SA / FP -------
 * New natives behind PointnetSAModuleMSG.forward / PointnetFPModule.forward
 * (pointnet2_modules.py:19-55, 127-156).  Eval-mode BatchNorm is folded by the host into a
 * per-channel (scale, shift); every layer is y = relu(scale * (W x) + shift).
 * Weights are passed pre-packed by prb_mlp_pack_weights (tile images in the tcgen05 shared-
 * memory operand layout), so the kernel stages them with plain bulk copies. */

typedef struct prb_mlp_desc {
    int num_layers;          /* 1..3 */
    int c_in;                /* input channels of layer 0 (incl. the 3 xyz channels for SA) */
    int c_out[3];            /* output channels per layer */
    const float *packed_w;   /* device, from prb_mlp_pack_weights */
    const float *scale;      /* device; layer after layer, each layer zero-padded to round_up(c_out,32) floats;
                              * NULL = the scale is already folded into the packed weights (y = relu(W'x + shift)),
                              * which lets the SA kernel pool raw accumulators and apply shift/ReLU once per centre */
    const float *shift;      /* device; same layout */
    int flags;               /* bit 0: the LAST layer is linear (no ReLU): y = W x + shift, e.g. detection heads */
} prb_mlp_desc;

/* bytes of the packed image for one MLP */
PRB_API size_t prb_mlp_packed_bytes(int num_layers, int c_in, const int *c_out);
/* host-side packing: w[l] is the (c_out[l], c_in_l) row-major conv weight; dst is HOST memory of
 * prb_mlp_packed_bytes() bytes which the caller then uploads */
PRB_API int prb_mlp_pack_weights(int num_layers, int c_in, const int *c_out, const float *const *w, void *dst);

/* grouped MLP + max-pool: for every centre p and every sample s, row = [xyz[idx]-new_xyz[p],
 * feats_pm[idx]] -> MLP -> max over s.  feats_pm is POINT-major (b,n,c_feat) (NULL if c_feat==0);
 * out is channel-major (b, out_stride_c, npoint) written at channel offset out_c_off. */
PRB_API int prb_sa_group_mlp_max(int b, int n, int npoint, int nsample, int c_feat, const float *xyz,
                         const float *new_xyz, const float *feats_pm, const int *idx,
                         const prb_mlp_desc *mlp, float *out, int out_stride_c, int out_c_off,
                         void *stream);

/* feature propagation: row(u) = [sum_k w[u,k]*known_pm[idx[u,k]], skip[:,u]] -> MLP.
 * known_pm point-major (b,m,c_known); skip channel-major (b,c_skip,n) or NULL; out (b,c_last,n) */
PRB_API int prb_fp_interp_mlp(int b, int n, int m, int c_known, int c_skip, const float *known_pm,
                      const int *idx, const float *weight, const float *skip,
                      const prb_mlp_desc *mlp, float *out, void *stream);

/* --- workspace-taking forms (what the Python mirror calls: no allocation inside the library) ---
 * kind: 0 = SA rows [rel xyz | feats], 1 = FP rows [interp | skip], 2 = plain rows.  `split` is the
 * channel where the first row source ends (3 for SA, c_known for FP, 0 for plain rows); it fixes
 * how layer-0 weight columns are permuted into K-chunks. */
PRB_API size_t prb_mlp_packed_bytes_ex(int kind, int split, int num_layers, int c_in, const int *c_out);
PRB_API int prb_mlp_pack_weights_ex(int kind, int split, int num_layers, int c_in, const int *c_out,
                                    const float *const *w, void *dst);
PRB_API size_t prb_sa_workspace_bytes(int b, int npoint, int nsample, int c_feat, int num_layers, const int *c_out);
PRB_API size_t prb_fp_workspace_bytes(int b, int n, int c_known, int c_skip, int num_layers, const int *c_out);
PRB_API size_t prb_rows_workspace_bytes(long rows, int c_in, int num_layers, const int *c_out);
/* as prb_sa_group_mlp_max / prb_fp_interp_mlp with caller scratch (device, *_workspace_bytes; may be
 * NULL/0 when the chain fits one launch).  out_pm: NULL, or a second POINT-major copy of the result,
 * (b, npoint, out_stride_c) at channel offset out_c_off for SA and (b, n, c_last) for FP -- the layout
 * the next level's gather reads, so no transpose kernel runs between levels. */
PRB_API int prb_sa_group_mlp_max_ws(int b, int n, int npoint, int nsample, int c_feat, const float *xyz,
                                    const float *new_xyz, const float *feats_pm, const int *idx,
                                    const prb_mlp_desc *mlp, float *out, float *out_pm, int out_stride_c,
                                    int out_c_off, void *workspace, size_t workspace_bytes, void *stream);
/* SA chains with c_feat <= 5: layer 0 is evaluated by the gather warps (CUDA cores) and only layers 1 .. L-1 run on the
 * tensor core.  l0_w: (c0, 8) device floats per layer-0 channel [wx, wy, wz, wf0 .. wf4] (BN scale folded in, zero beyond
 * 3 + c_feat), l0_shift: c0 device floats; `mlp`: layers 1 .. L-1 packed as plain rows (kind 2, c_in = c0), scale NULL.
 * Same output as prb_sa_group_mlp_max_ws up to fp32 summation order; the chain must fit one launch (no workspace). */
PRB_API int prb_sa_group_mlp_max_l0(int b, int n, int npoint, int nsample, int c_feat, const float *xyz,
                                    const float *new_xyz, const float *feats_pm, const int *idx, int c0,
                                    const float *l0_w, const float *l0_shift, const prb_mlp_desc *mlp, float *out,
                                    float *out_pm, int out_stride_c, int out_c_off, void *stream);
PRB_API int prb_fp_interp_mlp_ws(int b, int n, int m, int c_known, int c_skip, const float *known_pm,
                                 const int *idx, const float *weight, const float *skip,
                                 const prb_mlp_desc *mlp, float *out, float *out_pm, void *workspace,
                                 size_t workspace_bytes, void *stream);
/* plain row MLP: x_rows (rows, c_in) row-major -> out_rows (rows, out_pitch), out_pitch >= round_up(c_last,32);
 * replaces a pt_utils.SharedMLP applied to (B,C,N,1) tensors (lib/net/rcnn_net.py:58-66 xyz_up_layer / merge_down_layer) */
PRB_API int prb_mlp_rows(long rows, int c_in, const float *x_rows, const prb_mlp_desc *mlp, float *out_rows,
                         int out_pitch, void *workspace, size_t workspace_bytes, void *stream);
/* the same with strided inputs and an optional second K segment: layer 0 reads [a_rows[:, :c_a] | b_rows[:, :c_b]] (row
 * pitches in floats, any alignment; 128-bit loads when base and pitch are 16-byte aligned).  With c_b > 0 the weights are
 * packed with prb_mlp_pack_weights_ex(kind 1, split c_a), else kind 2.  This is merge_down_layer on cat(xyz_feature,
 * rpn_feature) (lib/net/rcnn_net.py:171-175) without materialising the concatenation, and xyz_up_layer on a column
 * slice of the pooled rows. */
PRB_API size_t prb_rows2_workspace_bytes(long rows, int c_a, int c_b, int num_layers, const int *c_out);
PRB_API int prb_mlp_rows2(long rows, int c_a, const float *a_rows, int a_pitch, int c_b, const float *b_rows, int b_pitch,
                          const prb_mlp_desc *mlp, float *out_rows, int out_pitch, void *workspace, size_t workspace_bytes,
                          void *stream);

/* ------------------------------------------------------------------ RPN proposal path (next to the hot path) -----
 * prb_decode_rpn_proposals replaces decode_bbox_target as called by the proposal layer (lib/utils/bbox_transform.py:
 * 24-121 from lib/rpn/proposal_layer.py:23-32): xyz (n,3), reg (n,c) -> out (n,7) [x, y = bottom centre, z, h, w, l, ry];
 * anchor_hwl = 3 HOST floats (cfg.CLS_MEAN_SIZE[0]).  Every torch op of the reference is one fp32 rounding here too.
 * prb_rpn_proposals replaces ProposalLayer.forward's per-scene loop (lib/rpn/proposal_layer.py:34-142): order = the
 * indices of torch.sort(scores, descending) (b,n) int64; distance_based selects the (0,40] / (40,80] split with the
 * 70/30 top-n quotas, otherwise the score-based variant; normal_nms: nms_normal_gpu instead of nms_gpu.  Outputs
 * (b, post_nms_top_n, 7) and (b, post_nms_top_n), zero rows behind the survivors.  No host synchronisation.
 * Deviations on degenerate inputs: equal scores keep the order of `order` (the reference re-sorts each slice with an
 * unstable sort); an empty near range yields zero rows (the reference asserts). */
PRB_API int prb_decode_rpn_proposals(long n, int c, const float *xyz, const float *reg, const float *anchor_hwl,
                                     float loc_scope, float loc_bin_size, int num_head_bin, int get_xz_fine, float *out,
                                     void *stream);
PRB_API size_t prb_rpn_proposals_workspace_bytes(int b, int post_nms_top_n);
PRB_API int prb_rpn_proposals(int b, int n, const float *boxes, const float *scores, const long long *order,
                              int distance_based, int pre_nms_top_n, int post_nms_top_n, float nms_thresh, int normal_nms,
                              float *out_boxes, float *out_scores, void *workspace, size_t workspace_bytes, void *stream);

/* diagnostics (PRB_MLP_TRACE=1): clock64 stamps of CTA 0 at the phase boundaries of its first 32 tiles (32 x 16) */
PRB_API int prb_debug_mlp_trace(long long *dst);
/* pipelined kernel (prb_options.mlp_trace): cycles CTA 0's roles spent in each class of barrier wait during the last traced
 * launch, 8 x 8 int64 (slot 7 of a row = total cycles of the role's loop): issuer A {x/z_free, a_full, b0_full}, issuer B
 * {z_free, ready, b1_full, fence, mma issue, commit}, weight producer 0 {b0_empty}, producer 1 {b1_empty}, gather warp 0
 * {a_empty}, epilogue warp 0 {r_full, z_full} */
PRB_API int prb_debug_pipe_trace(long long *dst);
/* measured plan choices so far: up to max_entries rows of 18 ints {mode_in, mode_out, layers, nsample, K chunks of layer 0,
 * tiles, np0, np1, np2, winning build, then 4 x (candidate build, measured microseconds; 0 = no candidate)}; builds: 2 = two
 * CTAs per SM (4 epilogue + 4 gather warps), 1 = one CTA 8 + 8, 3 = one CTA 8 + 12, 4 = three CTAs 4 + 4; returns the rows */
PRB_API int prb_debug_tuned_plans(int *dst, int max_entries);

/* --- uniform-grid neighbour search: same results, bit for bit, as prb_ball_query(_msg2) / prb_three_nn
 * (first-nsample-in-index-order and lexicographic (d2, idx) rules kept; queries the grid cannot answer
 * exactly fall back to the exhaustive kernels inside the call).  Used for n >= a few thousand points. */
PRB_API size_t prb_grid_workspace_bytes(int b, int n_points, int n_queries);
PRB_API int prb_ball_query_grid(int b, int n, int m, int nr, const float *radius, const int *nsample,
                                const float *new_xyz, const float *xyz, int *const *idx, void *workspace,
                                size_t workspace_bytes, void *stream);
PRB_API int prb_three_nn_grid(int b, int n, int m, const float *unknown, const float *known, float *dist2,
                              int *idx, float *weight, void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------ roipool3d_cuda ------
 * replaces lib/utils/roipool3d/src/roipool3d.cpp:48-79 (forward) -> roipool3d_kernel.cu:209-237.
 * xyz (B,N,3), boxes3d (B,M,7) ALREADY enlarged, pts_feature (B,N,C) -> pooled (B,M,S,3+C),
 * empty_flag (B,M) int32; both outputs zero-filled by the caller (rows of empty boxes stay 0).
 * rois_canonical: NULL, or (B,M,7) original RoIs -> the canonical transform of
 * lib/net/rcnn_net.py:146-152 is applied to the xyz columns while they are written. */
PRB_API int prb_roipool3d(int B, int N, int M, int C, int S, const float *xyz, const float *boxes3d,
                  const float *pts_feature, float *pooled, int *empty_flag,
                  const float *rois_canonical, void *stream);
/* two-pass form (what the Python mirror calls): pass A reads a scene's points once per tile of boxes and writes the
 * per-box index lists into caller scratch (prb_roipool3d_workspace_bytes), pass B streams the pooled rows with
 * 128-bit stores.  zero_fill_empty != 0: the kernel zeroes the rows of empty boxes itself, so `pooled` may be
 * uninitialised (saves the caller's 558 MB memset at C4); 0: untouched, as the reference leaves them. */
PRB_API size_t prb_roipool3d_workspace_bytes(int B, int N, int M, int S);
PRB_API int prb_roipool3d_ws(int B, int N, int M, int C, int S, const float *xyz, const float *boxes3d,
                     const float *pts_feature, float *pooled, int *empty_flag, const float *rois_canonical,
                     int zero_fill_empty, void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------ iou3d_cuda ----------
 * replaces lib/utils/iou3d/src/iou3d.cpp:31-71 (matrices) and :73-170 (NMS) */
PRB_API int prb_boxes_overlap_bev(int num_a, const float *boxes_a, int num_b, const float *boxes_b,
                          float *ans_overlap, void *stream);
PRB_API int prb_boxes_iou_bev(int num_a, const float *boxes_a, int num_b, const float *boxes_b,
                      float *ans_iou, void *stream);

/* fused 3D IoU: what iou3d_utils.boxes_iou3d_gpu (lib/utils/iou3d/iou3d_utils.py:21-53) computes with two BEV
 * conversions, the overlap kernel and ~12 torch ops, in ONE launch and with the same fp32 roundings.
 * prb_boxes_iou3d: boxes_a (batch,na,7), boxes_b (batch,nb,7) [x,y,z,h,w,l,ry] -> out (batch,na,nb): all (RoI x GT)
 * pairs of a batch at once (lib/rpn/proposal_target_layer.py:104 calls the reference once per scene).
 * prb_boxes_iou3d_aligned: out[k] = IoU3D(boxes_a[k], boxes_b[k]) -- the aug loop's 1x1 calls (:232), batched. */
PRB_API int prb_boxes_iou3d(int batch, int na, const float *boxes_a, int nb, const float *boxes_b, float *out, void *stream);
PRB_API int prb_boxes_iou3d_aligned(int n, const float *boxes_a, const float *boxes_b, float *out, void *stream);

/* scratch for one NMS call over n boxes */
PRB_API size_t prb_nms_workspace_bytes(int n);
/* device-resident NMS: boxes (n,5) score-sorted; keep_dev (n) int64 kept positions in order;
 * num_dev (1) int32.  normal != 0 selects the axis-aligned IoU (nms_normal_gpu). No host sync. */
PRB_API int prb_nms_device(const float *boxes, int n, float thresh, int normal, long long *keep_dev,
                   int *num_dev, void *workspace, void *stream);
/* reference signature (keep on the HOST, count returned): runs prb_nms_device, then one small
 * D2H of (count + kept indices) and a stream synchronise.  *num_out = number kept. */
PRB_API int prb_nms_host(const float *boxes, int n, float thresh, int normal, long long *keep_host,
                 int *num_out, void *workspace, void *stream);
/* suppression bitmask only (n, ceil(n/64)) uint64, upper-triangle tiles; lower tiles zero */
PRB_API int prb_nms_mask(const float *boxes, int n, float thresh, int normal, unsigned long long *mask,
                 void *stream);

/* ------------------------------------------------------------------ input pipeline / KITTI output ------
 * SURVEY.md 8(f) rank 4: lib/datasets/kitti_rcnn_dataset.py:246-394 (get_rpn_sample, generate_rpn_training_labels)
 * and tools/eval_rcnn.py:69-94 (save_kitti_format), batched on the device.  A batch of raw scans is RAGGED:
 * lidar (total, stride>=3[,intensity]) holds the scenes back to back, offsets (b+1) int32 (device) delimits them. */

/* calib (b,32) per scene: M[12] (4x3 row-major, rect = [x y z 1].M with M = V2C^T.R0^T, calibration.py:51-59),
 * P2[12] (3x4 row-major), image height, image width, range box x0,x1,y0,y1,z0,z1 (PC_AREA_SCOPE; read if use_range).
 * rect (total,3): rectified coordinates of EVERY point; flags (total) uint8: bit 0 = valid (projects into the image,
 * depth >= 0, inside the range box: get_valid_flag, kitti_rcnn_dataset.py:198-219), bit 1 = near (rect z < 40 m);
 * counts (b,2) int32 or NULL: valid points, valid far points per scene. */
PRB_API int prb_kitti_prepare_points(int b, int total, const int *offsets, const float *lidar, int stride, const float *calib,
                             int use_range, float *rect, unsigned char *flags, int *counts, void *stream);
/* the npoints draw of kitti_rcnn_dataset.py:285-303 per scene, on the device: every valid far point + a random subset
 * (without replacement) of the valid near points, or every valid point + random extra copies when there are fewer
 * than npoints, in random order.  choice (b,npoints) int32 indexes the scene's RAW points.  Counter-based hashes of
 * (seed, scene, point) replace np.random: same distribution, not the same stream.  cand_scratch (total) int32.
 * status (b) int32 or NULL: 1 = scene without a valid point (rows zero).  npoints <= 16384. */
PRB_API int prb_kitti_draw_points(int b, int total, const int *offsets, const unsigned char *flags, int npoints, unsigned seed,
                          int *cand_scratch, int *choice, int *status, void *stream);
/* rows of the network input: rect[choice] (+ intensity - 0.5 when channels == 4), with the scene's augmentation
 * (aug (b,4) DOUBLE: cos, sin of the y rotation, scale, flip 0/1, applied in the order of data_augmentation,
 * kitti_rcnn_dataset.py:526-568; NULL = none); rows of scenes with status != 0 are zero.  Any of pts_input (b,npoints,channels), pts_rect (b,npoints,3),
 * intensity (b,npoints) may be NULL. */
PRB_API int prb_kitti_gather_points(int b, int npoints, const int *offsets, const float *rect, const float *lidar, int stride,
                            const int *choice, const double *aug, const int *status, int channels, float *pts_input,
                            float *pts_rect, float *intensity, void *stream);
/* generate_rpn_training_labels (kitti_rcnn_dataset.py:355-391) for a batch: pts_rect (b,n,3), gt_boxes3d (b,g,7),
 * gt_count (b) or NULL (then all-zero rows of a padded batch are skipped) -> cls_label (b,n) int32 in {1,0,-1},
 * reg_label (b,n,7) [dx,dy,dz,h,w,l,ry].  Boxes are visited in order and later boxes overwrite, as in the reference;
 * the inside test is exact box geometry instead of a Delaunay triangulation of the corners.  g <= 128. */
PRB_API int prb_rpn_training_labels(int b, int n, int g, const float *pts_rect, const float *gt_boxes3d, const int *gt_count,
                            float extra_width, int *cls_label, float *reg_label, void *stream);
/* save_kitti_format's arithmetic (eval_rcnn.py:69-82, calibration.py:106-124): boxes3d (n,7) -> img_boxes (n,4) clipped
 * to the image, alpha (n), valid (n) int32 (box narrower / lower than 0.8 of the image). */
PRB_API int prb_kitti_image_boxes(int n, const float *boxes3d, const float *P2, float img_h, float img_w, float *img_boxes,
                          float *alpha, int *valid, void *stream);
/* the same for a batch: boxes3d (b,m,7), scene k with its own P2 (b,12) and image size img_hw (b,2) [height, width] */
PRB_API int prb_kitti_image_boxes_batch(int b, int m, const float *boxes3d, const float *P2, const float *img_hw, float *img_boxes,
                                float *alpha, int *valid, void *stream);
/* HOST function: the text of one KITTI result file (eval_rcnn.py:85-94) from host arrays; returns the bytes needed
 * (without terminator), writes at most cap bytes. */
PRB_API size_t prb_kitti_format_detections(const char *cls_name, int n, const float *boxes3d, const float *img_boxes,
                                   const float *alpha, const float *scores, const int *valid, char *buf, size_t cap);

#ifdef __cplusplus
}
#endif
#endif /* POINTRCNN_B200_H_ */
