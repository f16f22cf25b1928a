/*
 * b2r.h -- C ABI of libb2r.so: the B200-native (sm_100a) PointNet++ set-abstraction ops.
 *
 * This is the drop-in boundary for the reference's pybind module `pointnet2._ext`
 * (/root/reference/detection/Votenet/pointnet2/_ext_src/src/bindings.cpp:11-24).  Every entry
 * point below replaces one `at::Tensor`-level function of that module; the file:line it
 * replaces is cited on each declaration (paths relative to .../pointnet2/_ext_src/).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes.  All data pointers are DEVICE pointers on the
 *     current CUDA device, contiguous, float32 / int32 -- exactly what the reference's
 *     CHECK_CONTIGUOUS / CHECK_IS_FLOAT / CHECK_IS_INT macros (include/utils.h:10-30) demand.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Launches are
 *     asynchronous on that stream, no host synchronisation, re-entrant, no global state
 *     (the reference launches on at::cuda::getCurrentCUDAStream(), e.g. sampling_gpu.cu:30-31).
 *   - Outputs are fully written by the callee (including the zero fill the reference gets from
 *     torch::zeros, e.g. ball_query.cpp:24-26, sampling.cpp:57-59): callers may pass
 *     uninitialised memory.
 *   - Return value: B2R_OK (0) or a negative b2r_status.  Never exit()s -- unlike the
 *     reference's CUDA_CHECK_ERRORS (include/cuda_utils.h:35-44).  b2r_last_error() gives a
 *     thread-local human-readable detail string for the last failing call.
 *   - 64-bit offset arithmetic throughout (the reference uses 32-bit int offsets,
 *     group_points_gpu.cu:19-21); every single dimension must still fit in int32.
 */
#ifndef B2R_H_
#define B2R_H_

#if defined(__GNUC__)
#define B2R_API __attribute__((visibility("default")))
#else
#define B2R_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef enum b2r_status {
  B2R_OK = 0,
  B2R_ERR_INVALID_ARG = -1, /* null pointer, negative size, misaligned buffer */
  B2R_ERR_CUDA = -2,        /* a CUDA runtime call / kernel launch failed */
  B2R_ERR_UNSUPPORTED = -3  /* size outside what the kernels support */
} b2r_status;

/* library version (major*10000 + minor*100 + patch) and error helpers */
B2R_API int b2r_version(void);
B2R_API const char *b2r_status_string(int status);
B2R_API const char *b2r_last_error(void);
/* sizeof() of the descriptor structs as THIS build of the library sees them (0: b2r_sa_layer,
 * 1: b2r_sa_layer_bwd_desc, 2: b2r_dense_layer, 3: b2r_dense_layer_bwd, 4: b2r_adam_desc; -1 otherwise): lets a binding in another language verify its mirror
 * of the struct layout before the first launch (tests/test_capi_symbols.py does). */
B2R_API int b2r_struct_bytes(int which);

/* The reference's power-of-two thread-count rule (include/cuda_utils.h:20-24).  Exposed because
 * it fixes the FPS tie order (see b2r_fps) and callers/tests may want to inspect it. */
B2R_API int b2r_ref_block_threads(int work_size);

/* ------------------------------------------------------------------------------------------
 * furthest_point_sampling(points, nsamples)            src/sampling.cpp:70-91,
 *                                                       kernel src/sampling_gpu.cu:74-178
 * xyz (B,N,3) f32  ->  idx (B,npoint) i32.  idx[b,0] = 0; bit-exact with the reference,
 * including the |p|^2 <= 1e-3 exclusion (sampling_gpu.cu:105-106) and the winner among exactly
 * equal distances (which in the reference is decided by its 512-lane strided scan + shared-memory
 * tree, sampling_gpu.cu:64-70,113-173).  No global scratch is needed: the running min-distances
 * live in registers across a thread-block cluster.
 */
B2R_API int b2r_fps(const float *xyz, int B, int N, int npoint, int *idx, void *stream);

/* Same sampling, same indices, with the caller choosing how many SMs a scene may hold:
 * cluster_hint = 0 picks the lowest-latency cluster (b2r_fps); 1..16 asks for that many CTAs per
 * scene (raised only as far as the register-resident capacity needs).  A narrow cluster is for
 * FPS that runs BESIDE other kernels -- the geometry pre-pass of the next batch on a side stream
 * (backbone_module.Pointnet2Backbone.geometry_prepass) -- where it is off the critical path. */
B2R_API int b2r_fps_ex(const float *xyz, int B, int N, int npoint, int *idx, int cluster_hint,
                       void *stream);

/* The same sampling on spatially sorted buckets (csrc/fps_bucket.cu) -- the variant the Python
 * shim calls.  Points are first ordered by a Morton cell code (one counting sort per scene); every
 * warp owns a compact bucket with its bounding box and SKIPS an iteration's distance updates when
 * the new sample is provably too far to lower any of its running min-distances (the bound is
 * evaluated with the reference's own rounding sequence, so only updates that would change nothing
 * are skipped: indices stay bit-identical to b2r_fps and to the reference).  Warps exchange
 * candidates in one DSMEM hop into a table replicated in every CTA of the scene's cluster.
 * workspace: b2r_fps_workspace_bytes(B,N) bytes of device memory (the sorted order), caller-owned
 * so the call allocates nothing (CUDA-graph capturable).  cluster_hint as in b2r_fps_ex. */
B2R_API long long b2r_fps_workspace_bytes(int B, int N);
B2R_API int b2r_fps_ws(const float *xyz, int B, int N, int npoint, int *idx, int cluster_hint,
                       void *workspace, long long workspace_bytes, void *stream);
/* The two halves of b2r_fps_ws separately: the sort depends on xyz alone, so a caller that knows its
 * next batch early (the pipelined training step) can run it ahead of time and keep only the
 * sampling itself on its dependency chain.  b2r_fps_sort is a no-op for scenes of <= 4096 points. */
B2R_API int b2r_fps_sort(const float *xyz, int B, int N, void *workspace, long long workspace_bytes,
                         void *stream);
B2R_API int b2r_fps_ws_presorted(const float *xyz, int B, int N, int npoint, int *idx, int cluster_hint,
                                 void *workspace, long long workspace_bytes, void *stream);

/* Launch geometry b2r_fps would use for (B,N): cluster size, threads per CTA, points per thread
 * and dynamic shared memory bytes.  Any out pointer may be NULL. */
B2R_API int b2r_fps_plan(int B, int N, int *cluster_size, int *threads, int *points_per_thread,
                 int *smem_bytes);

/* ------------------------------------------------------------------------------------------
 * gather_points(points, idx)                            src/sampling.cpp:20-43,
 *                                                       kernel src/sampling_gpu.cu:13-25
 * features (B,C,N) f32, idx (B,M) i32  ->  out (B,C,M):  out[b,c,j] = features[b,c,idx[b,j]]
 */
B2R_API int b2r_gather_fwd(const float *features, const int *idx, int B, int C, int N, int M, float *out,
                   void *stream);

/* gather_points_grad(grad_out, idx, n)                  src/sampling.cpp:45-69,
 *                                                       kernel src/sampling_gpu.cu:39-52
 * grad_out (B,C,M), idx (B,M)  ->  grad_features (B,C,N) = scatter-add into zeros */
B2R_API int b2r_gather_bwd(const float *grad_out, const int *idx, int B, int C, int N, int M,
                   float *grad_features, void *stream);

/* ------------------------------------------------------------------------------------------
 * ball_query(new_xyz, xyz, radius, nsample)             src/ball_query.cpp:13-37,
 *                                                       kernel src/ball_query_gpu.cu:14-49
 * new_xyz (B,M,3), xyz (B,N,3)  ->  idx (B,M,nsample) i32: the first `nsample` point indices k
 * (ascending) with fma(dz,dz,fma(dx,dx,dy*dy)) < radius*radius; slots past the count repeat the
 * first hit; an empty ball yields zeros.  Bit-exact with the reference.
 */
B2R_API int b2r_ball_query(const float *new_xyz, const float *xyz, int B, int N, int M, float radius,
                   int nsample, int *idx, void *stream);

/* Same result, bit for bit, through a hashed uniform grid (cell = radius): a centre visits the 27
 * cells around it instead of all N points, collects the hits and sorts them by index.  Needs a
 * caller-provided device workspace of b2r_ball_query_workspace_bytes(B, N) bytes (contents are
 * scratch).  Falls back to b2r_ball_query for N < 1024 or nsample > 480. */
B2R_API long long b2r_ball_query_workspace_bytes(int B, int N);
B2R_API int b2r_ball_query_grid(const float *new_xyz, const float *xyz, int B, int N, int M,
                                float radius, int nsample, int *idx, void *workspace,
                                long long workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------
 * group_points(points, idx)                             src/group_points.cpp:17-40,
 *                                                       kernel src/group_points_gpu.cu:13-33
 * features (B,C,N), idx (B,NP,NS)  ->  out (B,C,NP,NS)
 */
B2R_API int b2r_group_fwd(const float *features, const int *idx, int B, int C, int N, int NP, int NS,
                  float *out, void *stream);

/* group_points_grad(grad_out, idx, n)                   src/group_points.cpp:42-65,
 *                                                       kernel src/group_points_gpu.cu:48-69
 * grad_out (B,C,NP,NS), idx (B,NP,NS)  ->  grad_features (B,C,N) */
B2R_API int b2r_group_bwd(const float *grad_out, const int *idx, int B, int C, int N, int NP, int NS,
                  float *grad_features, void *stream);

/* ------------------------------------------------------------------------------------------
 * three_nn(unknowns, knows)                             src/interpolate.cpp:19-45,
 *                                                       kernel src/interpolate_gpu.cu:14-64
 * unknown (B,n,3), known (B,m,3)  ->  dist2 (B,n,3) f32 (SQUARED distances, ascending),
 * idx (B,n,3) i32.  Strict '<' insertion: the earlier index wins ties.  m<3 leaves +inf / 0.
 */
B2R_API int b2r_three_nn(const float *unknown, const float *known, int B, int n, int m, float *dist2,
                 int *idx, void *stream);

/* three_interpolate(points, idx, weight)                src/interpolate.cpp:47-75,
 *                                                       kernel src/interpolate_gpu.cu:77-106
 * features (B,C,m), idx (B,n,3), weight (B,n,3)  ->  out (B,C,n) */
B2R_API int b2r_three_interp_fwd(const float *features, const int *idx, const float *weight, int B, int C,
                         int m, int n, float *out, void *stream);

/* three_interpolate_grad(grad_out, idx, weight, m)      src/interpolate.cpp:76-104,
 *                                                       kernel src/interpolate_gpu.cu:121-148
 * grad_out (B,C,n)  ->  grad_features (B,C,m) */
B2R_API int b2r_three_interp_bwd(const float *grad_out, const int *idx, const float *weight, int B, int C,
                         int n, int m, float *grad_features, void *stream);

/* ------------------------------------------------------------------------------------------
 * Deterministic, atomic-free backward of grouping / three_interpolate (csrc/movers_staged.cu).
 * The reference scatters with atomicAdd (group_points_gpu.cu:48-69, interpolate_gpu.cu:121-148):
 * the L2 atomic units cap that at a few percent of the HBM roofline and the sum order changes
 * from run to run.  Here the index is inverted once per index tensor into a plan (entries sorted
 * by target, each list by entry id) and every (b,c) row is gathered from shared-memory staged
 * tiles of grad_out in that fixed order: bit-identical results across runs, no memset.
 *   entries = NP*NS with entries_per_source = 1 (grouping: idx (B,NP,NS), targets in [0,N))
 *   entries = 3*n   with entries_per_source = 3 (three_interpolate: idx (B,n,3), targets in [0,m),
 *             weight (B,n,3) is permuted into the plan; pass NULL for grouping)
 * plan: b2r_scatter_plan_bytes(...) bytes of device memory, caller-owned. */
B2R_API long long b2r_scatter_plan_bytes(int B, long long entries, int N, int entries_per_source,
                                         int weighted);
B2R_API int b2r_scatter_plan(const int *idx, const float *weight, int B, long long entries, int N,
                             int entries_per_source, void *plan, long long plan_bytes, void *stream);
/* group_points_grad through a plan of idx (B,NP,NS): grad_out (B,C,NP,NS) -> grad_features (B,C,N) */
B2R_API int b2r_group_bwd_plan(const float *grad_out, const void *plan, int B, int C, int N, int NP,
                               int NS, float *grad_features, void *stream);
/* three_interpolate_grad through a plan of (idx, weight): grad_out (B,C,n) -> grad_features (B,C,m) */
B2R_API int b2r_three_interp_bwd_plan(const float *grad_out, const void *plan, int B, int C, int n,
                                      int m, float *grad_features, void *stream);

/* ------------------------------------------------------------------------------------------
 * Fused QueryAndGroup tail (reference Python: pointnet2_utils.py:347-366, i.e. two
 * grouping_operation calls + in-place `-= new_xyz` + `/= radius` + torch.cat, five HBM passes)
 * in ONE pass:
 *   out[b, 0:3,  j, s] = (xyz[b, idx[b,j,s], :] - new_xyz[b, j, :]) (/ radius if normalize)
 *   out[b, 3:3+C,j, s] = features[b, :, idx[b,j,s]]            (C may be 0, features NULL)
 * xyz (B,N,3), new_xyz (B,NP,3), features (B,C,N) or NULL, idx (B,NP,NS) -> out (B,3+C,NP,NS).
 * The division is a true IEEE division by `radius` as in the reference.
 */
B2R_API int b2r_query_group_fwd(const float *xyz, const float *new_xyz, const float *features,
                        const int *idx, int B, int C, int N, int NP, int NS, float radius,
                        int normalize_xyz, float *out, void *stream);

/* Backward of the above.  grad_out (B,3+C,NP,NS).  Any of the three outputs may be NULL
 * (= that input needs no gradient).  grad_xyz (B,N,3), grad_new_xyz (B,NP,3),
 * grad_features (B,C,N); all fully written (zero-filled then accumulated). */
B2R_API int b2r_query_group_bwd(const float *grad_out, const int *idx, int B, int C, int N, int NP, int NS,
                        float radius, int normalize_xyz, float *grad_xyz, float *grad_new_xyz,
                        float *grad_features, void *stream);


/* ------------------------------------------------------------------------------------------
 * Fused SharedMLP layer of a set-abstraction block on tcgen05 tensor cores (csrc/mlp.cu).
 *
 * Replaces, inside PointnetSAModuleVotes.forward (reference pointnet2_modules.py:245-267), the
 * library chain  QueryAndGroup -> [cuDNN 1x1 Conv2d -> BatchNorm2d -> ReLU] x3 -> max_pool2d
 * (reference pytorch_utils.py:11-36,67-120).  ONE call runs ONE conv layer as a TF32 GEMM
 *     z[position, co] = sum_k W[co, k] * x[position, k]          positions = B*NP*NS
 * with the memory-bound neighbours fused in:
 *   mode 0      x rows are gathered on the fly: [features(idx) ..., (xyz(idx)-new_xyz)/radius]
 *               (the grouped (B,3+C,NP,NS) tensor is never materialised)
 *   mode 1      x = relu(scale_prev * z_prev + shift_prev)  (previous layer's BatchNorm+ReLU)
 *   epilogue 0  store raw z (M,Cout) position-major + accumulate per-channel sum / sum of squares
 *   epilogue 1  statistics + max AND min of raw z over each centre's NS samples (+ arg indices);
 *               b2r_pool_finalize turns them into max_pool(relu(bn(z))) exactly
 * Weights are passed as the packed image produced by b2r_mlp_pack_weight (TF32-rounded,
 * 128-byte-swizzled K-major shared-memory layout, staged by one TMA bulk copy).
 * Limits: Cout <= 256 per launch (wider layers: the channel slices below), B*NP*NS % 32 == 0
 * (gather layers: NP*NS % 32 == 0), NS in {16,32,64} for epilogue 1; otherwise
 * B2R_ERR_UNSUPPORTED (callers then use the unfused path).
 */
typedef struct b2r_sa_layer {
  int B, N, NP, NS;   /* scenes, source points per scene, centres per scene, samples per centre */
  int Cin, Cout;      /* mode 0: Cin = 3 + feature channels (reference order [xyz, features]) */
  int mode, epilogue;
  const float *xyz;      /* mode 0: (B,N,3) */
  const float *new_xyz;  /* mode 0: (B,NP,3) */
  const float *feat_t;   /* mode 0: (B,N,Cin-3) POINT-major features, NULL when Cin == 3 */
  const int *idx;        /* mode 0: (B,NP,NS) ball-query indices */
  float radius;
  int normalize_xyz;
  const float *z_prev;      /* mode 1: (M,Cin) raw conv output of the previous layer */
  const float *scale_prev;  /* mode 1: (Cin) */
  const float *shift_prev;  /* mode 1: (Cin) */
  const float *w_image;     /* from b2r_mlp_pack_weight(w, Cout, Cin, mode == 0) */
  float *z;                 /* epilogue 0: (M,Cout) */
  double *stats;            /* (2,Cout) sum, sum of squares; ACCUMULATED (caller zeroes); may be NULL */
  float *zmax, *zmin;       /* epilogue 1: (B*NP,Cout) */
  int *amax, *amin;         /* epilogue 1: (B*NP,Cout) sample index in [0,NS) */
  int sm_limit;             /* 0 = one CTA on every SM; else at most this many CTAs, leaving the
                               other SMs to kernels on concurrent streams (geometry pre-pass) */
  /* Pad-free position space from b2r_compact_plan (all three, or all NULL).  When set, a
   * "position" is an entry of the plan instead of (b, centre, sample): mode 0 gathers through
   * cidx / ccen instead of idx, z / z_prev hold b2r_compact_capacity(B,NP,NS) rows, statistics
   * weight every centre's first sample by 1 + (NS - class size) so they equal the padded sums,
   * and the number of tiles is read from cmeta on the device.  amax / amin are then sample
   * indices inside the centre's class-size run (consistent with b2r_sa_layer_bwd). */
  const int *cidx, *ccen, *cmeta;
  /* Channel slice (all zero = the whole layer in one launch).  A layer too large for one launch
   * runs as the grid of launches b2r_sa_layer_fwd_slices gives; each launch covers output channels
   * [co0, co0 + co_n) (co_n = 0: all) and, for gather layers, feature channels [ci0, ci0 + ci_n)
   * (ci_n = 0: all; ci0 and ci_n multiples of 8).  Cin / Cout stay the WHOLE layer's; z, stats,
   * zmax/zmin/amax/amin keep the whole layer's pitch and the launch writes its own columns.
   * w_image packs the slice's weight: rows co0.., columns [xyz, features ci0..ci0+ci_n), with the
   * xyz columns ZERO unless ci0 == 0 (b2r_mlp_pack_weight(w_slice, co_n, 3 + ci_n, 1, ...)).
   * accumulate != 0 (epilogue 0 only): z += this launch's partial product instead of z = ...; the
   * feature slices of one output slice run in increasing ci0 order, the first with accumulate = 0,
   * and only the last passes stats (they are sums over the finished z). */
  int co0, co_n, ci0, ci_n, accumulate;
} b2r_sa_layer;

B2R_API long long b2r_mlp_weight_image_bytes(int Cout, int Cin, int gather);
/* w (Cout,Cin) row-major fp32 = nn.Conv2d(Cin,Cout,1).weight; gather != 0 for mode-0 layers */
B2R_API int b2r_mlp_pack_weight(const float *w, int Cout, int Cin, int gather, float *image,
                                void *stream);
B2R_API int b2r_sa_layer_fwd(const b2r_sa_layer *desc, void *stream);
/* 1 when b2r_sa_layer_fwd covers a layer of this shape, in one launch or in the channel slices of
 * b2r_sa_layer_fwd_slices, 0 otherwise (same rules as the launch). */
B2R_API int b2r_sa_layer_fwd_supported(int B, int NP, int NS, int Cin, int Cout, int gather,
                                       int pooled);

/* Slice grid of a layer (depends on the channel counts only): returns the number of launches
 * (0 = not covered; 1 = the whole layer, *co_step = Cout and *ci_step = 0).  Output slices are
 * [j*co_step, min(Cout, (j+1)*co_step)); gather layers may also be cut into feature slices
 * [i*ci_step, min(Cin-3, (i+1)*ci_step)) (ci_step = 0: none).  Launch order: output slice by
 * output slice, feature slices in increasing order inside each. */
B2R_API int b2r_sa_layer_fwd_slices(int Cin, int Cout, int gather, int pooled, int *co_step,
                                    int *ci_step);

/* Positions per tile the launch would use for a layer of this shape (0 = unsupported); compact:
 * with a b2r_compact_plan.  Diagnostic (DESIGN.md tile table, tests). */
B2R_API int b2r_sa_layer_fwd_tile(int B, int NP, int NS, int Cin, int Cout, int gather, int pooled,
                                  int compact);

/* BatchNorm bookkeeping from accumulated statistics (replaces the statistics half of
 * nn.BatchNorm2d in training mode, reference pytorch_utils.py:55-58): scale = gamma*invstd,
 * shift = beta - mean*scale; running stats updated with `momentum` (unbiased variance) when
 * running_mean/var are non-NULL (both or neither, else B2R_ERR_INVALID_ARG);
 * *num_batches_tracked (int64, may be NULL) is incremented.
 * mean_out / invstd_out (C) are optional (saved for backward). */
B2R_API int b2r_bn_finalize(const double *stats, int C, double count, const float *gamma,
                            const float *beta, float eps, float momentum, float *running_mean,
                            float *running_var, float *scale, float *shift, float *mean_out,
                            float *invstd_out, long long *num_batches_tracked, void *stream);

/* b2r_bn_finalize with the momentum in device memory (one float), read when the kernel runs: a
 * captured CUDA graph then follows a momentum written between replays.  Same validation, plus
 * B2R_ERR_INVALID_ARG when running_mean/var are given and `momentum` is NULL. */
B2R_API int b2r_bn_finalize_dev(const double *stats, int C, double count, const float *gamma,
                                const float *beta, float eps, const float *momentum,
                                float *running_mean, float *running_var, float *scale,
                                float *shift, float *mean_out, float *invstd_out,
                                long long *num_batches_tracked, void *stream);

/* out = relu(scale*(scale>=0 ? zmax : zmin) + shift): (B,C,NP) channel-major (reference layout)
 * and/or (B,NP,C) point-major (the next layer's gather source).  Either output may be NULL. */
B2R_API int b2r_pool_finalize(const float *zmax, const float *zmin, const float *scale,
                              const float *shift, int B, int NP, int C, float *out_cm,
                              float *out_pm, void *stream);

/* (B,C,N) channel-major -> (B,N,C) point-major */
B2R_API int b2r_to_point_major(const float *in, int B, int C, int N, float *out, void *stream);

/* ------------------------------------------------------------------------------------------
 * Backward of the fused SharedMLP block (csrc/mlp_bwd.cu).  Replaces what autograd runs for
 * PointnetSAModuleVotes' MLP + pooling (reference pointnet2_modules.py:245-267): max_pool2d
 * backward, 3 x [ReLU backward, cuDNN BatchNorm backward, cuDNN dgrad + wgrad], torch.cat /
 * div / sub backward and two group_points_grad scatters (src/group_points_gpu.cu:48-69).
 *
 *   b2r_pool_bwd_prep      grad of the pooled output -> the ONE sample per (centre, channel) it
 *                          reaches (dysel, asel) + BatchNorm-backward sums of the top layer
 *   b2r_bn_bwd_finalize    sums -> per-channel coefficients of dz = a*gr + b*z + c, dgamma, dbeta
 *   b2r_sa_layer_bwd       ONE layer (BF16 operands, FP32 accumulate): dW (+)= dz^T x  and
 *                          gr_prev = (dz W) * relu-mask with the next BatchNorm-backward sums
 *                          (dense layers), or the scatter-add of dz W into the point-major
 *                          feature / xyz gradients (gather layer).  For the pooled top layer z is
 *                          recomputed inside the kernel (the forward never stored it).
 */
typedef struct b2r_sa_layer_bwd_desc {
  int B, N, NP, NS;
  int Cin, Cout;            /* of THIS layer (mode 0: Cin = 3 + feature channels) */
  int mode;                 /* 0: gather layer (layer 0), 1: dense layer */
  /* the layer's input, recomputed exactly like the forward prologue */
  const float *xyz, *new_xyz, *feat_t;
  const int *idx;
  float radius;
  int normalize_xyz;
  const float *z_prev, *scale_prev, *shift_prev; /* mode 1 */
  const void *w_image_bf16; /* b2r_mlp_pack_weight_bf16 image; NULL only when neither dgrad nor
                               the top-layer recomputation is needed */
  /* the layer's output gradient, one of three forms: */
  const float *dz;          /* (a) dz (M,Cout) given directly, or NULL */
  const float *gr, *z;      /* (b) dense: gr = dL/d(bn output, ReLU-masked) and z, (M,Cout) each */
  const float *dysel;       /* (c) pooled top layer: routed output gradient (B*NP,Cout) ... */
  const int *asel;          /*     ... and the sample it reaches, from b2r_pool_bwd_prep; z is
                                   recomputed on the tensor cores */
  const float *coef_a, *coef_b, *coef_c; /* (b),(c): dz = a*g + b*z + c, b2r_bn_bwd_finalize */
  /* outputs */
  float *dW;                /* (Cout,Cin) nn.Conv2d layout; ACCUMULATED (caller zeroes) */
  float *gr_prev;           /* mode 1: (M,Cin) ReLU-masked gradient of the layer below */
  double *stats_prev;       /* mode 1: (2,Cin) sum(gr_prev), sum(gr_prev*z_prev); ACCUMULATED */
  float *g_feat_t;          /* mode 0: (B,N,Cin-3) point-major, ACCUMULATED; NULL = not needed */
  float *g_xyz;             /* mode 0: (B,N,3) ACCUMULATED; NULL = not needed */
  float *g_new_xyz;         /* mode 0: (B,NP,3) ACCUMULATED; NULL = not needed */
  int sm_limit;             /* as b2r_sa_layer.sm_limit: 0 = every SM, else at most this many CTAs */
  const int *cidx, *ccen, *cmeta; /* as b2r_sa_layer: the forward's plan (gr, z, z_prev, gr_prev
                               are then in its position space; gradients carry the positions'
                               multiplicities, see csrc/compact.cu) */
  /* Channel slice, as b2r_sa_layer (all zero = the whole layer; grid from
   * b2r_sa_layer_bwd_slices).  dz / gr / z / dysel / asel keep the whole layer's pitch (Cout) and
   * coef_a/b/c the whole layer's length; the launch reads its output channels [co0, co0 + co_n)
   * and adds rows co0.. (and, gather layers, the columns of its feature slice) of dW.  A feature
   * slice computes the gradient of its own feature channels; the xyz / centre gradients belong to
   * the slice with ci0 == 0 (g_xyz, g_new_xyz are ignored by the others).
   * accumulate != 0 (dense layers only): gr_prev += this slice's (dz W) * mask instead of
   * gr_prev = ...; every output slice after the first passes it, and all add their partial
   * BatchNorm-backward sums into stats_prev.  Gather layers always scatter-add, so the flag is
   * rejected there (B2R_ERR_INVALID_ARG). */
  int co0, co_n, ci0, ci_n, accumulate;
} b2r_sa_layer_bwd_desc;

B2R_API long long b2r_mlp_weight_bf16_image_bytes(int Cout, int Cin, int gather);
B2R_API int b2r_mlp_pack_weight_bf16(const float *w, int Cout, int Cin, int gather, void *image,
                                     void *stream);
B2R_API int b2r_sa_layer_bwd(const b2r_sa_layer_bwd_desc *desc, void *stream);
/* 1 when b2r_sa_layer_bwd covers a layer of this shape (shared memory, TMEM columns, divisibility),
 * 0 otherwise: lets the host decide BEFORE the forward whether to take the fused path. */
B2R_API int b2r_sa_layer_bwd_supported(int B, int NP, int NS, int Cin, int Cout, int gather,
                                       int top);
/* Slice grid of the backward, as b2r_sa_layer_fwd_slices (sized for dgrad on). */
B2R_API int b2r_sa_layer_bwd_slices(int Cin, int Cout, int gather, int top, int *co_step,
                                    int *ci_step);

B2R_API int b2r_sa_layer_bwd_tile(int B, int NP, int NS, int Cin, int Cout, int gather, int top,
                                  int dgrad, int compact);

/* dout_cm (B,C,NP) and/or dout_pm (B,NP,C) (summed; either may be NULL) -> dysel (B*NP,C),
 * asel (B*NP,C), stats (2,C) double ACCUMULATED: sum(dysel), sum(dysel * zsel). */
B2R_API int b2r_pool_bwd_prep(const float *dout_cm, const float *dout_pm, const float *zmax,
                              const float *zmin, const int *amax, const int *amin,
                              const float *scale, const float *shift, int B, int NP, int C,
                              float *dysel, int *asel, double *stats, void *stream);

/* stats (2,C) = sum(gr), sum(gr*z) over `count` positions -> coefficients of
 * dz = coef_a*gr + coef_b*z + coef_c (training != 0: batch statistics; 0: running statistics),
 * the epilogue-2 form (k1,k2,gs), and dgamma / dbeta.  Any output may be NULL. */
B2R_API int b2r_bn_bwd_finalize(const double *stats, int C, double count, const float *gamma,
                                const float *mean, const float *invstd, int training,
                                float *coef_a, float *coef_b, float *coef_c, float *k1, float *k2,
                                float *gs, float *dgamma, float *dbeta, void *stream);
/* The same with one more output: dbias_conv (C) = sum over positions of dz, the gradient of a bias
 * the convolution added in front of this BatchNorm (nn.Conv1d(bias=True) -> BatchNorm1d in the
 * voting / proposal heads).  NULL = not needed. */
B2R_API int b2r_bn_bwd_finalize_ex(const double *stats, int C, double count, const float *gamma,
                                   const float *mean, const float *invstd, int training,
                                   float *coef_a, float *coef_b, float *coef_c, float *k1,
                                   float *k2, float *gs, float *dgamma, float *dbeta,
                                   float *dbias_conv, void *stream);

/* ------------------------------------------------------------------------------------------
 * Pad-free position space of a set-abstraction block (csrc/compact.cu).
 *
 * The reference's ball query pads a centre's unused slots with copies of its first hit
 * (src/ball_query_gpu.cu:38-46) and QueryAndGroup + SharedMLP + max_pool2d
 * (pointnet2_modules.py:245-267) then compute every copy.  A copy has the same activations as
 * sample 0 in every layer, so the fused block may compute each centre on its first
 * u = 8/16/32/64 >= cnt samples only (cnt = 1 + last s with idx[s] != idx[0]) and give sample 0
 * the weight 1 + (NS - u) in every sum over positions: same results up to fp32 summation order.
 * b2r_compact_plan orders the centres by (u, centre id) and writes, per position p of that
 * space: cidx[p] = b*N + idx (global source row), ccen[p] = b*NP + j (global centre, -1 = dead
 * padding); meta (16 ints): [0..3] cumulative end of the classes 8/16/32/64 (each padded to a
 * multiple of 128 positions), [4..7] end of the live positions of each class, [8] total
 * positions, [10..13] centres per class.  NS must be 16, 32 or 64.
 * cidx / ccen hold b2r_compact_capacity(B,NP,NS) ints; workspace b2r_compact_workspace_bytes. */
B2R_API long long b2r_compact_capacity(int B, int NP, int NS);
B2R_API long long b2r_compact_workspace_bytes(int B, int NP);
B2R_API int b2r_compact_plan(const int *idx, int B, int N, int NP, int NS, int *cidx, int *ccen,
                             int *meta, void *workspace, void *stream);

/* ------------------------------------------------------------------------------------------
 * Wide 1x1-conv layers on POINT-major tensors (csrc/dense.cu): the SharedMLP of
 * PointnetFPModule (reference pointnet2_modules.py:505-514), VotingModule's conv1..3 + bn1..2
 * (models/voting_module.py:38-65) and ProposalModule's conv1..3 + bn1..2
 * (models/proposal_module.py:115-119), which the reference runs as cuDNN Conv1d/Conv2d +
 * BatchNorm + ReLU on (B,C,n) tensors.  Here a layer is  z (M,Cout) = x (M,Cin) W^T (+ bias)
 * with M = B*n positions, TF32 operands / FP32 accumulate on tcgen05, both operands streamed in
 * 32-deep K chunks; BatchNorm statistics, the previous layer's BatchNorm+ReLU (applied while
 * loading), the ReLU mask and the BatchNorm-backward sums are fused in.  Any Cin, Cout, M.
 *
 * b2r_dense_pack     W (Cout,Cin) row-major -> the swizzled TF32 images the kernels stage by TMA:
 *                    w_img (forward) and / or wt_img (W^T, input gradient); sizes from
 *                    b2r_dense_image_bytes(Cout,Cin) and b2r_dense_image_bytes(Cin,Cout).
 * b2r_dense_fwd      x = in, or relu(in*sc_in + sh_in) when sc_in != NULL; z = x W^T + bias;
 *                    stats (2,Cout) += sum z, sum z^2 (double; NULL = none).
 * b2r_dense_bwd      dz = g (ca == NULL) or ca*g + cb*zz + cc (b2r_bn_bwd_finalize);
 *                    gin (M,Cin) = (dz W) * [in*sc_in + sh_in > 0]  (no mask when sc_in == NULL),
 *                    stats_in (2,Cin) += sum gin, sum gin*in; dW (Cout,Cin) += dz^T x.
 *                    gin and dW are optional (NULL).  sc_in / sh_in / ca / cb / cc must be
 *                    readable up to the next multiple of 4 elements and 16-byte aligned, like the
 *                    rows of in / g / zz (ld % 4 == 0).
 */
typedef struct b2r_dense_layer {
  int M, Cin, Cout;
  const float *in;          /* (M, ld_in) */
  int ld_in;
  const float *sc_in, *sh_in; /* (Cin) or NULL */
  const float *w_img;
  const float *bias;        /* (Cout) or NULL */
  float *z;                 /* (M, ld_z) */
  int ld_z;
  double *stats;            /* (2, Cout) ACCUMULATED, or NULL */
} b2r_dense_layer;

typedef struct b2r_dense_layer_bwd {
  int M, Cin, Cout;
  const float *in;          /* (M, ld_in): the layer's input (before its BatchNorm+ReLU prologue) */
  int ld_in;
  const float *sc_in, *sh_in;
  const float *g, *zz;      /* (M, ld_g) */
  int ld_g;
  const float *ca, *cb, *cc; /* (Cout) or NULL */
  const float *wt_img;
  float *gin;               /* (M, ld_gin) or NULL */
  int ld_gin;
  double *stats_in;         /* (2, Cin) ACCUMULATED, or NULL */
  float *dW;                /* (Cout, Cin) ACCUMULATED, or NULL */
} b2r_dense_layer_bwd;

B2R_API long long b2r_dense_image_bytes(int rows, int k);
B2R_API int b2r_dense_pack(const float *w, int Cout, int Cin, float *w_img, float *wt_img,
                           void *stream);
B2R_API int b2r_dense_fwd(const b2r_dense_layer *desc, void *stream);
B2R_API int b2r_dense_bwd(const b2r_dense_layer_bwd *desc, void *stream);

/* ------------------------------------------------------------------------------------------
 * Point-major glue around the dense layers (csrc/heads.cu).
 *
 * b2r_interp_cat_fwd / _bwd: PointnetFPModule's three_interpolate + torch.cat([interpolated,
 *   skip], dim=1) (reference pointnet2_modules.py:492-504, kernels src/interpolate_gpu.cu:77-148)
 *   in one pass: known (B,m,C2), skip (B,n,C1) or NULL, idx / weight (B,n,3) ->
 *   out (B*n, C2+C1) = [fma(p3,w3, fma(p1,w1, p2*w2)), skip]; backward: g (B*n, ld_g) ->
 *   g_known (B,m,C2) ACCUMULATED (caller zeroes) and g_skip (B*n,C1) written; either may be NULL.
 * b2r_vote_tail_fwd / _bwd: VotingModule's offset / residual split + VoteNet's L2 feature
 *   normalisation (models/voting_module.py:56-64, models/votenet.py:93-94): net (M, ld_net) =
 *   [offset(3), residual(C), pad] -> vote_xyz (M,3) = seed_xyz + offset, out (M,C) = v / |v|_2
 *   with v = seed_feat + residual, norm (M); backward: g_out (M,C) / g_vote_xyz (M,3) (either
 *   may be NULL) -> g_net (M, ld_net) fully written, g_seed_feat (M,C) (may be NULL); the seed
 *   xyz gradient is g_vote_xyz itself. */
B2R_API int b2r_interp_cat_fwd(const float *known, const float *skip, const int *idx,
                               const float *weight, int B, int n, int m, int C2, int C1,
                               float *out, void *stream);
B2R_API int b2r_interp_cat_bwd(const float *g, int ld_g, const int *idx, const float *weight, int B,
                               int n, int m, int C2, int C1, float *g_known, float *g_skip,
                               void *stream);
B2R_API int b2r_vote_tail_fwd(const float *net, int ld_net, const float *seed_xyz,
                              const float *seed_feat, long long M, int C, float *vote_xyz,
                              float *out, float *norm, void *stream);
B2R_API int b2r_vote_tail_bwd(const float *g_out, const float *g_vote_xyz, const float *out,
                              const float *norm, long long M, int C, int ld_net, float *g_net,
                              float *g_seed_feat, void *stream);

/* ------------------------------------------------------------------------------------------
 * Loss-side nearest-neighbour matching (SURVEY 8f row 4): the two arg-min vectors of
 * nn_distance(pc1, pc2)  (reference detection/Votenet/utils/nn_distance.py:34-61) without the
 * four (B,N,M,C) tiled tensors it materialises.  pc1 (B,N,C), pc2 (B,M,C), C <= 4;
 * mode 0: sum d^2, 1: sum |d| (l1=True), 2: sum huber(d, delta) (l1smooth=True).
 * idx1 (B,N) / idx2 (B,M) int64 like torch.min's indices (either may be NULL); lowest index on
 * ties.  The host mirror recomputes the matched distances with torch ops so that autograd
 * routes gradients to the matched pairs exactly like torch.min's backward.
 */
B2R_API int b2r_nn_argmin(const float *pc1, const float *pc2, int B, int N, int M, int C, int mode,
                          float delta, long long *idx1, long long *idx2, void *stream);

/* ------------------------------------------------------------------------------------------
 * Adam over one flat fp32 buffer (csrc/adam.cu) -- the optimizer step at the end of the training
 * step (reference: optim.Adam over net.parameters(), train_Votenet_FSB.py:176-181) as ONE streaming
 * kernel instead of three multi-tensor launches.  params / grads / exp_avg / exp_avg_sq: n floats
 * each, 16-byte aligned; state: b2r_adam_state_bytes() bytes of zero-initialised device memory (the
 * step counter, advanced on the device: graph-replayable).  grads are multiplied by grad_scale
 * first (1/world_size after a sum all-reduce).  torch.optim.Adam arithmetic (amsgrad=False). */
B2R_API int b2r_adam_state_bytes(void);
B2R_API int b2r_adam_flat_step(float *params, const float *grads, float *exp_avg, float *exp_avg_sq,
                               long long n, void *state, float lr, float beta1, float beta2, float eps,
                               float weight_decay, float grad_scale, void *stream);

/* Parameter groups (torch.optim param_groups) of the flat buffer: elements [start, end) with their
 * own learning rate and weight decay.  The table lives in DEVICE memory and is read by every
 * launch, so rates written into it between CUDA-graph replays (a learning-rate schedule) apply to
 * the next replay.  Entries are sorted and disjoint; start is a multiple of 4 and end is a multiple
 * of 4 or n, so that every 16-byte vector of the buffer lies in one group.  Elements outside every
 * group are left untouched. */
#define B2R_ADAM_MAX_GROUPS 64
typedef struct b2r_adam_group {
  long long start, end;
  float lr, weight_decay;
} b2r_adam_group;

/* One Adam / AdamW step over parameter groups (b2r_struct_bytes(4) is sizeof this struct).
 * Buffers as for b2r_adam_flat_step (n floats each, 16-byte aligned; state: the step counter).
 * decoupled = 0: torch.optim.Adam's L2 decay g += wd*p; 1: torch.optim.AdamW's p *= 1 - lr*wd
 * before the moment update.  The gradient is multiplied by grad_scale and then, when clip_coef is
 * not NULL, by the device scalar *clip_coef (b2r_flat_grad_norm's coef_out). */
typedef struct b2r_adam_desc {
  float *params;
  const float *grads;
  float *exp_avg, *exp_avg_sq;
  long long n;
  void *state;
  const b2r_adam_group *groups; /* device table, n_groups entries (1..B2R_ADAM_MAX_GROUPS) */
  int n_groups;
  float beta1, beta2, eps;
  float grad_scale;
  int decoupled;
  const float *clip_coef; /* device scalar or NULL */
} b2r_adam_desc;
B2R_API int b2r_adam_flat_step_groups(const b2r_adam_desc *desc, void *stream);

/* Global L2 norm of grad_scale * grads (n floats, 16-byte aligned) -- torch.nn.utils.
 * clip_grad_norm_(..., max_norm, norm_type=2) without modifying the gradients.  Writes the norm to
 * the device scalar *norm_out and min(max_norm / (norm + 1e-6), 1) to *coef_out (fp32, torch's
 * clip_coef_clamped: a NaN norm gives NaN, an infinite one 0).  Two launches: a fixed grid (its
 * size depends on n only) of fp64 partial sums of squares, then one block that adds the partials
 * in a fixed order.  No atomics: identical gradients give a bit-identical norm.  No host
 * synchronisation: graph-capturable.  workspace: b2r_flat_grad_norm_workspace_bytes(n) bytes of
 * device memory, 16-byte aligned (-1 for n < 0). */
B2R_API long long b2r_flat_grad_norm_workspace_bytes(long long n);
B2R_API int b2r_flat_grad_norm(const float *grads, long long n, float grad_scale, float max_norm,
                               void *workspace, float *norm_out, float *coef_out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* B2R_H_ */
