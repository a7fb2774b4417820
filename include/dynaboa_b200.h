/* libdynaboa_b200 -- C ABI of the B200-native DynaBOA hot path.
 *
 * The reference (syguan96/DynaBOA) has no FFI/plugin boundary of its own: its hot path is Python
 * calling stock PyTorch ops (SURVEY.md §8b).  This header is the boundary the B200 implementation
 * introduces underneath the reference's Python API; each entry point names the reference code it
 * replaces.  Conventions:
 *   - every pointer is a DEVICE pointer to fp32 data unless stated otherwise; buffers are owned by
 *     the caller (torch-allocated) and must outlive the call;
 *   - `stream` is a cudaStream_t passed as void*; kernels are enqueued on it and never synchronise;
 *   - return value: 0 = ok, <0 = error (DBOA_ERR_*); no exceptions cross the ABI;
 *   - one host thread per device (the reference is single-threaded on this path).
 * Reference-side binding (ctypes) is shown in INTEGRATION.md.
 */
#ifndef DYNABOA_B200_H
#define DYNABOA_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define DBOA_OK 0
#define DBOA_ERR_ARG (-1)
#define DBOA_ERR_SHAPE (-2)
#define DBOA_ERR_CUDA (-3)
#define DBOA_ERR_UNSUPPORTED (-4)

typedef void* dboa_stream_t;

/* ---- library state ------------------------------------------------------------------------- */
const char* dboa_version(void);
int dboa_last_cuda_error(void);            /* cudaError_t of the last failed launch */
long long dboa_launch_count(void);         /* kernels launched by this library so far */
/* which convolution products of the HMR plan run on the tcgen05 TF32x3 kernel -- 0: none (fp32 CUDA cores); 1: forward;
 * 2: forward + dgrad + wgrad; 3 (default): forward + dgrad, weight gradients on CUDA cores */
int dboa_set_tensor_core_conv(int mode);

/* 1 (default): dboa_hmr_forward runs the fused plan -- every GroupNorm applied by the consuming convolution on load, its
 * statistics produced by the epilogue of the producing one (3 launches per bottleneck); 0: one convolution and one
 * GroupNorm launch per layer (round-1 plan, kept as the A/B reference).  Both fill the same tape. */
int dboa_set_fused_forward(int enable);
int dboa_get_fused_forward(void);
/* the same switch for dboa_hmr_backward: 1 = fused data-gradient chain (csrc/dgrad_wide.cu: parity-green, fewer launches, but
 * measured slower end to end), 0 (default) = GroupNorm-backward and data-gradient launches per layer */
int dboa_set_fused_backward(int enable);
/* CTAs (= SMs) the fused convolutions of the following dboa_hmr_forward calls may use; 0 = all.  Forwards issued side by side
 * on different streams share the device when each is given about half of it (a fused launch owns its SMs). */
int dboa_set_forward_cta_budget(int n);
/* Split-K limits of the planner of one tcgen05 kernel -- kernel 0: fused convolution (csrc/conv_wide.cu), 1: fused data gradient
 * (csrc/dgrad_wide.cu), 2: weight gradient (csrc/conv_wgrad_wide.cu).  A launch splits the reduction of a tile into nz K-slices
 * (nz = thread-block cluster size, a power of two <= max_nz) while the launch stays within max_ctas CTAs and every slice keeps at
 * least min_kb k-blocks.  A negative argument restores that limit's default (environment: DBOA_FUSED_MAX_CTAS / _MAX_NZ / _MINKB
 * for kernel 0, DBOA_DGRAD_MAX_CTAS / _MAX_NZ for 1, DBOA_WGRAD_MAX_CTAS / _MAX_NZ for 2; min_kb 2, 2, 1).  max_ctas = 0 does
 * not mean the same for every kernel: kernel 0 takes it as "every SM" (as dboa_set_forward_cta_budget), kernel 1 as "twice the
 * tiles, at most 128", kernel 2 clamps it to 1 (no split).  Kernel 0's max_ctas is the budget dboa_set_forward_cta_budget sets.
 * Returns DBOA_ERR_ARG for another kernel index. */
int dboa_set_split_limits(int kernel, int max_ctas, int max_nz, int min_kb);
/* Plan of the most recent launch of `kernel` (indices as above) in this process: out = {nz, k-blocks per slice, operand ring
 * depth, grid size in CTAs, k-blocks of the last slice}; all zero before the first launch.  DBOA_ERR_ARG for another index. */
int dboa_last_wide_plan(int kernel, long long out[5]);
/* 1: the fused convolution / data-gradient kernels keep the transformed activation operand (TF32 hi and lo parts) in tensor
 * memory and the tensor core reads only the weight operand from shared memory; 0: both operands in shared memory (the A/B
 * reference of the same kernels).  Same results to fp32 rounding of the same products (the split is identical).
 * Environment: DBOA_OPERAND_TMEM. */
int dboa_set_operand_tmem(int enable);
int dboa_get_operand_tmem(void);
/* 1: consecutive fused convolution launches of dboa_hmr_forward depend on each other through per-launch counters in the tape
 * (every producer CTA signals after its last store, the consumer's readers spin with acquire loads) instead of waiting for the
 * producer grid to complete and flush.  Same results; needs programmatic dependent launch (DBOA_PDL).  Environment: DBOA_CHAIN_FLAGS. */
int dboa_set_chain_flags(int enable);
int dboa_get_chain_flags(void);
/* Host-only self test (no CUDA call, runs without a GPU) of the TMA tensor-map cache: `n` insertions into a cache bounded at
 * `bound` entries while the caller, like a launch, holds the pointers of its last `window` (<= 16) lookups; evictions must leave
 * those pointers intact (they are freed one eviction later).  0 = ok, 1 + i = a held map was corrupted after insertion i. */
int dboa_selftest_map_cache(int bound, int n, int window);

/* ---- HMR regressor: parameter arena and tape layout ----------------------------------------
 * replaces: model/hmr.py:67-124 (HMR.__init__/_make_layer state_dict contract).
 * The 169 parameters live in ONE flat fp32 arena; entry i (in nn.Module.parameters() order) is the
 * strided view (offset, shape, stride) of it.  Conv weights are stored [Cout][kh][kw][Cin]. */
int dboa_hmr_num_params(void);
long long dboa_hmr_arena_floats(void);
int dboa_hmr_param_info(int i, char* name, int name_cap, long long* offset, int* ndim, long long shape[4], long long stride[4]);
long long dboa_hmr_tape_floats(int B);      /* activations saved by the forward (also holds the features) */
long long dboa_hmr_scratch_floats(int B);   /* scratch shared by forward (split-K) and backward */
/* feature i of HMR.forward(need_feature=True) (model/hmr.py:138-168) as a strided view of the tape */
int dboa_hmr_feature_info(int B, int i, long long* offset, int* ndim, long long shape[4], long long stride[4]);

/* replaces: model/hmr.py:127-181 HMR.forward (+ utils/geometry.py:47-61 rot6d_to_rotmat).
 * image: (B,3,224,224) NCHW.  drop_masks: NULL (eval) or (3,2,B,1024) keep-masks already scaled by 1/(1-p).
 * outputs: rotmat (B,24,3,3), shape (B,10), cam (B,3), pose6d (B,144). */
int dboa_hmr_forward(const float* arena, const float* init_pose, const float* init_shape, const float* init_cam,
                     const float* image, int B, const float* drop_masks, float* tape, float* scratch,
                     float* rotmat, float* shape, float* cam, float* pose6d, dboa_stream_t stream);
/* replaces: autograd backward of the above (torch.autograd.grad in learn2learn MAML.adapt, loss.backward()
 * at dynaboa_benchmark.py:140,150).  grad_arena is ACCUMULATED into (+=), same layout as the arena. */
int dboa_hmr_backward(const float* arena, const float* tape, int B, int masked /* forward used drop_masks */,
                      const float* d_rotmat, const float* d_shape, const float* d_cam, float* grad_arena, float* scratch,
                      dboa_stream_t stream);

/* Gradient buckets of the NEXT dboa_hmr_backward call, for overlapping the data-parallel all-reduce with the backward
 * (SURVEY.md section 8e).  Bucket k spans the floats [dboa_hmr_bucket_offset(k), dboa_hmr_bucket_offset(k - 1)) of the gradient
 * arena (offset(-1) = arena size): 0 = layer4 + regressor head, 1 = layer3, 2 = stem + layer1 + layer2 -- the order in which the
 * backward completes them.  ev0..2 are cudaEvent_t handles; event k is recorded when every kernel writing bucket k is ordered
 * before it.  Arm only for the LAST backward call that accumulates into the arena. */
int dboa_hmr_backward_buckets(void* ev0, void* ev1, void* ev2);
long long dboa_hmr_bucket_offset(int k);

/* ---- single operators (unit-parity surface; same kernels the plan above launches) ----------- */
/* replaces: nn.Conv2d forward / backward (model/hmr.py:29-34,72,113); NHWC activations, weights [Cout][Kpitch] */
int dboa_conv2d_fwd(const float* x, const float* w, float* y, int B, int Hi, int Wi, int Cin, int Cout, int k, int stride, int pad,
                    int Kpitch, float* ws, long long ws_floats, dboa_stream_t stream);
int dboa_conv2d_dgrad(const float* dy, const float* w, float* dx, int B, int Hi, int Wi, int Cin, int Cout, int k, int stride, int pad,
                      int Kpitch, int accumulate, float* ws, long long ws_floats, dboa_stream_t stream);
int dboa_conv2d_wgrad(const float* dy, const float* x, float* dw, int B, int Hi, int Wi, int Cin, int Cout, int k, int stride, int pad,
                      int Kpitch, float* ws, long long ws_floats, dboa_stream_t stream);
/* 1x1 / stride-1 convolution as a tcgen05 TF32x3 GEMM: y[M][Cout] = x[M][Cin] * w[Cout][Cin]^T (fp32-accurate);
 * needs dboa_set_tensor_core_conv(1); returns DBOA_ERR_UNSUPPORTED for shapes it does not take (Cin % 32, Cout % 64) */
int dboa_conv1x1_tc_fwd(const float* x, const float* w, float* y, int M, int Cin, int Cout, float* ws, long long ws_floats,
                        dboa_stream_t stream);
/* general convolution forward as a tcgen05 TF32x3 implicit GEMM (same arguments as dboa_conv2d_fwd; Cin % 64 == 0,
 * Cout % 64 == 0, Kpitch == k*k*Cin).  The stand-alone tensor-core entry points are launched with ordinary stream
 * serialization (inside dboa_hmr_forward/backward the same kernels use programmatic dependent launch and prefetch
 * weight tiles before their dependency wait, which needs the plan's guarantee that the preceding kernel does not write
 * the weights); DBOA_CABI_PDL=1 in the environment opts in for callers that can give that guarantee. */
int dboa_conv2d_tc_fwd(const float* x, const float* w, float* y, int B, int Hi, int Wi, int Cin, int Cout, int k, int stride, int pad,
                       int Kpitch, dboa_stream_t stream);
/* data / weight gradient on the same tensor-core kernel (needs dboa_set_tensor_core_conv(2 or 3)); dw is accumulated (+=) */
int dboa_conv2d_tc_dgrad(const float* dy, const float* w, float* dx, int B, int Hi, int Wi, int Cin, int Cout, int k, int stride, int pad,
                         int Kpitch, int accumulate, dboa_stream_t stream);
int dboa_conv2d_tc_wgrad(const float* dy, const float* x, float* dw, int B, int Hi, int Wi, int Cin, int Cout, int k, int stride, int pad,
                         int Kpitch, dboa_stream_t stream);
/* weight gradient on tcgen05 with MN-major operands fed by TMA (csrc/conv_wgrad_wide.cu): dw += dy^T * im2col(x); stride 1,
 * Cout % 128 == 0, Cin % 64 == 0, k in {1, 3}, pad k/2, square images of 56 / 28 / 14 / 7 (DBOA_ERR_UNSUPPORTED otherwise) */
int dboa_conv2d_wgrad_tma(const float* dy, const float* x, float* dw, int B, int Hi, int Wi, int Cin, int Cout, int k, int stride, int pad,
                          int Kpitch, dboa_stream_t stream);
/* Fused tcgen05 convolution, the unit the forward plan is made of (csrc/conv_wide.cu).
 * replaces: nn.Conv2d + the nn.GroupNorm(4, C) / ReLU / residual add that PRECEDES it in Bottleneck.forward
 * (model/hmr.py:40-60), + the statistics pass of the GroupNorm that follows it.
 *   y = conv(T(x), w);  part_out[b][g] += (sum y, sum y^2) of group g of sample b, as 64-bit fixed point (scale 2^24):
 *   integer atomics, exact and order independent.  part_out (long long [B][4][2]) must be ZERO before the launch.
 *   mode 0: T(x) = x;  1: relu(gn(x));  2: relu(gn(x) + res);  3: relu(gn(x) + gn2(res))
 * gn statistics come from `part_in` (`part2_in`): the accumulators a previous call filled for x (res).
 * a_out / stats_out / stats2_out (optional): T(x) materialised, (mean, rstd) [B][4][2] of the GroupNorm(s).
 * Up to 2 problems of equal mode, operand and reduction length share one launch.
 * Cin % 64 == 0, Cout % 64 == 0, k in {1, 3}, stride 1, pad k/2, H <= 128 (DBOA_ERR_UNSUPPORTED otherwise). */
typedef struct dboa_fused_conv {
    const float *x, *res, *w;
    float *a_out, *stats_out, *stats2_out;
    const float *part_in, *part2_in, *gamma, *beta, *gamma2, *beta2;
    float *y, *part_out;
    int mode;
    int Hi, Cin, Cout, k, stride, pad;
} dboa_fused_conv;
long long dboa_conv_fused_part_floats(int B, int Ho, int Cout);   /* size of part_out in floats (= B * 16) */
int dboa_conv_fused_fwd(const dboa_fused_conv* probs, int nprob, int B, dboa_stream_t stream);

/* Fused data gradient, the unit the backward plan is made of (csrc/dgrad_wide.cu).
 * replaces: the autograd backward of nn.GroupNorm (layer c) -> nn.Conv2d data gradient (layer c) -> residual add -> ReLU mask of
 * the producing layer p, + the reduction pass of GroupNorm_p's backward (model/hmr.py:40-60 under loss.backward()).
 *   dy  = rstd (dz gamma - m1 - x^ m2)                with (m1, m2) = sums_c / N, x^ = (y_c - mean) rstd     [dy_out: optional store]
 *   dX  = conv_c^T(dy) + addend                       stride 1, k in {1, 3}, Cin % 64 == 0, Cout % 64 == 0
 *   mask == NULL: out (+)= dX;   else out = dz_p = dX * (mask > 0) and, for each of the nprep GroupNorms of layer p,
 *   prep_sums[j][b][g] += (sum q, sum q x^), prep_dgb[j][c] += (d gamma, d beta) as 64-bit fixed point (scale 2^28; long long
 *   buffers the caller zeroes; integer atomics: exact and order independent). */
typedef struct dboa_dgrad_args {
    const float *dz, *y_c, *w, *stats_c, *sums_c, *gamma_c;
    float* dy_out;
    const float* addend;
    float* out;
    const float* mask;
    const float *prep_y[2], *prep_stats[2], *prep_gamma[2];
    float *prep_sums[2], *prep_dgb[2];
    int nprep, accumulate;
} dboa_dgrad_args;
int dboa_dgrad_fused(const dboa_dgrad_args* f, int B, int H, int Cin, int Cout, int k, dboa_stream_t stream);

/* replaces: nn.GroupNorm(4, C) + ReLU (+ residual) forward / backward (model/hmr.py:14-18,40-60).
 * C / 16 must be a power of two; one launch each (thread-block clusters).  `partial` is caller-provided scratch of
 * dboa_gn_*partial_floats() floats; the forward size is 0 in this version and the pointer may then be NULL. */
long long dboa_gn_partial_floats(int B, int HW, int C);
long long dboa_gn_bwd_partial_floats(int B, int HW, int C);
int dboa_groupnorm_fwd(const float* y, const float* gamma, const float* beta, const float* residual, float* out, float* stats,
                       float* partial, int B, int HW, int C, int relu, dboa_stream_t stream);
int dboa_groupnorm_bwd(const float* dout, const float* mask_src, const float* y, const float* stats, const float* gamma, float* dy,
                       float* dgamma, float* dbeta, float* partial, int B, int HW, int C, dboa_stream_t stream);
int dboa_maxpool_fwd(const float* x, float* y, unsigned char* idx, int B, int H, int W, int C, dboa_stream_t stream);
int dboa_maxpool_bwd(const float* dy, const unsigned char* idx, float* dx, int B, int H, int W, int C, dboa_stream_t stream);

/* ---- rotations (utils/geometry.py) ---------------------------------------------------------- */
int dboa_rot6d_fwd(const float* x6, float* R, int n, dboa_stream_t stream);                       /* :47-61 */
int dboa_rot6d_bwd(const float* x6, const float* dR, float* dx6, int n, dboa_stream_t stream);
/* kind 0: batch_rodrigues :9-45 (quaternion route); kind 1: smplx lbs.batch_rodrigues (pose2rot=True) */
int dboa_rodrigues(const float* aa, float* R, int n, int kind, dboa_stream_t stream);
int dboa_rotmat_to_aa_fwd(const float* R, float* aa, int n, dboa_stream_t stream);              /* :184-306 */
int dboa_rotmat_to_aa_bwd(const float* R, const float* daa, float* dR, int n, dboa_stream_t stream);

/* ---- SMPL (model/smpl.py:25-37 over smplx lbs) ---------------------------------------------- */
typedef struct dboa_smpl_model {
    const float* v_template;   /* (6890,3) */
    const float* blend_dirs;   /* (217, 20670): rows 0..9 shapedirs as (l, v*3+k), rows 10..216 posedirs */
    const float* J_template;   /* (24,3)   = J_regressor @ v_template */
    const float* J_shapedirs;  /* (24,3,10) = J_regressor @ shapedirs */
    const int* parents;        /* (24,) */
    const float* lbs_weights;  /* (6890,24) */
    const float* J_extra;      /* (9,6890) reference config.JOINT_REGRESSOR_TRAIN_EXTRA */
    const int* joint_map;      /* (49,) into [24 kinematic | 21 vertex picks | 9 extra] */
    const int* vertex_ids;     /* (21,) smplx vertex_joint_selector picks */
} dboa_smpl_model;
long long dboa_smpl_tape_floats(int B);
long long dboa_smpl_scratch_floats(int B);
/* betas (B,10), rotmat (B,24,3,3) -> vertices (B,6890,3), joints (B,49,3) */
int dboa_smpl_forward(const dboa_smpl_model* m, const float* betas, const float* rotmat, int B, float* vertices, float* joints,
                      float* tape, dboa_stream_t stream);
/* d(joints) -> d(rotmat), d(betas) (vertices carry no loss on the adaptation path: SURVEY.md Appendix A) */
int dboa_smpl_backward(const dboa_smpl_model* m, const float* rotmat, int B, const float* tape, const float* d_joints, float* scratch,
                       float* d_rotmat, float* d_betas, int accumulate, dboa_stream_t stream);

/* ---- projection and losses (base_adaptor.py) ------------------------------------------------ */
int dboa_project_fwd(const float* cam, const float* j3d, float* p2d, int B, int NJ, dboa_stream_t stream);      /* :160-170 */
int dboa_project_bwd(const float* cam, const float* j3d, const float* dp2d, float* dj3d, float* dcam, int B, int NJ, int acc_j,
                     int acc_cam, dboa_stream_t stream);
/* GMM pose prior (:405-409, utils/smplify/prior.py:181-196): prior_b[b] = min_m NLL; d_rotmat = scale * d prior_b / dR */
int dboa_pose_prior(const float* rotmat, const float* means, const float* precisions, const float* neg_log_w, float* prior_b,
                    float* d_rotmat, float scale, int B, dboa_stream_t stream);
/* MaxMixturePrior.forward(pose, betas) itself (utils/smplify/prior.py:227-231) on a (B,69) axis-angle body pose */
int dboa_gmm_prior(const float* pose69, const float* means, const float* precisions, const float* neg_log_w, float* prior_b,
                   float* d_pose, float scale, int B, dboa_stream_t stream);
typedef struct dboa_loss_args {
    int B;
    const float *p2d, *j3d, *R, *beta;      /* predictions: (B,49,2) (B,49,3) (B,24,3,3) (B,10) */
    const float* kp;                        /* (B,49,3) keypoints + confidence, or NULL */
    const float* prior_b;                   /* (B,) per-body pose prior values, or NULL */
    const float *t_p2d, *t_j3d, *t_beta, *t_R; /* consistency / label targets, or NULL each */
    const float* gt_s3d;                    /* (B,24,4) labelled 3D joints, or NULL (needs kp) */
    float w[8];                             /* weights: s2d, shape, pose, t_p2d, t_j3d, t_beta, t_R, s3d */
    float* terms;                           /* (9,) out: the 8 unweighted terms, then the weighted total */
    float *dp2d, *dj3d, *dR, *dbeta;        /* out: gradients of the weighted total (NULL to skip) */
    int dR_accumulate;                      /* 1: dR already holds the pose-prior gradient */
    int kp_first, kp_count;                 /* joints [kp_first, kp_first + kp_count) of the 49 carry the 2D re-projection term; 0, 0 = the
                                               benchmark's 24 ground-truth joints (25, 24); the webcam client compares the 25 OpenPose
                                               joints (0, 25), reference dynaboa_webcam.py:236,246,262 */
} dboa_loss_args;
int dboa_loss_multi(const dboa_loss_args* args, dboa_stream_t stream);        /* :234-241,283-291,331-337,360-370,401,412-422 */
int dboa_loss_motion(const float* p_cur, const float* p_hist, const float* kp_cur, const float* kp_hist, float weight, float* term,
                     float* dp_cur, float* dp_hist, int B, int accumulate_cur, dboa_stream_t stream);               /* :379-398 */
/* the same on joints [first, first + count): reference dynaboa_webcam.py:161-181 uses the 25 OpenPose joints (0, 25) */
int dboa_loss_motion_joints(const float* p_cur, const float* p_hist, const float* kp_cur, const float* kp_hist, float weight, float* term,
                            float* dp_cur, float* dp_hist, int B, int accumulate_cur, int first, int count, dboa_stream_t stream);

/* ---- whole-model sweeps, feature test, retrieval -------------------------------------------- */
int dboa_sgd_update(const float* p, const float* g, float* out, float lr, long long n, dboa_stream_t stream);   /* l2l maml_update */
int dboa_adam_ema(float* p, const float* g, float* m, float* v, float* teacher /* or NULL */, long long n, float lr, float beta1,
                  float beta2, float eps, int step, float alpha, dboa_stream_t stream);     /* base_adaptor.py:126,193-201 */
int dboa_ema_update(float* teacher, const float* p, long long n, float alpha, dboa_stream_t stream);
/* Adam(+EMA) on g * gscale: the data-parallel mean of an all-reduced (summed) gradient without a separate sweep */
int dboa_adam_ema_scaled(float* p, const float* g, float* m, float* v, float* teacher /* or NULL */, long long n, float lr, float beta1,
                         float beta2, float eps, int step, float alpha, float gscale, dboa_stream_t stream);
/* stream-ordered fill / device-to-device copy on the copy engine (gradient arenas, frame staging: no ATen kernels in a step) */
int dboa_fill_zero(void* dst, long long bytes, dboa_stream_t stream);
int dboa_copy_async(void* dst, const void* src, long long bytes, dboa_stream_t stream);
/* cal_feature_diff :211-219: cosine similarity of npairs (<=16) flattened tensor pairs; host arrays of device pointers */
int dboa_cosine_pairs(const float* const* a, const float* const* b, const long long* n, int npairs, float* partial,
                      long long partial_floats, float* out, float eps, dboa_stream_t stream);
/* the same reduction, returning per pair the three sums (a.b, |a|^2, |b|^2) in double, [npairs][3]: under data-parallel
 * adaptation they are all-reduced before the cosine is formed, so that every rank takes the same branch of the
 * dynamic loop (dynaboa_benchmark.py:161-192; cal_feature_diff flattens across the batch, base_adaptor.py:215).
 * partial: dboa_cosine_partial_floats(n, npairs) floats of scratch. */
long long dboa_cosine_partial_floats(const long long* n, int npairs);
int dboa_cosine_terms(const float* const* a, const float* const* b, const long long* n, int npairs, float* partial,
                      long long partial_floats, double* terms, dboa_stream_t stream);
/* retrieval :82-84: index of the centre with the smallest cosine distance to feat (D,) among centers (K,D) */
int dboa_retrieval_nearest(const float* feat, const float* centers, int K, int D, int* best, float* dists, dboa_stream_t stream);

/* ---- input side: crop + resize + normalise, keypoint transform (utils/dataprocess.py:13-96, boa_dataset/pw3d.py:127-163) ---
 * img: device image (H,W,3) RGB, float32 0..255 or uint8 (is_u8).  The crop box [ul, ul + (Wc, Hc)) (integer corners as the
 * reference computes them; zero outside the frame) is resized to res x res as  out = Wy . crop . Wx^T : wx (res,Tx) / wy (res,Ty)
 * are the rows of the banded matrices (skimage.transform.resize = Gaussian pre-filter + order-1 zoom, mirror boundaries,
 * composed on the host), sx / sy (res,) int32 their first crop column / row.  Host arrays mean3 / std3: channel statistics.
 * tmp: Hc * res * 3 floats of scratch.  out: (3,res,res) = (resized / 255 - mean) / std. */
int dboa_crop_resize_normalize(const void* img, int is_u8, int H, int W, int ul_x, int ul_y, int Hc, const float* wx, const int* sx, int Tx,
                               const float* wy, const int* sy, int Ty, int res, const float* mean3, const float* std3, float* tmp,
                               float* out, dboa_stream_t stream);
/* kp (n,3) pixel keypoints + confidence -> out (n,3): p = trunc(t . (x, y, 1)) + 1 in double as utils/dataprocess.py:39-46 on kp + 1,
 * then 2 p / res - 1; t00, t02, t11, t12: the non-zero entries of get_transform(center, scale, res) (:13-37, rot = 0) */
int dboa_keypoint_transform(const float* kp, int n, double t00, double t02, double t11, double t12, int res, float* out,
                            dboa_stream_t stream);

/* ---- evaluation metrics (dynaboa_benchmark.py:217-240, utils/pose_utils.py:9-64) -----------------
 * pred_verts, gt_verts_joints (gender-selected SMPL mesh), gt_verts_pve (neutral mesh): (B,NV,3);
 * J_regressor (NJ,NV) dense; joint_map (n_map,) int32 indices into the NJ regressed joints (H36M_TO_J14).
 * Joints are centred on regressed joint 0 (pelvis) like the reference.  out (B,3) = MPJPE, PA-MPJPE (similarity
 * Procrustes, 3x3 SVD on the device) and PVE per sample, in the unit of the meshes (metres).
 * scratch: dboa_eval_scratch_floats(B, NJ) floats.  NJ, n_map <= 32. */
long long dboa_eval_scratch_floats(int B, int NJ);
int dboa_eval_metrics(const float* pred_verts, const float* gt_verts_joints, const float* gt_verts_pve, const float* J_regressor, int NJ,
                      int NV, const int* joint_map, int n_map, float* scratch, float* out, int B, dboa_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* DYNABOA_B200_H */
