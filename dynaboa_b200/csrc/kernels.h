// Internal launcher prototypes shared between the kernel translation units, the per-op C-ABI
// wrappers (cabi.cu) and the whole-network plan (hmr_plan.cu).  Not part of the public ABI.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

namespace dboa {

struct ConvDims {
    int B, Hi, Wi, Cin, Ho, Wo, Cout, kh, kw, stride, pad, Kpitch;
};

// ---- conv.cu (fp32 CUDA-core implicit GEMM)
int conv_fwd(const float* x, const float* w, float* y, const ConvDims& d, float* ws, size_t ws_floats, cudaStream_t st);
int conv_dgrad(const float* dy, const float* w, float* dx, const ConvDims& d, int accumulate, float* ws, size_t ws_floats, cudaStream_t st);
int conv_wgrad(const float* dy, const float* x, float* dw, const ConvDims& d, float* ws, size_t ws_floats, cudaStream_t st);

// ---- conv_tc.cu (tcgen05 TF32x3 GEMM for 1x1 / stride-1 convolutions); returns DBOA_ERR_UNSUPPORTED when the shape is not taken
// `pdl`: launch with programmatic stream serialization.  The forward / data-gradient kernels prefetch WEIGHT tiles before
// their dependency wait, which is only safe when the preceding kernel in the stream does not write the weights (true inside
// the network plan; the stand-alone C-ABI wrappers pass false).
int conv_tc_fwd(const float* x, const float* w, float* y, const ConvDims& d, cudaStream_t st, bool pdl = true);
int conv_tc_dgrad(const float* dy, const float* w, float* dx, const ConvDims& d, int accumulate, cudaStream_t st, bool pdl = true);
int conv_tc_wgrad(const float* dy, const float* x, float* dw, const ConvDims& d, cudaStream_t st, bool pdl = true);
bool conv_tc_bwd_enabled();
bool conv_tc_wgrad_enabled();
int conv1x1_tc_fwd(const float* x, const float* w, float* y, int M, int Cin, int Cout, cudaStream_t st, bool pdl = true);
bool conv_tc_enabled();
void conv_tc_set_enabled(bool on);
void conv_tc_set_mode(int mode);                      // 0 off, 1 forward, 2 forward + dgrad + wgrad, 3 forward + dgrad

// ---- description of one fused convolution (conv_wide.cu)
struct FusedConv {
    const float *x, *res, *w;                 // operand source (see `mode`), second source (modes 2, 3), weights [Cout][k*k*Cin]
    float *a_out, *stats_out, *stats2_out;    // optional tape stores: transformed operand, (mean, rstd) [B][4][2] of the operand's GroupNorm(s)
    const float *part_in, *part2_in;          // statistics accumulators of x / res left by their producers
    const float *gamma, *beta, *gamma2, *beta2;
    float *y, *part_out;                      // raw output [B][Ho][Ho][Cout] and its statistics accumulators
    int mode;                                 // 0: x as is; 1: relu(gn(x)); 2: relu(gn(x) + res); 3: relu(gn(x) + gn2(res))
    int S_in, S2_in;                          // unused
    int Hi, Cin, Cout, k, stride, pad, Ho;    // square images
};
// ---- conv_wide.cu (fused convolution: both operands through TMA, 16 transform warps, fixed-point statistics)
// part_in / part_out point to the fixed-point accumulators (long long [B][4][2], ZEROED by the caller
// before the producing launch); S_in / S2_in are unused.  Stride-1 convolutions only.
bool conv_wide_ok(const FusedConv& d);
int conv_wide_plan(const FusedConv* d, int nprob, int B);
void conv_wide_set_cta_budget(int n);                                  // 0: all SMs
// split-K limits of the planners (a negative argument restores the environment default; see dboa_set_split_limits)
void conv_wide_set_limits(int max_ctas, int max_nz, int min_kb);
void dgrad_wide_set_limits(int max_ctas, int max_nz, int min_kb);
void conv_wgrad_wide_set_limits(int max_ctas, int max_nz, int min_kb);
inline int clamp_split(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }
// plan of the most recent launch of kernel 0 (conv_wide), 1 (dgrad_wide), 2 (conv_wgrad_wide): K-slices (= cluster size),
// k-blocks per slice, operand ring depth, grid size, k-blocks of the last slice
struct WidePlan { long long nz, per, D, grid, last; };
void wide_plan_note(int kernel, int nz, int per, int D, int grid, int nkb);
bool wide_plan_last(int kernel, long long out[5]);
int map_cache_selftest(int bound, int n, int window);                   // host-only check of the tensor-map cache's eviction rule
void conv_wide_set_operand_tmem(bool on);                              // transformed activation operand of conv_wide / dgrad_wide in tensor memory
bool conv_wide_operand_tmem();
// chain dependency between consecutive fused launches of one forward (conv_wide.cu: chain_wait): the launch waits until
// *wait_flag >= wait_count instead of for the completion of its predecessor grid (wait_flag NULL: ordinary dependency), every CTA
// of it increments *signal_flag when its outputs are stored, and *signal_count receives the number of CTAs (the next wait_count)
struct ChainDep {
    const unsigned* wait_flag; unsigned wait_count;
    unsigned* signal_flag; unsigned* signal_count;
};
int conv_wide_launch(const FusedConv* d, int nprob, int B, int nz, const float* next_w, size_t next_bytes, cudaStream_t st, bool pdl,
                     const ChainDep* dep = nullptr);
int gn_acc_res_avgpool(const float* y, const float* res, const float* acc, const float* gamma, const float* beta, float* a_out, float* stats_out,
                       float* out, int B, int HW, int C, int ld, int ncopy, size_t copy_stride, cudaStream_t st);

// ---- conv_wgrad_wide.cu (tcgen05 weight gradient, MN-major operands through TMA); dw is accumulated (+=)
// 7x7 / stride-2 stem weight gradient: row-per-CTA partials + fixed-order reduction (stem_wgrad.cu); needs 64 * 147 floats of
// workspace per partial (DBOA_ERR_UNSUPPORTED for any other shape or without workspace)
bool stem_wgrad_ok(const ConvDims& d);
int stem_wgrad(const float* dy, const float* x, float* dw, const ConvDims& d, float* ws, size_t ws_floats, cudaStream_t st);
bool conv_wgrad_wide_ok(const ConvDims& d);
int conv_wgrad_wide(const float* dy, const float* x, float* dw, const ConvDims& d, cudaStream_t st, bool pdl);

// ---- dgrad_wide.cu (fused data gradient: GroupNorm backward of the operand on load, ReLU mask + the next GroupNorm backward's
// sums in the epilogue; see the file header).  All sums are 64-bit fixed point (long long, scale 2^28), zeroed by the caller.
struct DgradPrep {
    const float* y;            // raw output of the layer whose GroupNorm backward is prepared [B][H][W][C]
    const float* stats;        // its (mean, rstd) [B][4][2]
    const float* gamma;
    float* sums;               // long long [B][4][2]: sum q, sum q x^   (q = dz gamma)
    float* dgb;                // long long [C][2]: d gamma, d beta
};
struct DgradFused {
    const float *dz, *y_c, *w;                     // masked gradient w.r.t. GroupNorm_c's output, raw output of conv c, weights of conv c
    const float *stats_c, *sums_c, *gamma_c;       // GroupNorm_c: (mean, rstd), backward sums (long long), gamma
    float* dy_out;                                 // dy_c materialised for the weight gradient, or NULL
    const float* addend;                           // added to dX before the mask (shortcut gradient), or NULL
    float* out;                                    // mask == NULL: dX (accumulate: +=); else dz of the producing layer
    const float* mask;                             // post-activation output of the producing layer, or NULL
    DgradPrep prep[2];
    int nprep, accumulate;
};
bool dgrad_wide_ok(const ConvDims& d);
int dgrad_wide(const DgradFused& f, const ConvDims& d, cudaStream_t st, bool pdl);
int gn_bwd_prep(const float* dA, const float* mask, float* out, const DgradPrep& p, int B, int HW, int C, cudaStream_t st);
struct GnFinishItem;
int gn_dgb_finish(const GnFinishItem* items_dev, int n_items, const float* dgb, float* G, cudaStream_t st);

// ---- groupnorm.cu (single-launch cluster kernels)
size_t gn_partial_floats(int B, int HW, int C);     // forward scratch (none; kept for the C ABI)
size_t gn_bwd_partial_floats(int B, int HW, int C); // backward scratch: per-sample dgamma / dbeta rows
// out = relu?( gn(y) [+ res] ); writes (mean, rstd) to stats[B][4][2]
// backward: dz = dout * (mask_src > 0 if mask_src else 1); dy = GN backward; dgamma/dbeta accumulate (+=)
int gn_fwd_fused(const float* y, const float* gamma, const float* beta, const float* res, float* out, float* stats, float* partial,
                 int B, int HW, int C, int relu, cudaStream_t st);
// defer = 1 (B > 1 only): leave the per-sample dgamma / dbeta rows in `partial` for gn_param_finish instead of reducing them here
int gn_bwd_fused(const float* dout, const float* mask_src, const float* y, const float* stats, const float* gamma, float* dy,
                 float* dgamma, float* dbeta, float* partial, int B, int HW, int C, cudaStream_t st, int defer = 0);
struct GnFinishItem { long long g_off, b_off, cum_channels; int C; };
int gn_param_finish(const GnFinishItem* items_dev, int n_items, const float* rows, float* G, int B, cudaStream_t st);
// ---- norm_pool.cu
int relu_mask(const float* dout, const float* mask_src, float* dz, size_t n, cudaStream_t st);
int nchw_to_nhwc(const float* x, float* y, int B, int C, int H, int W, cudaStream_t st);
int maxpool3x3s2_fwd(const float* x, float* y, unsigned char* idx, int B, int H, int W, int C, cudaStream_t st);
int maxpool3x3s2_bwd(const float* dy, const unsigned char* idx, float* dx, int B, int H, int W, int C, cudaStream_t st);
// mean over HW -> out rows with leading dimension ld, replicated `ncopy` times `copy_stride` floats apart
int avgpool_fwd(const float* x, float* out, int B, int HW, int C, int ld, int ncopy, size_t copy_stride, cudaStream_t st);
int avgpool_bwd(const float* dxf, int ld, float* dx, int B, int HW, int C, cudaStream_t st);

// ---- head.cu
// y[b][n] = (addend ? addend[b][n] : 0) + bias[n] + sum_k x[b][k] W[n][k];  pre <- y (before mask), post <- y*mask
int linear_fwd(const float* x, int ldx, const float* W, int ldw, const float* bias, const float* addend, int ld_add,
               const float* mask, float* pre, float* post, int ld_out, float* post2, int ld_out2,
               int B, int N, int K, cudaStream_t st);
// dx[b][k] = sum_n dy[b][n] W[n][k] (k < K)
int linear_dgrad(const float* dy, int ldy, const float* W, int ldw, float* dx, int ldx, int B, int N, int K,
                 float* ws, size_t ws_floats, cudaStream_t st);
// dW[n][k] += sum_r dy[r][n] x[r][k];  db[n] += sum_r dy[r][n]
int linear_wgrad(const float* dy, int ldy, const float* x, int ldx, float* dW, int ldw, float* db, int R, int N, int K, cudaStream_t st);
int rot6d_fwd_launch(const float* pose6d, float* rotmat, int n, cudaStream_t st);
int rot6d_bwd_launch(const float* pose6d, const float* drot, float* dpose, int n, cudaStream_t st);
int ew_mul(const float* a, const float* b, float* out, size_t n, cudaStream_t st);
int ew_add_rows(float* dst, int ld_dst, const float* a, int lda, const float* b, int ldb, int B, int n, cudaStream_t st);

// ---- dataprocess.cu (crop + anti-aliased resize + normalise, keypoint transform)
int crop_resize_normalize(const void* img, int is_u8, int H, int W, int ul_x, int ul_y, int Hc, const float* wx, const int* sx, int Tx,
                          const float* wy, const int* sy, int Ty, int res, const float mean[3], const float stdv[3], float* tmp, float* out,
                          cudaStream_t st);
int keypoint_transform(const float* kp, int n, double t00, double t02, double t11, double t12, int res, float* out, cudaStream_t st);

// ---- eval.cu (evaluation metrics on the device)
size_t eval_scratch_floats(int B, int NJ);
int eval_metrics(const float* pred_verts, const float* gt_verts_joints, const float* gt_verts_pve, const float* Jreg, int NJ, int NV,
                 const int* joint_map, int n_map, float* scratch, float* out, int B, cudaStream_t st);

}  // namespace dboa
