// extern "C" surface of libdynaboa_b200 (see include/dynaboa_b200.h for the contract of each entry).
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "kernels.h"
#include "losses.h"
#include "optim.h"
#include "rotmath.cuh"
#include "smpl.h"

namespace dboa {
int hmr_forward(const float* P, const float* init_pose, const float* init_shape, const float* init_cam, const float* image, int B,
                const float* drop_masks, float* T, float* scratch, float* rotmat, float* shape, float* cam, float* pose6d,
                cudaStream_t st);
int hmr_backward(const float* P, const float* T, int B, int masked, const float* d_rotmat, const float* d_shape, const float* d_cam,
                 float* G, float* scratch, cudaStream_t st);
void hmr_arm_bucket_events(cudaEvent_t e0, cudaEvent_t e1, cudaEvent_t e2);
long long hmr_bucket_offset(int k);
void hmr_set_fused_forward(bool on);
void hmr_set_fused_backward(bool on);
void hmr_set_chain_flags(bool on);
bool hmr_chain_flags();
bool hmr_fused_forward();
int hmr_num_params();
long long hmr_arena_floats();
int hmr_param_info(int i, char* name, int cap, long long* off, int* ndim, long long shape[4], long long stride[4]);
long long hmr_tape_floats(int B);
long long hmr_scratch_floats(int B);
int hmr_feature_info(int B, int i, long long* off, int* ndim, long long shape[4], long long stride[4]);

__global__ void r2aa_fwd_kernel(const float* __restrict__ R, float* __restrict__ aa, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float Ri[9], a[3];
    for (int k = 0; k < 9; ++k) Ri[k] = R[(size_t)i * 9 + k];
    r2aa_fwd(Ri, a);
    for (int k = 0; k < 3; ++k) aa[(size_t)i * 3 + k] = a[k];
}
__global__ void r2aa_bwd_kernel(const float* __restrict__ R, const float* __restrict__ daa, float* __restrict__ dR, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float Ri[9], d[3], g[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int k = 0; k < 9; ++k) Ri[k] = R[(size_t)i * 9 + k];
    for (int k = 0; k < 3; ++k) d[k] = daa[(size_t)i * 3 + k];
    r2aa_bwd(Ri, d, g);
    for (int k = 0; k < 9; ++k) dR[(size_t)i * 9 + k] = g[k];
}
}  // namespace dboa

using namespace dboa;
#define ST(s) reinterpret_cast<cudaStream_t>(s)

static ConvDims make_dims(int B, int Hi, int Wi, int Cin, int Cout, int k, int stride, int pad, int Kpitch) {
    ConvDims d;
    d.B = B; d.Hi = Hi; d.Wi = Wi; d.Cin = Cin; d.Cout = Cout; d.kh = k; d.kw = k; d.stride = stride; d.pad = pad; d.Kpitch = Kpitch;
    d.Ho = (Hi + 2 * pad - k) / stride + 1; d.Wo = (Wi + 2 * pad - k) / stride + 1;
    return d;
}

// The tensor-core kernels prefetch weight tiles before their dependency wait, which is only safe when the caller knows that
// the preceding kernel in the stream does not write the weights (the network plan does).  The stand-alone entry points are
// therefore launched with ordinary stream serialization; DBOA_CABI_PDL=1 opts in (scripts/conv_microbench.py chains).
static bool cabi_pdl() {
    static const bool on = [] { const char* e = getenv("DBOA_CABI_PDL"); return e && e[0] == '1'; }();
    return on;
}

extern "C" {

const char* dboa_version(void) { return "dynaboa_b200 0.1 (sm_100a)"; }
int dboa_last_cuda_error(void) { return g_last_cuda_error; }
long long dboa_launch_count(void) { return g_launch_count; }
int dboa_set_tensor_core_conv(int enable) { conv_tc_set_mode(enable); return DBOA_OK; }

int dboa_set_fused_forward(int enable) { hmr_set_fused_forward(enable != 0); return DBOA_OK; }
int dboa_get_fused_forward(void) { return hmr_fused_forward() ? 1 : 0; }
int dboa_set_fused_backward(int enable) { hmr_set_fused_backward(enable != 0); return DBOA_OK; }
int dboa_set_forward_cta_budget(int n) { conv_wide_set_cta_budget(n < 0 ? 0 : n); return DBOA_OK; }
int dboa_set_split_limits(int kernel, int max_ctas, int max_nz, int min_kb) {
    switch (kernel) {
        case 0: conv_wide_set_limits(max_ctas, max_nz, min_kb); return DBOA_OK;
        case 1: dgrad_wide_set_limits(max_ctas, max_nz, min_kb); return DBOA_OK;
        case 2: conv_wgrad_wide_set_limits(max_ctas, max_nz, min_kb); return DBOA_OK;
        default: return DBOA_ERR_ARG;
    }
}
int dboa_last_wide_plan(int kernel, long long out[5]) {
    if (!out) return DBOA_ERR_ARG;
    return wide_plan_last(kernel, out) ? DBOA_OK : DBOA_ERR_ARG;
}
int dboa_set_operand_tmem(int enable) { conv_wide_set_operand_tmem(enable != 0); return DBOA_OK; }
int dboa_selftest_map_cache(int bound, int n, int window) { return map_cache_selftest(bound, n, window); }
int dboa_set_chain_flags(int enable) { hmr_set_chain_flags(enable != 0); return DBOA_OK; }
int dboa_get_chain_flags(void) { return hmr_chain_flags() ? 1 : 0; }
int dboa_get_operand_tmem(void) { return conv_wide_operand_tmem() ? 1 : 0; }

int dboa_hmr_num_params(void) { return hmr_num_params(); }
long long dboa_hmr_arena_floats(void) { return hmr_arena_floats(); }
int dboa_hmr_param_info(int i, char* name, int name_cap, long long* offset, int* ndim, long long shape[4], long long stride[4]) {
    if (!offset || !ndim || !shape || !stride) return DBOA_ERR_ARG;
    return hmr_param_info(i, name, name_cap, offset, ndim, shape, stride);
}
long long dboa_hmr_tape_floats(int B) { return hmr_tape_floats(B); }
long long dboa_hmr_scratch_floats(int B) { return hmr_scratch_floats(B); }
int dboa_hmr_feature_info(int B, int i, long long* offset, int* ndim, long long shape[4], long long stride[4]) {
    if (!offset || !ndim || !shape || !stride) return DBOA_ERR_ARG;
    return hmr_feature_info(B, i, offset, ndim, shape, stride);
}
int dboa_hmr_forward(const float* arena, const float* init_pose, const float* init_shape, const float* init_cam, const float* image,
                     int B, const float* drop_masks, float* tape, float* scratch, float* rotmat, float* shape, float* cam, float* pose6d,
                     dboa_stream_t stream) {
    if (!arena || !init_pose || !init_shape || !init_cam || !image || !tape || !scratch || !rotmat || !shape || !cam) return DBOA_ERR_ARG;
    return hmr_forward(arena, init_pose, init_shape, init_cam, image, B, drop_masks, tape, scratch, rotmat, shape, cam, pose6d, ST(stream));
}
int dboa_hmr_backward(const float* arena, const float* tape, int B, int masked, const float* d_rotmat, const float* d_shape,
                      const float* d_cam, float* grad_arena, float* scratch, dboa_stream_t stream) {
    if (!arena || !tape || !grad_arena || !scratch) return DBOA_ERR_ARG;
    return hmr_backward(arena, tape, B, masked, d_rotmat, d_shape, d_cam, grad_arena, scratch, ST(stream));
}

int dboa_conv2d_fwd(const float* x, const float* w, float* y, int B, int Hi, int Wi, int Cin, int Cout, int k, int stride, int pad, int Kpitch,
                    float* ws, long long ws_floats, dboa_stream_t stream) {
    if (!x || !w || !y) return DBOA_ERR_ARG;
    return conv_fwd(x, w, y, make_dims(B, Hi, Wi, Cin, Cout, k, stride, pad, Kpitch), ws, ws ? (size_t)ws_floats : 0, ST(stream));
}
int dboa_conv2d_dgrad(const float* dy, const float* w, float* dx, int B, int Hi, int Wi, int Cin, int Cout, int k, int stride, int pad,
                      int Kpitch, int accumulate, float* ws, long long ws_floats, dboa_stream_t stream) {
    if (!dy || !w || !dx) return DBOA_ERR_ARG;
    return conv_dgrad(dy, w, dx, make_dims(B, Hi, Wi, Cin, Cout, k, stride, pad, Kpitch), accumulate, ws, ws ? (size_t)ws_floats : 0, ST(stream));
}
int dboa_conv2d_wgrad(const float* dy, const float* x, float* dw, int B, int Hi, int Wi, int Cin, int Cout, int k, int stride, int pad,
                      int Kpitch, float* ws, long long ws_floats, dboa_stream_t stream) {
    if (!dy || !x || !dw) return DBOA_ERR_ARG;
    return conv_wgrad(dy, x, dw, make_dims(B, Hi, Wi, Cin, Cout, k, stride, pad, Kpitch), ws, ws ? (size_t)ws_floats : 0, ST(stream));
}
int dboa_conv1x1_tc_fwd(const float* x, const float* w, float* y, int M, int Cin, int Cout, float* ws, long long ws_floats,
                        dboa_stream_t stream) {
    if (!x || !w || !y) return DBOA_ERR_ARG;
    (void)ws; (void)ws_floats;                 /* kept in the signature: the split-K reduction lives in shared memory (DSMEM) now */
    return conv1x1_tc_fwd(x, w, y, M, Cin, Cout, ST(stream), cabi_pdl());
}
int dboa_conv2d_tc_fwd(const float* x, const float* w, float* y, int B, int Hi, int Wi, int Cin, int Cout, int k, int stride, int pad,
                       int Kpitch, dboa_stream_t stream) {
    if (!x || !w || !y) return DBOA_ERR_ARG;
    return conv_tc_fwd(x, w, y, make_dims(B, Hi, Wi, Cin, Cout, k, stride, pad, Kpitch), ST(stream), cabi_pdl());
}
int dboa_conv2d_tc_dgrad(const float* dy, const float* w, float* dx, int B, int Hi, int Wi, int Cin, int Cout, int k, int stride, int pad,
                         int Kpitch, int accumulate, dboa_stream_t stream) {
    if (!dy || !w || !dx) return DBOA_ERR_ARG;
    return conv_tc_dgrad(dy, w, dx, make_dims(B, Hi, Wi, Cin, Cout, k, stride, pad, Kpitch), accumulate, ST(stream), cabi_pdl());
}
int dboa_conv2d_tc_wgrad(const float* dy, const float* x, float* dw, int B, int Hi, int Wi, int Cin, int Cout, int k, int stride, int pad,
                         int Kpitch, dboa_stream_t stream) {
    if (!dy || !x || !dw) return DBOA_ERR_ARG;
    return conv_tc_wgrad(dy, x, dw, make_dims(B, Hi, Wi, Cin, Cout, k, stride, pad, Kpitch), ST(stream), cabi_pdl());
}
int dboa_conv2d_wgrad_tma(const float* dy, const float* x, float* dw, int B, int Hi, int Wi, int Cin, int Cout, int k, int stride, int pad,
                          int Kpitch, dboa_stream_t stream) {
    if (!dy || !x || !dw) return DBOA_ERR_ARG;
    return conv_wgrad_wide(dy, x, dw, make_dims(B, Hi, Wi, Cin, Cout, k, stride, pad, Kpitch), ST(stream), false);
}
int dboa_dgrad_fused(const dboa_dgrad_args* f, int B, int H, int Cin, int Cout, int k, dboa_stream_t stream) {
    if (!f || !f->dz || !f->y_c || !f->w || !f->stats_c || !f->sums_c || !f->gamma_c || !f->out) return DBOA_ERR_ARG;
    DgradFused d;
    memset(&d, 0, sizeof d);
    d.dz = f->dz; d.y_c = f->y_c; d.w = f->w; d.stats_c = f->stats_c; d.sums_c = f->sums_c; d.gamma_c = f->gamma_c; d.dy_out = f->dy_out;
    d.addend = f->addend; d.out = f->out; d.mask = f->mask; d.nprep = f->nprep; d.accumulate = f->accumulate;
    for (int j = 0; j < 2; ++j) {
        d.prep[j].y = f->prep_y[j]; d.prep[j].stats = f->prep_stats[j]; d.prep[j].gamma = f->prep_gamma[j];
        d.prep[j].sums = f->prep_sums[j]; d.prep[j].dgb = f->prep_dgb[j];
        if (f->mask && j < f->nprep && (!d.prep[j].y || !d.prep[j].stats || !d.prep[j].gamma || !d.prep[j].sums || !d.prep[j].dgb)) return DBOA_ERR_ARG;
    }
    return dgrad_wide(d, make_dims(B, H, H, Cin, Cout, k, 1, k / 2, k * k * Cin), ST(stream), cabi_pdl());
}
long long dboa_conv_fused_part_floats(int B, int Ho, int Cout) { (void)Ho; (void)Cout; return (long long)B * 16; }
int dboa_conv_fused_fwd(const dboa_fused_conv* probs, int nprob, int B, dboa_stream_t stream) {
    if (!probs || nprob < 1 || nprob > 2 || B < 1) return DBOA_ERR_ARG;
    FusedConv d[2];
    for (int i = 0; i < nprob; ++i) {
        const dboa_fused_conv& c = probs[i];
        if (!c.x || !c.w || !c.y || !c.part_out) return DBOA_ERR_ARG;
        if (c.mode >= 1 && (!c.part_in || !c.gamma || !c.beta)) return DBOA_ERR_ARG;
        if (c.mode >= 2 && !c.res) return DBOA_ERR_ARG;
        if (c.mode == 3 && (!c.part2_in || !c.gamma2 || !c.beta2)) return DBOA_ERR_ARG;
        FusedConv& f = d[i];
        memset(&f, 0, sizeof f);
        f.x = c.x; f.res = c.res; f.w = c.w; f.a_out = c.a_out; f.stats_out = c.stats_out; f.stats2_out = c.stats2_out;
        f.part_in = c.part_in; f.part2_in = c.part2_in; f.gamma = c.gamma; f.beta = c.beta; f.gamma2 = c.gamma2; f.beta2 = c.beta2;
        f.y = c.y; f.part_out = c.part_out; f.mode = c.mode;
        f.Hi = c.Hi; f.Cin = c.Cin; f.Cout = c.Cout; f.k = c.k; f.stride = c.stride; f.pad = c.pad;
        f.Ho = (c.Hi + 2 * c.pad - c.k) / c.stride + 1;
        if (!conv_wide_ok(f)) return DBOA_ERR_UNSUPPORTED;
    }
    const int nz = conv_wide_plan(d, nprob, B);
    return conv_wide_launch(d, nprob, B, nz, nullptr, 0, ST(stream), cabi_pdl());
}
long long dboa_gn_partial_floats(int B, int HW, int C) { return (long long)gn_partial_floats(B, HW, C); }
long long dboa_gn_bwd_partial_floats(int B, int HW, int C) { return (long long)gn_bwd_partial_floats(B, HW, C); }
int dboa_groupnorm_fwd(const float* y, const float* gamma, const float* beta, const float* residual, float* out, float* stats, float* partial,
                       int B, int HW, int C, int relu, dboa_stream_t stream) {
    if (!y || !gamma || !beta || !out || !stats) return DBOA_ERR_ARG;       // `partial` may be NULL: dboa_gn_partial_floats() is 0
    return gn_fwd_fused(y, gamma, beta, residual, out, stats, partial, B, HW, C, relu, ST(stream));
}
int dboa_groupnorm_bwd(const float* dout, const float* mask_src, const float* y, const float* stats, const float* gamma, float* dy,
                       float* dgamma, float* dbeta, float* partial, int B, int HW, int C, dboa_stream_t stream) {
    if (!dout || !y || !stats || !gamma || !dy || !dgamma || !dbeta || !partial) return DBOA_ERR_ARG;
    return gn_bwd_fused(dout, mask_src, y, stats, gamma, dy, dgamma, dbeta, partial, B, HW, C, ST(stream));
}
int dboa_maxpool_fwd(const float* x, float* y, unsigned char* idx, int B, int H, int W, int C, dboa_stream_t stream) {
    if (!x || !y || !idx || (H & 1) || (W & 1) || (C & 3)) return DBOA_ERR_ARG;
    return maxpool3x3s2_fwd(x, y, idx, B, H, W, C, ST(stream));
}
int dboa_maxpool_bwd(const float* dy, const unsigned char* idx, float* dx, int B, int H, int W, int C, dboa_stream_t stream) {
    if (!dy || !idx || !dx || (H & 1) || (W & 1) || (C & 3)) return DBOA_ERR_ARG;
    return maxpool3x3s2_bwd(dy, idx, dx, B, H, W, C, ST(stream));
}

int dboa_rot6d_fwd(const float* x6, float* R, int n, dboa_stream_t stream) {
    if (!x6 || !R || n < 0) return DBOA_ERR_ARG;
    return n ? rot6d_fwd_launch(x6, R, n, ST(stream)) : DBOA_OK;
}
int dboa_rot6d_bwd(const float* x6, const float* dR, float* dx6, int n, dboa_stream_t stream) {
    if (!x6 || !dR || !dx6 || n < 0) return DBOA_ERR_ARG;
    return n ? rot6d_bwd_launch(x6, dR, dx6, n, ST(stream)) : DBOA_OK;
}
int dboa_rodrigues(const float* aa, float* R, int n, int kind, dboa_stream_t stream) {
    if (!aa || !R || n < 0 || kind < 0 || kind > 1) return DBOA_ERR_ARG;
    return n ? rodrigues_launch(aa, R, n, kind, ST(stream)) : DBOA_OK;
}
int dboa_rotmat_to_aa_fwd(const float* R, float* aa, int n, dboa_stream_t stream) {
    if (!R || !aa || n < 0) return DBOA_ERR_ARG;
    if (!n) return DBOA_OK;
    r2aa_fwd_kernel<<<ceil_div(n, 128), 128, 0, ST(stream)>>>(R, aa, n);
    return check_launch();
}
int dboa_rotmat_to_aa_bwd(const float* R, const float* daa, float* dR, int n, dboa_stream_t stream) {
    if (!R || !daa || !dR || n < 0) return DBOA_ERR_ARG;
    if (!n) return DBOA_OK;
    r2aa_bwd_kernel<<<ceil_div(n, 128), 128, 0, ST(stream)>>>(R, daa, dR, n);
    return check_launch();
}

long long dboa_smpl_tape_floats(int B) { return (long long)SmplTape::floats(B); }
long long dboa_smpl_scratch_floats(int B) { return (long long)SmplScratch::floats(B); }
int dboa_smpl_forward(const dboa_smpl_model* m, const float* betas, const float* rotmat, int B, float* vertices, float* joints, float* tape,
                      dboa_stream_t stream) {
    if (!m || !betas || !rotmat || !vertices || !joints || !tape || B < 1) return DBOA_ERR_ARG;
    return smpl_forward(*m, betas, rotmat, B, vertices, joints, tape, ST(stream));
}
int dboa_smpl_backward(const dboa_smpl_model* m, const float* rotmat, int B, const float* tape, const float* d_joints, float* scratch,
                       float* d_rotmat, float* d_betas, int accumulate, dboa_stream_t stream) {
    if (!m || !rotmat || !tape || !d_joints || !scratch || !d_rotmat || !d_betas || B < 1) return DBOA_ERR_ARG;
    return smpl_backward(*m, rotmat, B, tape, d_joints, scratch, d_rotmat, d_betas, accumulate, ST(stream));
}

int dboa_project_fwd(const float* cam, const float* j3d, float* p2d, int B, int NJ, dboa_stream_t stream) {
    if (!cam || !j3d || !p2d || B < 1 || NJ < 1) return DBOA_ERR_ARG;
    return project_fwd_launch(cam, j3d, p2d, B, NJ, ST(stream));
}
int dboa_project_bwd(const float* cam, const float* j3d, const float* dp2d, float* dj3d, float* dcam, int B, int NJ, int acc_j, int acc_cam,
                     dboa_stream_t stream) {
    if (!cam || !j3d || !dp2d || !dj3d || !dcam || B < 1 || NJ < 1) return DBOA_ERR_ARG;
    return project_bwd_launch(cam, j3d, dp2d, dj3d, dcam, B, NJ, acc_j, acc_cam, ST(stream));
}
int dboa_pose_prior(const float* rotmat, const float* means, const float* precisions, const float* neg_log_w, float* prior_b, float* d_rotmat,
                    float scale, int B, dboa_stream_t stream) {
    if (!rotmat || !means || !precisions || !neg_log_w || !prior_b || B < 1) return DBOA_ERR_ARG;
    return pose_prior_launch(rotmat, means, precisions, neg_log_w, prior_b, d_rotmat, scale, B, ST(stream));
}
int dboa_gmm_prior(const float* pose69, const float* means, const float* precisions, const float* neg_log_w, float* prior_b, float* d_pose,
                   float scale, int B, dboa_stream_t stream) {
    if (!pose69 || !means || !precisions || !neg_log_w || !prior_b || B < 1) return DBOA_ERR_ARG;
    return gmm_prior_launch(pose69, means, precisions, neg_log_w, prior_b, d_pose, scale, B, ST(stream));
}
int dboa_loss_multi(const dboa_loss_args* a, dboa_stream_t stream) {
    if (!a || !a->p2d || !a->j3d || !a->R || !a->beta || !a->terms) return DBOA_ERR_ARG;
    if (a->gt_s3d && !a->kp) return DBOA_ERR_ARG;
    return loss_multi_launch(*a, ST(stream));
}
int dboa_loss_motion(const float* p_cur, const float* p_hist, const float* kp_cur, const float* kp_hist, float weight, float* term,
                     float* dp_cur, float* dp_hist, int B, int accumulate_cur, dboa_stream_t stream) {
    if (!p_cur || !p_hist || !kp_cur || !kp_hist || !term || !dp_cur || !dp_hist || B < 1) return DBOA_ERR_ARG;
    return loss_motion_launch(p_cur, p_hist, kp_cur, kp_hist, weight, term, dp_cur, dp_hist, B, accumulate_cur, 25, 24, ST(stream));
}
int dboa_loss_motion_joints(const float* p_cur, const float* p_hist, const float* kp_cur, const float* kp_hist, float weight, float* term,
                            float* dp_cur, float* dp_hist, int B, int accumulate_cur, int first, int count, dboa_stream_t stream) {
    if (!p_cur || !p_hist || !kp_cur || !kp_hist || !term || !dp_cur || !dp_hist || B < 1) return DBOA_ERR_ARG;
    return loss_motion_launch(p_cur, p_hist, kp_cur, kp_hist, weight, term, dp_cur, dp_hist, B, accumulate_cur, first, count, ST(stream));
}

int dboa_sgd_update(const float* p, const float* g, float* out, float lr, long long n, dboa_stream_t stream) {
    if (!p || !g || !out || n < 0) return DBOA_ERR_ARG;
    return sgd_update(p, g, out, lr, (size_t)n, ST(stream));
}
int dboa_adam_ema(float* p, const float* g, float* m, float* v, float* teacher, long long n, float lr, float beta1, float beta2, float eps,
                  int step, float alpha, dboa_stream_t stream) {
    if (!p || !g || !m || !v || n < 0) return DBOA_ERR_ARG;
    return adam_ema(p, g, m, v, teacher, (size_t)n, lr, beta1, beta2, eps, step, alpha, 1.0f, ST(stream));
}
int dboa_adam_ema_scaled(float* p, const float* g, float* m, float* v, float* teacher, long long n, float lr, float beta1, float beta2, float eps,
                         int step, float alpha, float gscale, dboa_stream_t stream) {
    if (!p || !g || !m || !v || n < 0) return DBOA_ERR_ARG;
    return adam_ema(p, g, m, v, teacher, (size_t)n, lr, beta1, beta2, eps, step, alpha, gscale, ST(stream));
}
int dboa_fill_zero(void* dst, long long bytes, dboa_stream_t stream) {
    if (!dst || bytes < 0) return DBOA_ERR_ARG;
    return cudaMemsetAsync(dst, 0, (size_t)bytes, ST(stream)) == cudaSuccess ? DBOA_OK : DBOA_ERR_CUDA;
}
int dboa_copy_async(void* dst, const void* src, long long bytes, dboa_stream_t stream) {
    if (!dst || !src || bytes < 0) return DBOA_ERR_ARG;
    return cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyDeviceToDevice, ST(stream)) == cudaSuccess ? DBOA_OK : DBOA_ERR_CUDA;
}
int dboa_hmr_backward_buckets(void* ev0, void* ev1, void* ev2) {
    if (!ev0 || !ev1 || !ev2) return DBOA_ERR_ARG;
    hmr_arm_bucket_events(reinterpret_cast<cudaEvent_t>(ev0), reinterpret_cast<cudaEvent_t>(ev1), reinterpret_cast<cudaEvent_t>(ev2));
    return DBOA_OK;
}
long long dboa_hmr_bucket_offset(int k) { return hmr_bucket_offset(k); }
int dboa_ema_update(float* teacher, const float* p, long long n, float alpha, dboa_stream_t stream) {
    if (!teacher || !p || n < 0) return DBOA_ERR_ARG;
    return ema_update(teacher, p, (size_t)n, alpha, ST(stream));
}
int dboa_cosine_pairs(const float* const* a, const float* const* b, const long long* n, int npairs, float* partial, long long partial_floats,
                      float* out, float eps, dboa_stream_t stream) {
    if (!a || !b || !n || !partial || !out || npairs < 1 || npairs > 16) return DBOA_ERR_ARG;
    CosinePairs cp;
    cp.npairs = npairs;
    for (int i = 0; i < npairs; ++i) { cp.a[i] = a[i]; cp.b[i] = b[i]; cp.n[i] = n[i]; }
    return cosine_pairs(cp, partial, (size_t)partial_floats, out, nullptr, eps, ST(stream));
}
long long dboa_cosine_partial_floats(const long long* n, int npairs) {
    if (!n || npairs < 1 || npairs > 16) return DBOA_ERR_ARG;
    return cosine_partial_floats(n, npairs);
}
int dboa_cosine_terms(const float* const* a, const float* const* b, const long long* n, int npairs, float* partial, long long partial_floats,
                      double* terms, dboa_stream_t stream) {
    if (!a || !b || !n || !partial || !terms || npairs < 1 || npairs > 16) return DBOA_ERR_ARG;
    CosinePairs cp;
    cp.npairs = npairs;
    for (int i = 0; i < npairs; ++i) { cp.a[i] = a[i]; cp.b[i] = b[i]; cp.n[i] = n[i]; }
    return cosine_pairs(cp, partial, (size_t)partial_floats, nullptr, terms, 0.f, ST(stream));
}
int dboa_retrieval_nearest(const float* feat, const float* centers, int K, int D, int* best, float* dists, dboa_stream_t stream) {
    if (!feat || !centers || !best || !dists) return DBOA_ERR_ARG;
    return retrieval_nearest(feat, centers, K, D, best, dists, ST(stream));
}

int dboa_crop_resize_normalize(const void* img, int is_u8, int H, int W, int ul_x, int ul_y, int Hc, const float* wx, const int* sx, int Tx,
                               const float* wy, const int* sy, int Ty, int res, const float* mean3, const float* std3, float* tmp, float* out,
                               dboa_stream_t stream) {
    if (!img || !wx || !sx || !wy || !sy || !mean3 || !std3 || !tmp || !out) return DBOA_ERR_ARG;
    return crop_resize_normalize(img, is_u8, H, W, ul_x, ul_y, Hc, wx, sx, Tx, wy, sy, Ty, res, mean3, std3, tmp, out, ST(stream));
}
int dboa_keypoint_transform(const float* kp, int n, double t00, double t02, double t11, double t12, int res, float* out, dboa_stream_t stream) {
    if (!kp || !out || n < 0) return DBOA_ERR_ARG;
    return keypoint_transform(kp, n, t00, t02, t11, t12, res, out, ST(stream));
}

long long dboa_eval_scratch_floats(int B, int NJ) { return (long long)eval_scratch_floats(B, NJ); }
int dboa_eval_metrics(const float* pred_verts, const float* gt_verts_joints, const float* gt_verts_pve, const float* J_regressor, int NJ,
                      int NV, const int* joint_map, int n_map, float* scratch, float* out, int B, dboa_stream_t stream) {
    if (!pred_verts || !gt_verts_joints || !gt_verts_pve || !J_regressor || !joint_map || !scratch || !out) return DBOA_ERR_ARG;
    return eval_metrics(pred_verts, gt_verts_joints, gt_verts_pve, J_regressor, NJ, NV, joint_map, n_map, scratch, out, B, ST(stream));
}

}  // extern "C"
