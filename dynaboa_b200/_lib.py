"""ctypes binding of libdynaboa_b200.so (the C ABI declared in include/dynaboa_b200.h).

There is no CPU fallback: if the shared object is missing or a call fails, this module raises.
Tensors cross the boundary as raw device pointers (``tensor.data_ptr()``) plus sizes; kernels are
enqueued on torch's current CUDA stream.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('DBOA_LIB_PATH') or os.path.join(_HERE, 'libdynaboa_b200.so')     # the override is for A/B experiments

P, I, L, F = C.c_void_p, C.c_int, C.c_longlong, C.c_float


class SmplModelStruct(C.Structure):
    _fields_ = [(n, P) for n in ('v_template', 'blend_dirs', 'J_template', 'J_shapedirs', 'parents', 'lbs_weights',
                                 'J_extra', 'joint_map', 'vertex_ids')]


class LossArgsStruct(C.Structure):
    _fields_ = ([('B', I)] + [(n, P) for n in ('p2d', 'j3d', 'R', 'beta', 'kp', 'prior_b', 't_p2d', 't_j3d', 't_beta',
                                                 't_R', 'gt_s3d')]
                + [('w', F * 8), ('terms', P), ('dp2d', P), ('dj3d', P), ('dR', P), ('dbeta', P), ('dR_accumulate', I), ('kp_first', I), ('kp_count', I)])


class FusedConvStruct(C.Structure):
    _fields_ = ([(n, P) for n in ('x', 'res', 'w', 'a_out', 'stats_out', 'stats2_out', 'part_in', 'part2_in', 'gamma', 'beta',
                                  'gamma2', 'beta2', 'y', 'part_out')]
                + [(n, I) for n in ('mode', 'Hi', 'Cin', 'Cout', 'k', 'stride', 'pad')])


class DgradFusedStruct(C.Structure):
    _fields_ = ([(n, P) for n in ('dz', 'y_c', 'w', 'stats_c', 'sums_c', 'gamma_c', 'dy_out', 'addend', 'out', 'mask')]
                + [('prep_y', P * 2), ('prep_stats', P * 2), ('prep_gamma', P * 2), ('prep_sums', P * 2), ('prep_dgb', P * 2), ('nprep', I),
                   ('accumulate', I)])


# name -> (restype, argtypes); mirrors include/dynaboa_b200.h one to one
SIGNATURES = {
    'dboa_version': (C.c_char_p, []),
    'dboa_last_cuda_error': (I, []),
    'dboa_launch_count': (L, []),
    'dboa_set_tensor_core_conv': (I, [I]),
    'dboa_set_fused_forward': (I, [I]),
    'dboa_get_fused_forward': (I, []),
    'dboa_set_fused_backward': (I, [I]),
    'dboa_set_forward_cta_budget': (I, [I]),
    'dboa_set_split_limits': (I, [I, I, I, I]),
    'dboa_last_wide_plan': (I, [I, C.POINTER(L)]),
    'dboa_set_operand_tmem': (I, [I]),
    'dboa_get_operand_tmem': (I, []),
    'dboa_set_chain_flags': (I, [I]),
    'dboa_get_chain_flags': (I, []),
    'dboa_selftest_map_cache': (I, [I, I, I]),
    'dboa_dgrad_fused': (I, [C.POINTER(DgradFusedStruct), I, I, I, I, I, P]),
    'dboa_conv_fused_part_floats': (L, [I, I, I]),
    'dboa_conv_fused_fwd': (I, [C.POINTER(FusedConvStruct), I, I, P]),
    'dboa_hmr_num_params': (I, []),
    'dboa_hmr_arena_floats': (L, []),
    'dboa_hmr_param_info': (I, [I, C.c_char_p, I, C.POINTER(L), C.POINTER(I), C.POINTER(L), C.POINTER(L)]),
    'dboa_hmr_tape_floats': (L, [I]),
    'dboa_hmr_scratch_floats': (L, [I]),
    'dboa_hmr_feature_info': (I, [I, I, C.POINTER(L), C.POINTER(I), C.POINTER(L), C.POINTER(L)]),
    'dboa_hmr_forward': (I, [P, P, P, P, P, I, P, P, P, P, P, P, P, P]),
    'dboa_hmr_backward': (I, [P, P, I, I, P, P, P, P, P, P]),
    'dboa_conv2d_fwd': (I, [P, P, P, I, I, I, I, I, I, I, I, I, P, L, P]),
    'dboa_conv2d_dgrad': (I, [P, P, P, I, I, I, I, I, I, I, I, I, I, P, L, P]),
    'dboa_conv2d_wgrad': (I, [P, P, P, I, I, I, I, I, I, I, I, I, P, L, P]),
    'dboa_conv1x1_tc_fwd': (I, [P, P, P, I, I, I, P, L, P]),
    'dboa_conv2d_tc_fwd': (I, [P, P, P, I, I, I, I, I, I, I, I, I, P]),
    'dboa_conv2d_tc_dgrad': (I, [P, P, P, I, I, I, I, I, I, I, I, I, I, P]),
    'dboa_conv2d_tc_wgrad': (I, [P, P, P, I, I, I, I, I, I, I, I, I, P]),
    'dboa_conv2d_wgrad_tma': (I, [P, P, P, I, I, I, I, I, I, I, I, I, P]),
    'dboa_gn_partial_floats': (L, [I, I, I]),
    'dboa_gn_bwd_partial_floats': (L, [I, I, I]),
    'dboa_groupnorm_fwd': (I, [P, P, P, P, P, P, P, I, I, I, I, P]),
    'dboa_groupnorm_bwd': (I, [P, P, P, P, P, P, P, P, P, I, I, I, P]),
    'dboa_maxpool_fwd': (I, [P, P, P, I, I, I, I, P]),
    'dboa_maxpool_bwd': (I, [P, P, P, I, I, I, I, P]),
    'dboa_rot6d_fwd': (I, [P, P, I, P]),
    'dboa_rot6d_bwd': (I, [P, P, P, I, P]),
    'dboa_rodrigues': (I, [P, P, I, I, P]),
    'dboa_rotmat_to_aa_fwd': (I, [P, P, I, P]),
    'dboa_rotmat_to_aa_bwd': (I, [P, P, P, I, P]),
    'dboa_smpl_tape_floats': (L, [I]),
    'dboa_smpl_scratch_floats': (L, [I]),
    'dboa_smpl_forward': (I, [C.POINTER(SmplModelStruct), P, P, I, P, P, P, P]),
    'dboa_smpl_backward': (I, [C.POINTER(SmplModelStruct), P, I, P, P, P, P, P, I, P]),
    'dboa_project_fwd': (I, [P, P, P, I, I, P]),
    'dboa_project_bwd': (I, [P, P, P, P, P, I, I, I, I, P]),
    'dboa_pose_prior': (I, [P, P, P, P, P, P, F, I, P]),
    'dboa_gmm_prior': (I, [P, P, P, P, P, P, F, I, P]),
    'dboa_loss_multi': (I, [C.POINTER(LossArgsStruct), P]),
    'dboa_loss_motion': (I, [P, P, P, P, F, P, P, P, I, I, P]),
    'dboa_loss_motion_joints': (I, [P, P, P, P, F, P, P, P, I, I, I, I, P]),
    'dboa_sgd_update': (I, [P, P, P, F, L, P]),
    'dboa_adam_ema': (I, [P, P, P, P, P, L, F, F, F, F, I, F, P]),
    'dboa_ema_update': (I, [P, P, L, F, P]),
    'dboa_adam_ema_scaled': (I, [P, P, P, P, P, L, F, F, F, F, I, F, F, P]),
    'dboa_fill_zero': (I, [P, L, P]),
    'dboa_copy_async': (I, [P, P, L, P]),
    'dboa_hmr_backward_buckets': (I, [P, P, P]),
    'dboa_hmr_bucket_offset': (L, [I]),
    'dboa_cosine_pairs': (I, [C.POINTER(P), C.POINTER(P), C.POINTER(L), I, P, L, P, F, P]),
    'dboa_cosine_partial_floats': (L, [C.POINTER(L), I]),
    'dboa_cosine_terms': (I, [C.POINTER(P), C.POINTER(P), C.POINTER(L), I, P, L, P, P]),
    'dboa_retrieval_nearest': (I, [P, P, I, I, P, P, P]),
    'dboa_crop_resize_normalize': (I, [P, I, I, I, I, I, I, P, P, I, P, P, I, I, P, P, P, P, P]),
    'dboa_keypoint_transform': (I, [P, I, C.c_double, C.c_double, C.c_double, C.c_double, I, P, P]),
    'dboa_eval_scratch_floats': (L, [I, I]),
    'dboa_eval_metrics': (I, [P, P, P, P, I, I, P, I, P, P, I, P]),
}

_ERRORS = {-1: 'DBOA_ERR_ARG', -2: 'DBOA_ERR_SHAPE', -3: 'DBOA_ERR_CUDA', -4: 'DBOA_ERR_UNSUPPORTED'}
_lib = None


def load():
    """Load the shared library (once) and attach argument types.  Raises if it is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f'{LIB_PATH} is missing: run `python -m dynaboa_b200.build` (nvcc, sm_100a). '
                               'dynaboa_b200 has no CPU or PyTorch fallback.')
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def ptr(t):
    """Device pointer of a tensor (None -> NULL).  The tensor must be a contiguous-enough fp32/int32 view."""
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def check(status, what):
    if status != 0:
        lib = load()
        extra = f' (cudaError {lib.dboa_last_cuda_error()})' if status == -3 else ''
        raise RuntimeError(f'{what} failed: {_ERRORS.get(status, status)}{extra}')


def call(name, *args):
    """Invoke an int-returning entry point and raise on a non-zero status."""
    check(getattr(load(), name)(*args), name)


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError('dynaboa_b200 runs on CUDA tensors only (no CPU path)')
