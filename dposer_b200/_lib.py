"""ctypes binding of libdposer_b200.so (the C ABI declared in include/dposer_b200.h).

There is NO CPU fallback: if the library is missing, or there is no CUDA device, every
compute call raises.  Error codes map onto the exception types the reference raises
(ValueError / NotImplementedError / RuntimeError).
"""
import ctypes as C
import os

from . import build as _build

OK, EINVAL, ECUDA, ENOMEM, EUNSUPPORTED = 0, -1, -2, -3, -4
ENGINE_AUTO, ENGINE_FP32, ENGINE_TC = 0, 1, 2
SAMPLER_IMPUTE, SAMPLER_NOISE_GIVEN = 1 << 4, 1 << 5
LBS_CONST_TAIL, LBS_NO_SAVE = 1 << 4, 1 << 5
COEF_STRIDE = 8
POSE_DIM, HIDDEN, EMBED, NUM_DENSE = 63, 1024, 512, 5
POSE_DIM_ROT6D = 126
POSE_DIMS = (POSE_DIM, POSE_DIM_ROT6D)      # pose widths a score handle can be built for (axis-angle, rot6d)

_f32p = C.POINTER(C.c_float)
_i32p = C.POINTER(C.c_int32)


class ScoreWeights(C.Structure):
    _fields_ = [('pre_w', _f32p), ('pre_b', _f32p), ('pre_t_w', _f32p), ('pre_t_b', _f32p),
                ('pre_gn_w', _f32p), ('pre_gn_b', _f32p), ('temb_w', _f32p), ('temb_b', _f32p),
                ('blk_w', _f32p * 4), ('blk_b', _f32p * 4), ('blk_t_w', _f32p * 4), ('blk_t_b', _f32p * 4),
                ('blk_gn_w', _f32p * 4), ('blk_gn_b', _f32p * 4), ('post_w', _f32p), ('post_b', _f32p),
                ('emb_freqs', _f32p)]


class StepTables(C.Structure):
    _fields_ = [('n_steps', C.c_int), ('coef', C.c_void_p), ('time_table', C.c_void_p)]


class BodyTensors(C.Structure):
    _fields_ = [('V', C.c_int), ('J', C.c_int), ('S', C.c_int),
                ('v_template', _f32p), ('shapedirs', _f32p), ('posedirs', _f32p), ('J_regressor', _f32p),
                ('lbs_weights', _f32p), ('parents', _i32p), ('n_extra', C.c_int), ('extra_vids', _i32p),
                ('n_lmk', C.c_int), ('lmk_faces', _i32p), ('lmk_bary', _f32p)]


EXPORTS = ['dpb_version', 'dpb_last_error', 'dpb_device_info', 'dpb_score_create', 'dpb_score_create_dim',
           'dpb_score_pose_dim', 'dpb_normal_fill_dim', 'dpb_langevin_norms_dim', 'dpb_langevin_update_dim', 'dpb_score_destroy',
           'dpb_score_time_table', 'dpb_score_workspace_bytes', 'dpb_score_forward', 'dpb_score_jvp',
           'dpb_score_jvp_workspace_bytes', 'dpb_sampler_run_pc', 'dpb_sampler_pc_workspace_bytes', 'dpb_sampler_run',
           'dpb_langevin_norms', 'dpb_langevin_update', 'dpb_normal_fill', 'dpb_prior_loss', 'dpb_lbs_create',
           'dpb_lbs_destroy', 'dpb_lbs_set_const_tail', 'dpb_lbs_num_joints_out', 'dpb_lbs_workspace_bytes', 'dpb_lbs_forward',
           'dpb_lbs_backward', 'dpb_lbs_backward_scratch_bytes', 'dpb_lbs_backward_scratch_bytes_joints', 'dpb_apd_partial', 'dpb_mean_point_error', 'dpb_fit_loss',
           'dpb_motion_loss', 'dpb_camera_fit_loss', 'dpb_adam_step', 'dpb_affine_cols', 'dpb_axis_to_rot6d_cols',
           'dpb_axis_to_rot6d_cols_vjp', 'dpb_joint_map_gather',
           'dpb_joint_map_scatter', 'dpb_masked_mse_grad', 'dpb_seq_smooth3', 'dpb_train_create', 'dpb_train_destroy',
           'dpb_train_loss_grad', 'dpb_train_adam_scratch_bytes', 'dpb_train_grad_norm', 'dpb_train_adam', 'dpb_ema_update', 'dpb_train_set_seed_pointer', 'dpb_gemm_nt_workspace_bytes', 'dpb_gemm_nt', 'dpb_train_forward', 'dpb_train_backward', 'dpb_rows_axpby', 'dpb_weighted_sqdiff', 'dpb_rk45_stage', 'dpb_rk45_scratch_bytes', 'dpb_rk45_error',
           'dpb_pf_ode_rhs', 'dpb_selfisect_create', 'dpb_selfisect_destroy', 'dpb_selfisect_workspace_bytes',
           'dpb_selfisect_run', 'dpb_procrustes']

_lib = None


def library_path():
    # DPB_LIBRARY: developer knob, points at an instrumented build (build.py with DPB_BUILD_DEFINES)
    return os.environ.get('DPB_LIBRARY') or _build.LIB


def load():
    """Load (never build) the in-tree shared library; raise loudly if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise RuntimeError(f'{path} is missing: run `python -c "import __graft_entry__ as g; g.build()"` '
                           '(dposer_b200 has no CPU fallback)')
    lib = C.CDLL(path)
    vp, i64, u64, f32, sz = C.c_void_p, C.c_int64, C.c_uint64, C.c_float, C.c_size_t
    lib.dpb_version.restype = C.c_int
    lib.dpb_last_error.restype = C.c_char_p
    lib.dpb_device_info.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.dpb_score_create.argtypes = [C.POINTER(vp), C.POINTER(ScoreWeights), C.c_int]
    lib.dpb_score_create_dim.argtypes = [C.POINTER(vp), C.POINTER(ScoreWeights), C.c_int, C.c_int]
    lib.dpb_score_pose_dim.argtypes = [vp]
    lib.dpb_score_destroy.argtypes = [vp]
    lib.dpb_score_time_table.argtypes = [vp, vp, C.c_int, vp, vp]
    lib.dpb_score_workspace_bytes.argtypes = [vp, i64, C.c_int]
    lib.dpb_score_workspace_bytes.restype = sz
    lib.dpb_score_forward.argtypes = [vp, vp, vp, vp, vp, f32, vp, i64, C.c_int, vp, sz, vp]
    lib.dpb_sampler_run.argtypes = [vp, vp, C.POINTER(StepTables), vp, vp, vp, u64, u64, vp, vp, i64, C.c_int, vp,
                                    sz, vp]
    lib.dpb_langevin_norms.argtypes = [vp, vp, vp, i64, vp]
    lib.dpb_langevin_update.argtypes = [vp, vp, vp, vp, vp, f32, f32, i64, vp]
    lib.dpb_normal_fill.argtypes = [vp, i64, u64, u64, C.c_int, vp]
    lib.dpb_langevin_norms_dim.argtypes = [vp, vp, vp, i64, C.c_int, vp]
    lib.dpb_langevin_update_dim.argtypes = [vp, vp, vp, vp, vp, f32, f32, i64, C.c_int, vp]
    lib.dpb_normal_fill_dim.argtypes = [vp, i64, u64, u64, C.c_int, C.c_int, vp]
    lib.dpb_prior_loss.argtypes = [vp, vp, vp, f32, f32, f32, C.c_int, f32, vp, u64, u64, vp, vp, vp, i64, C.c_int,
                                   vp, sz, vp]
    lib.dpb_sampler_pc_workspace_bytes.argtypes = [vp, i64]
    lib.dpb_sampler_pc_workspace_bytes.restype = sz
    lib.dpb_sampler_run_pc.argtypes = [vp, vp, C.POINTER(StepTables), vp, vp, f32, vp, vp, vp, C.c_uint64, C.c_uint64, vp,
                                       vp, i64, C.c_int, vp, sz, vp]
    lib.dpb_score_jvp_workspace_bytes.argtypes = [vp, i64]
    lib.dpb_score_jvp_workspace_bytes.restype = sz
    lib.dpb_score_jvp.argtypes = [vp, vp, vp, vp, vp, vp, f32, vp, vp, i64, vp, sz, vp]
    lib.dpb_lbs_create.argtypes = [C.POINTER(vp), C.POINTER(BodyTensors), C.c_int]
    lib.dpb_lbs_destroy.argtypes = [vp]
    lib.dpb_lbs_set_const_tail.argtypes = [vp, C.c_int, _f32p]
    lib.dpb_lbs_num_joints_out.argtypes = [vp]
    lib.dpb_lbs_workspace_bytes.argtypes = [vp, i64, C.c_int]
    lib.dpb_lbs_workspace_bytes.restype = sz
    lib.dpb_lbs_forward.argtypes = [vp, vp, vp, vp, vp, vp, i64, C.c_int, vp, sz, vp]
    lib.dpb_lbs_backward.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, i64, C.c_int, vp, sz, vp, sz, vp]
    lib.dpb_lbs_backward_scratch_bytes.argtypes = [vp, i64]
    lib.dpb_lbs_backward_scratch_bytes.restype = sz
    lib.dpb_lbs_backward_scratch_bytes_joints.argtypes = [vp, i64]
    lib.dpb_lbs_backward_scratch_bytes_joints.restype = sz
    lib.dpb_fit_loss.argtypes = [vp, vp, vp, vp, vp, C.c_int, vp, C.c_int, C.c_int, vp, f32, f32, f32, f32, vp, vp, vp,
                                 vp, vp, i64, vp]
    lib.dpb_apd_partial.argtypes = [vp, i64, C.c_int, i64, i64, vp, vp]
    lib.dpb_motion_loss.argtypes = [vp, vp, vp, i64, C.c_int, C.c_int, C.c_int, C.c_int, f32, f32, vp, vp, vp, vp]
    lib.dpb_camera_fit_loss.argtypes = [vp, vp, vp, vp, vp, vp, vp, f32, f32, C.c_int, vp, vp, vp, i64, vp]
    lib.dpb_adam_step.argtypes = [vp, i64, vp, vp, vp, i64, f32, vp, i64, f32, vp, vp, i64, f32, i64, C.c_int, f32, f32,
                                  f32, f32, C.c_int, vp]
    lib.dpb_seq_smooth3.argtypes = [vp, vp, i64, C.c_int, C.c_int, f32, f32, f32, C.c_int, vp]
    lib.dpb_masked_mse_grad.argtypes = [vp, vp, vp, vp, i64, vp]
    lib.dpb_affine_cols.argtypes = [vp, i64, vp, vp, vp, i64, i64, C.c_int, C.c_int, f32, vp]
    lib.dpb_axis_to_rot6d_cols.argtypes = [vp, i64, vp, vp, vp, i64, i64, C.c_int, vp]
    lib.dpb_axis_to_rot6d_cols_vjp.argtypes = [vp, i64, vp, vp, i64, vp, i64, i64, C.c_int, vp]
    lib.dpb_joint_map_gather.argtypes = [vp, C.c_int, vp, C.c_int, vp, i64, vp]
    lib.dpb_joint_map_scatter.argtypes = [vp, C.c_int, vp, C.c_int, vp, i64, vp]
    lib.dpb_train_create.argtypes = [C.POINTER(vp), i64, C.c_int]
    lib.dpb_train_destroy.argtypes = [vp]
    lib.dpb_train_loss_grad.argtypes = [vp, C.POINTER(ScoreWeights), C.POINTER(ScoreWeights), vp, vp, vp, vp, f32, u64, vp,
                                        vp, vp]
    lib.dpb_train_adam_scratch_bytes.restype = sz
    lib.dpb_train_forward.argtypes = [vp, C.POINTER(ScoreWeights), vp, vp, vp, f32, u64, vp, vp]
    lib.dpb_train_backward.argtypes = [vp, C.POINTER(ScoreWeights), C.POINTER(ScoreWeights), vp, vp, f32, u64, C.c_int, vp, vp]
    lib.dpb_rows_axpby.argtypes = [vp, vp, vp, vp, vp, C.c_int, i64, vp]
    lib.dpb_weighted_sqdiff.argtypes = [vp, vp, vp, i64, i64, f32, vp, vp, vp, vp]
    lib.dpb_train_grad_norm.argtypes = [vp, i64, vp, vp]
    lib.dpb_train_adam.argtypes = [vp, vp, vp, vp, i64, f32, f32, f32, f32, f32, i64, f32, vp, vp, vp]
    lib.dpb_train_set_seed_pointer.argtypes = [vp, vp]
    lib.dpb_ema_update.argtypes = [vp, vp, i64, f32, vp, vp]
    lib.dpb_gemm_nt_workspace_bytes.argtypes = [C.c_int, C.c_int, C.c_int]
    lib.dpb_gemm_nt_workspace_bytes.restype = sz
    lib.dpb_gemm_nt.argtypes = [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, sz, vp]
    f64 = C.c_double
    lib.dpb_rk45_stage.argtypes = [vp, vp, i64, f64, C.c_int, vp, vp, i64, vp]
    lib.dpb_rk45_scratch_bytes.restype = sz
    lib.dpb_rk45_error.argtypes = [vp, vp, vp, i64, f64, f64, f64, vp, vp]
    lib.dpb_pf_ode_rhs.argtypes = [vp, vp, vp, vp, f32, f32, vp, i64, vp]
    lib.dpb_mean_point_error.argtypes = [vp, vp, i64, C.c_int, vp, C.c_int, vp, vp]
    lib.dpb_selfisect_create.argtypes = [C.POINTER(vp), _i32p, C.c_int, C.c_int, C.c_int]
    lib.dpb_selfisect_destroy.argtypes = [vp]
    lib.dpb_selfisect_workspace_bytes.argtypes = [vp, i64]
    lib.dpb_selfisect_workspace_bytes.restype = sz
    lib.dpb_selfisect_run.argtypes = [vp, vp, i64, vp, vp, vp, sz, vp]
    lib.dpb_procrustes.argtypes = [vp, vp, i64, C.c_int, vp, C.c_int, vp, vp, vp, vp]
    for name in EXPORTS:
        fn = getattr(lib, name)
        if name not in ('dpb_last_error', 'dpb_score_workspace_bytes', 'dpb_lbs_workspace_bytes',
                        'dpb_lbs_backward_scratch_bytes', 'dpb_lbs_backward_scratch_bytes_joints',
                        'dpb_score_jvp_workspace_bytes', 'dpb_sampler_pc_workspace_bytes',
                        'dpb_train_adam_scratch_bytes', 'dpb_gemm_nt_workspace_bytes', 'dpb_rk45_scratch_bytes',
                        'dpb_selfisect_workspace_bytes'):
            fn.restype = C.c_int
    _lib = lib
    return lib


def check(rc, what=''):
    """Translate a DPB_E* code into the exception the reference would raise."""
    if rc == OK:
        return
    msg = load().dpb_last_error().decode() or what
    if rc == EINVAL:
        raise ValueError(msg)
    if rc == EUNSUPPORTED:
        raise NotImplementedError(msg)
    if rc == ENOMEM:
        raise MemoryError(msg)
    raise RuntimeError(msg)


def ptr(t):
    """Device (or host) pointer of a torch tensor, or None."""
    return None if t is None else C.c_void_p(t.data_ptr())


def host_f32(t):
    """A contiguous fp32 host array view and its ctypes pointer (keeps the array alive)."""
    import numpy as np
    a = np.ascontiguousarray(t.detach().cpu().float().numpy() if hasattr(t, 'detach') else np.asarray(t, np.float32))
    return a, a.ctypes.data_as(_f32p)


def host_i32(t):
    import numpy as np
    a = np.ascontiguousarray(np.asarray(t.detach().cpu().numpy() if hasattr(t, 'detach') else t, dtype=np.int32))
    return a, a.ctypes.data_as(_i32p)


def current_stream(device):
    import torch
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(t, name):
    if not t.is_cuda:
        raise RuntimeError(f'dposer_b200: `{name}` must live on a CUDA device -- there is no CPU fallback '
                           f'(got device {t.device})')
