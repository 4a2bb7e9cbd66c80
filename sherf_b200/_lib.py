"""ctypes binding of libsherf_b200.so (include/sherf_b200.h).  No fallback: if the library is missing or
fails to load, every product entry point raises -- there is deliberately no CPU / PyTorch path."""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

c_float_p = C.c_void_p          # device pointers travel as plain integers
c_int_p = C.c_void_p

MLP_FP32, MLP_TF32, MLP_TF32X3, MLP_BF16X3 = 0, 1, 2, 3
ABI_VERSION = 5


class SherfSmplModel(C.Structure):
    _fields_ = [('v_template', c_float_p), ('shapedirs', c_float_p), ('posedirs', c_float_p), ('j_regressor', c_float_p),
                ('weights', c_float_p), ('parents', C.c_int32 * 24), ('n_verts', C.c_int32)]


class SherfPose(C.Structure):
    _fields_ = [('poses', c_float_p), ('shapes', c_float_p), ('R', c_float_p), ('Th', c_float_p)]


class SherfFrame(C.Structure):
    _fields_ = [('target', SherfPose), ('canonical', SherfPose), ('obs', SherfPose), ('vertices', c_float_p),
                ('t_vertices', c_float_p), ('t_world_bounds', c_float_p), ('obs_K', c_float_p), ('obs_R', c_float_p),
                ('obs_T', c_float_p), ('sp_bounds', c_float_p), ('out_sh', C.c_int32 * 3)]


class SherfScene(C.Structure):
    _fields_ = [('planes', c_float_p), ('plane_ch', C.c_int32), ('plane_h', C.c_int32), ('plane_w', C.c_int32),
                ('obs_img', c_float_p), ('img_h', C.c_int32), ('img_w', C.c_int32),
                ('obs_feat', c_float_p), ('feat_ch', C.c_int32), ('feat_h', C.c_int32), ('feat_w', C.c_int32),
                ('vol', c_float_p * 3), ('vol_ch', C.c_int32 * 3), ('vol_dim', (C.c_int32 * 3) * 3)]


class SherfWeights(C.Structure):
    _fields_ = [('proj_w', c_float_p), ('proj_b', c_float_p), ('reproj_w', c_float_p), ('reproj_b', c_float_p),
                ('ln1_w', c_float_p), ('ln1_b', c_float_p), ('qkv_w', c_float_p), ('attn_out_w', c_float_p),
                ('attn_out_b', c_float_p), ('ln2_w', c_float_p), ('ln2_b', c_float_p), ('ff1_w', c_float_p),
                ('ff1_b', c_float_p), ('ff2_w', c_float_p), ('ff2_b', c_float_p), ('pts_w', c_float_p * 8),
                ('pts_b', c_float_p * 8), ('alpha_w', c_float_p), ('alpha_b', c_float_p), ('feature_w', c_float_p),
                ('feature_b', c_float_p), ('views_w', c_float_p), ('views_b', c_float_p), ('rgb_w', c_float_p),
                ('rgb_b', c_float_p)]


class SherfWeightGrads(C.Structure):
    """dL/d(param), same fields and order as SherfWeights (overwritten by sherf_render_backward; NULL = not wanted)."""
    _fields_ = list(SherfWeights._fields_)


class SherfOutGrads(C.Structure):
    _fields_ = [('rgb', c_float_p), ('depth', c_float_p), ('acc', c_float_p)]


class SherfInputGrads(C.Structure):
    _fields_ = [('planes', c_float_p), ('obs_feat', c_float_p), ('vol', c_float_p * 3)]


class SherfRays(C.Structure):
    _fields_ = [('origins', c_float_p), ('dirs', c_float_p), ('near_', c_float_p), ('far_', c_float_p),
                ('n_rays', C.c_int32), ('n_samples', C.c_int32), ('n_importance', C.c_int32), ('reserved', C.c_int32)]


class SherfOptions(C.Structure):
    _fields_ = [('white_back', C.c_int32), ('mlp_precision', C.c_int32), ('depth_clamp_min', C.c_float),
                ('depth_clamp_max', C.c_float), ('use_external_clamp', C.c_int32), ('density_noise', c_float_p),
                ('importance_u', c_float_p), ('density_noise_importance', c_float_p), ('weights_version', C.c_uint64), ('scene_version', C.c_uint64)]


class SherfOut(C.Structure):
    _fields_ = [('rgb', c_float_p), ('depth', c_float_p), ('acc', c_float_p)]


class SherfDebug(C.Structure):
    _fields_ = [('sample_vid', c_int_p), ('point_sample', c_int_p), ('point_vid3', c_int_p), ('point_can', c_float_p),
                ('point_cdir', c_float_p), ('point_uv', c_float_p), ('point_feat', c_float_p), ('point_tok', c_float_p),
                ('point_sigma', c_float_p), ('point_rgb', c_float_p), ('max_points', C.c_int64), ('max_feat_points', C.c_int64),
                ('coarse_weights', c_float_p), ('fine_depths', c_float_p), ('fine_bins', c_int_p), ('fine_sample_vid', c_int_p),
                ('fine_sigma', c_float_p), ('fine_rgb', c_float_p)]


class SherfSparseConv(C.Structure):
    _fields_ = [('weight', c_float_p), ('bn_weight', c_float_p), ('bn_bias', c_float_p), ('bn_mean', c_float_p), ('bn_var', c_float_p),
                ('c_in', C.c_int32), ('c_out', C.c_int32), ('kind', C.c_int32), ('reserved', C.c_int32)]


class SherfSparseEncoder(C.Structure):
    _fields_ = [('conv', SherfSparseConv * 13)]


class SherfSparseEncoderGrads(C.Structure):
    _fields_ = [('weight', c_float_p * 13), ('bn_weight', c_float_p * 13), ('bn_bias', c_float_p * 13)]


class SherfObservation(C.Structure):
    _fields_ = [('obs', SherfPose), ('canonical', SherfPose), ('obs_vertices', c_float_p), ('t_vertices', c_float_p), ('obs_K', c_float_p),
                ('obs_R', c_float_p), ('obs_T', c_float_p), ('faces', c_int_p), ('last_face', c_int_p), ('n_faces', C.c_int32),
                ('reserved', C.c_int32), ('obs_img', c_float_p), ('img_h', C.c_int32), ('img_w', C.c_int32), ('obs_feat', c_float_p),
                ('feat_ch', C.c_int32), ('feat_h', C.c_int32), ('feat_w', C.c_int32), ('reserved2', C.c_int32), ('proj_w', c_float_p),
                ('proj_b', c_float_p)]


EXPORTS = ['sherf_render_backward_after_forward', 'sherf_sparse_encoder_train_scratch_bytes', 'sherf_sparse_encode_train', 'sherf_sparse_encode_backward', 'sherf_prepare_observation_backward', 'sherf_backward_scratch_bytes', 'sherf_render_backward', 'sherf_smpl_vertices', 'sherf_count_survivors', 'sherf_observation_scratch_bytes', 'sherf_prepare_observation', 'sherf_debug_set_trace', 'sherf_sparse_encoder_scratch_bytes', 'sherf_sparse_encode', 'sherf_generate_rays', 'sherf_debug_sample_importance', 'sherf_debug_linear', 'sherf_scratch_bytes', 'sherf_render_forward', 'sherf_lbs_transforms', 'sherf_depth_range', 'sherf_last_error',
           'sherf_abi_version', 'sherf_last_launch_count', 'sherf_last_importance_point_count', 'sherf_set_profiling', 'sherf_last_stage_ms', 'sherf_last_host_us', 'sherf_nn_list_stats']

_lib = None


def lib_path() -> str:
    return _build.LIB_PATH


def load():
    """Returns the loaded library; raises RuntimeError (never falls back) if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise RuntimeError(f'{path} not found: build it with `python -m sherf_b200.build` (or __graft_entry__.build()); '
                           'sherf_b200 has no CPU or PyTorch fallback')
    lib = C.CDLL(path)
    lib.sherf_scratch_bytes.restype = C.c_size_t
    lib.sherf_scratch_bytes.argtypes = [C.POINTER(SherfScene), C.c_int32, C.c_int32, C.c_int32, C.c_int32]
    lib.sherf_render_forward.restype = C.c_int
    lib.sherf_render_forward.argtypes = [C.POINTER(SherfSmplModel), C.POINTER(SherfFrame), C.POINTER(SherfScene),
                                         C.POINTER(SherfWeights), C.POINTER(SherfRays), C.POINTER(SherfOptions),
                                         C.POINTER(SherfOut), C.POINTER(SherfDebug), C.c_void_p, C.c_size_t, C.c_void_p,
                                         C.POINTER(C.c_int64)]
    lib.sherf_backward_scratch_bytes.restype = C.c_size_t
    lib.sherf_backward_scratch_bytes.argtypes = [C.POINTER(SherfScene), C.c_int32, C.c_int32, C.c_int32]
    lib.sherf_render_backward.restype = C.c_int
    lib.sherf_render_backward.argtypes = [C.POINTER(SherfSmplModel), C.POINTER(SherfFrame), C.POINTER(SherfScene),
                                          C.POINTER(SherfWeights), C.POINTER(SherfRays), C.POINTER(SherfOptions),
                                          C.POINTER(SherfOutGrads), C.POINTER(SherfWeightGrads), C.POINTER(SherfInputGrads),
                                          C.c_void_p, C.c_size_t, C.c_void_p, C.POINTER(C.c_int64)]
    lib.sherf_render_backward_after_forward.restype = C.c_int
    lib.sherf_render_backward_after_forward.argtypes = lib.sherf_render_backward.argtypes[:-1] + [C.c_int64]
    lib.sherf_count_survivors.restype = C.c_int
    lib.sherf_count_survivors.argtypes = [C.POINTER(SherfSmplModel), C.POINTER(SherfFrame), C.POINTER(SherfScene), C.POINTER(SherfRays),
                                          C.POINTER(SherfOptions), C.c_void_p, C.c_size_t, C.c_void_p, C.POINTER(C.c_int64)]
    lib.sherf_smpl_vertices.restype = C.c_int
    lib.sherf_smpl_vertices.argtypes = [C.POINTER(SherfSmplModel), C.POINTER(SherfPose), C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.sherf_lbs_transforms.restype = C.c_int
    lib.sherf_lbs_transforms.argtypes = [C.POINTER(SherfSmplModel), C.POINTER(SherfPose), C.c_void_p, C.c_void_p, C.c_size_t,
                                         C.c_void_p]
    lib.sherf_depth_range.restype = C.c_int
    lib.sherf_depth_range.argtypes = [C.POINTER(SherfRays), C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_void_p, C.c_size_t,
                                      C.c_void_p]
    lib.sherf_debug_linear.restype = C.c_int
    lib.sherf_debug_linear.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.sherf_debug_sample_importance.restype = C.c_int
    lib.sherf_debug_sample_importance.argtypes = [C.POINTER(SherfRays), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.sherf_generate_rays.restype = C.c_int
    lib.sherf_generate_rays.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_int32, C.c_int32,
                                        C.POINTER(C.c_double), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.sherf_sparse_encoder_scratch_bytes.restype = C.c_size_t
    lib.sherf_sparse_encoder_scratch_bytes.argtypes = [C.c_int32, C.POINTER(C.c_int32)]
    lib.sherf_sparse_encode.restype = C.c_int
    lib.sherf_sparse_encode.argtypes = [C.POINTER(SherfSparseEncoder), C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.sherf_sparse_encoder_train_scratch_bytes.restype = C.c_size_t
    lib.sherf_sparse_encoder_train_scratch_bytes.argtypes = [C.c_int32, C.POINTER(C.c_int32)]
    lib.sherf_sparse_encode_train.restype = C.c_int
    lib.sherf_sparse_encode_train.argtypes = [C.POINTER(SherfSparseEncoder), C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.sherf_sparse_encode_backward.restype = C.c_int
    lib.sherf_sparse_encode_backward.argtypes = [C.POINTER(SherfSparseEncoder), C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.c_void_p, C.c_void_p,
                                                 C.c_void_p, C.POINTER(SherfSparseEncoderGrads), C.c_void_p, C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.sherf_prepare_observation_backward.restype = C.c_int
    lib.sherf_prepare_observation_backward.argtypes = [C.POINTER(SherfSmplModel), C.POINTER(SherfObservation), C.c_void_p, C.c_void_p, C.c_void_p,
                                                       C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.sherf_observation_scratch_bytes.restype = C.c_size_t
    lib.sherf_observation_scratch_bytes.argtypes = [C.c_int32]
    lib.sherf_prepare_observation.restype = C.c_int
    lib.sherf_prepare_observation.argtypes = [C.POINTER(SherfSmplModel), C.POINTER(SherfObservation), C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.POINTER(C.c_int32), C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.sherf_debug_set_trace.argtypes = [C.c_void_p]
    lib.sherf_last_error.restype = C.c_char_p
    lib.sherf_abi_version.restype = C.c_int
    lib.sherf_last_launch_count.restype = C.c_int64
    lib.sherf_last_importance_point_count.restype = C.c_int64
    lib.sherf_set_profiling.argtypes = [C.c_int]
    lib.sherf_last_stage_ms.restype = C.c_float
    lib.sherf_last_stage_ms.argtypes = [C.c_int]
    lib.sherf_nn_list_stats.restype = C.c_int
    lib.sherf_nn_list_stats.argtypes = [C.POINTER(C.c_double)]
    lib.sherf_last_host_us.restype = C.c_float
    lib.sherf_last_host_us.argtypes = [C.c_int]
    if lib.sherf_abi_version() != ABI_VERSION:
        raise RuntimeError('libsherf_b200.so ABI version mismatch')
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        raise RuntimeError(f'sherf_b200 error {rc}: {load().sherf_last_error().decode()}')
