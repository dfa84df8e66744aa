"""ctypes loader for the C-ABI library (include/smplpp_b200.h).  Fails loudly when the library is missing:
there is no CPU fallback and no alternate implementation."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# SMPLPP_B200_LIB: an instrumented build of the same library (scripts/build_dbg.sh), for kernel phase timers
LIB_PATH = os.environ.get("SMPLPP_B200_LIB") or os.path.join(HERE, "libsmplpp_b200.so")

c_f32p = C.POINTER(C.c_float)
c_f64p = C.POINTER(C.c_double)
c_i64p = C.POINTER(C.c_int64)
c_i32p = C.POINTER(C.c_int32)


class ModelDesc(C.Structure):
    _fields_ = [
        ("vertex_num", C.c_int64), ("face_num", C.c_int64), ("face_indices", c_i32p),
        ("shape_blend_shapes", c_f32p), ("pose_blend_shapes", c_f32p), ("vertices_template", c_f32p),
        ("joint_regressor", c_f32p), ("kinematic_tree", c_i64p), ("weights", c_f32p),
    ]


class VposerDesc(C.Structure):
    _fields_ = [("w0", c_f32p), ("b0", c_f32p), ("w3", c_f32p), ("b3", c_f32p), ("w5", c_f32p), ("b5", c_f32p)]


class MocapSummary(C.Structure):
    _fields_ = [("frames", C.c_int64), ("markers", C.c_int64), ("solved", C.c_int64), ("skipped", C.c_int64),
                ("failed", C.c_int64), ("mean_residual", C.c_double), ("max_residual", C.c_double)]


class IkOptions(C.Structure):
    _fields_ = [
        ("enable_vposer", C.c_int32), ("optimize_beta", C.c_int32), ("enable_qp", C.c_int32),
        ("enable_phi", C.c_int32), ("skip_if_too_few", C.c_int32), ("update_state", C.c_int32),
        ("normal_offset", C.c_float), ("normal_task_weight", C.c_float), ("phi_limit", C.c_float),
        ("delta_theta_reg", C.c_float), ("delta_phi_reg", C.c_float), ("delta_beta_reg", C.c_float),
        ("delta_beta_limit", C.c_float), ("vposer_latent_reg", C.c_float), ("vposer_hand_reg", C.c_float),
        ("reserved", C.c_int32 * 3),
    ]


# every symbol declared in include/smplpp_b200.h (tests check that the .so exports all of them)
EXPORTS = [
    "smplpp_last_error", "smplpp_launch_count", "smplpp_device_count",
    "smplpp_model_create", "smplpp_model_destroy", "smplpp_model_vertex_num", "smplpp_model_max_influences",
    "smplpp_forward_workspace_bytes", "smplpp_forward", "smplpp_forward_host", "smplpp_set_forward_variant",
    "smplpp_host_alloc", "smplpp_host_free", "smplpp_host_register", "smplpp_host_unregister",
    "smplpp_blend_shape", "smplpp_joint_regression", "smplpp_world_transformation", "smplpp_linear_blend_skinning",
    "smplpp_model_skinning", "smplpp_model_skinning34", "smplpp_normals",
    "smplpp_vposer_create", "smplpp_vposer_destroy", "smplpp_vposer_decode", "smplpp_rotmat_to_axis_angle",
    "smplpp_tasks_create", "smplpp_tasks_destroy", "smplpp_tasks_count", "smplpp_tasks_vertex_count", "smplpp_tasks_rest_shape",
    "smplpp_triangle_vertex_weights", "smplpp_ik_options_default", "smplpp_ik_theta_dim", "smplpp_ik_dim",
    "smplpp_task_positions", "smplpp_task_forward_workspace_bytes", "smplpp_task_forward", "smplpp_task_forward_host",
    "smplpp_closest_points", "smplpp_sweep_grid_bounds", "smplpp_sweep_grid_winding", "smplpp_ik_workspace_bytes", "smplpp_ik_step", "smplpp_ik_jacobian", "smplpp_ik_solve_host",
    "smplpp_ik_faces_workspace_bytes", "smplpp_ik_step_faces", "smplpp_ik_reproject_workspace_bytes", "smplpp_ik_reproject",
    "smplpp_ik_shared_beta_workspace_bytes", "smplpp_ik_shared_beta_reduce", "smplpp_ik_shared_beta_apply",
    "smplpp_ik_shared_beta_step", "smplpp_task_tangents", "smplpp_solve_mocap_motion",
    "smplpp_device_alloc", "smplpp_device_free", "smplpp_copy_to_device", "smplpp_copy_to_host", "smplpp_stream_synchronize",
    "smplpp_json_open", "smplpp_json_close", "smplpp_json_array", "smplpp_model_load_json", "smplpp_vposer_load_json",
    "smplpp_npz_open", "smplpp_model_load_npz",
    "smplpp_c3d_open", "smplpp_c3d_close", "smplpp_c3d_frame_count", "smplpp_c3d_point_count", "smplpp_c3d_frame_rate",
    "smplpp_c3d_label", "smplpp_c3d_units", "smplpp_c3d_find_label", "smplpp_c3d_read",
    "smplpp_write_mocap_body_yaml", "smplpp_mocap_body_open", "smplpp_mocap_body_close", "smplpp_mocap_body_task_count",
    "smplpp_mocap_body_task_name", "smplpp_mocap_body_get", "smplpp_write_motion_text", "smplpp_read_motion_text", "smplpp_write_obj",
]

_lib = None


class SmplppError(RuntimeError):
    """Counterpart of smplpp::Exception (src/toolbox/Exception.h:122): message "<module> Error: <text>"."""


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SmplppError(
                "smplpp_b200: CUDA extension %s is missing — run `python -m smplpp_b200.build` "
                "(there is no CPU fallback)" % LIB_PATH)
        _lib = C.CDLL(LIB_PATH)
        _lib.smplpp_last_error.restype = C.c_char_p
        _lib.smplpp_launch_count.restype = C.c_uint64
        _lib.smplpp_model_vertex_num.restype = C.c_int64
        for name in ("smplpp_c3d_frame_count", "smplpp_c3d_point_count", "smplpp_c3d_find_label"):
            getattr(_lib, name).restype = C.c_int64
        _lib.smplpp_c3d_frame_rate.restype = C.c_double
        _lib.smplpp_c3d_label.restype = C.c_char_p
        _lib.smplpp_c3d_units.restype = C.c_char_p
        _lib.smplpp_mocap_body_task_name.restype = C.c_char_p
        for name in ("smplpp_forward_workspace_bytes", "smplpp_ik_workspace_bytes",
                     "smplpp_ik_shared_beta_workspace_bytes", "smplpp_ik_faces_workspace_bytes",
                     "smplpp_ik_reproject_workspace_bytes"):
            if hasattr(_lib, name):
                getattr(_lib, name).restype = C.c_size_t
        _lib.smplpp_task_forward_workspace_bytes.restype = C.c_size_t
        _lib.smplpp_task_forward_workspace_bytes.argtypes = [C.c_void_p, C.c_int64]
        _lib.smplpp_task_forward.argtypes = [
            C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64,
            C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
        _lib.smplpp_task_forward_host.argtypes = [
            C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_float,
            C.c_void_p, C.c_void_p]
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        raise SmplppError(lib().smplpp_last_error().decode() or ("smplpp_b200 error %d" % rc))
