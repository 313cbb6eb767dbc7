"""ctypes binding of include/b200_gripper_sim.h (libgripper_sim_b200.so).

There is no fallback: if the library is missing or fails to load, importing this module raises.
"""
import ctypes as C
import os

from . import build as _build

HERE = os.path.dirname(os.path.abspath(__file__))


class GrsConfig(C.Structure):
    """grs_config — the fields RobotEnv reads from its config Namespace (reference config/base_config.py:13-43)."""
    _fields_ = [("max_steps", C.c_int32), ("time_horizon", C.c_int32), ("include_roll", C.c_int32),
                ("full_observation", C.c_int32), ("im_reward", C.c_int32), ("her_buffer", C.c_int32),
                ("direction", C.c_int32), ("width", C.c_int32), ("height", C.c_int32), ("auto_reset", C.c_int32),
                ("pos_tolerance", C.c_float), ("grasp_tolerance", C.c_float), ("max_translation", C.c_float),
                ("max_rotation", C.c_float), ("reset_noise_xy", C.c_float), ("reset_noise_yaw", C.c_float), ("seed", C.c_uint32)]


# record layouts (include/b200_gripper_sim.h)
INFO = dict(REWARD=0, DONE=1, STATUS=2, GRASP=3, PHEROMONE=4, OBJECT_GRASPED=5, GRIPPER_OPEN=6, REACHED_TARGET=7,
            REACHED_INITIAL=8, FAIL=9, NSUB_A=10, NSUB_B=11, NSUB_C=12, TOTAL_DISTANCE=13, LINE_DISTANCE=14,
            INIT_OBJ_POS=15, FINAL_OBJ_POS=18, GRIPPER_POS=21, ACHIEVED=24, DESIRED=26, SOLVER_ITERS=28, NCON_MAX=29,
            FLAGS=30, EPISODE_STEP=31, EPISODE_RETURN=32, EPISODE_SUBSTEPS=33, TARGET_QPOS=34, OBJECT=39, STRIDE=40)
STATE_STRIDE, RENDER_STATE_STRIDE, DEBUG_STRIDE = 64, 96, 2048
# debug-step dump layout (csrc/env_kernels.cuh DBG_*)
DBG = dict(M=0, BIAS=169, FSMOOTH=182, ASMOOTH=195, NCON=208, NEFC=209, NLIM=210, ITERS=211, QACC=212, FCON=225, D=238,
           AREF=293, FORCE=348, J=403, CONTACT=1118, MU=1298)

SYMBOLS = ["grs_last_error", "grs_default_config", "grs_create", "grs_create_scenes", "grs_num_scenes", "grs_destroy", "grs_num_envs", "grs_action_dim",
           "grs_obs_shape", "grs_stream", "grs_reset", "grs_step", "grs_step_host", "grs_reset_host", "grs_substep",
           "grs_buffer", "grs_get_state", "grs_set_state", "grs_max_contacts", "grs_get_contacts", "grs_debug_step",
           "grs_model_get", "grs_model_get_int", "grs_model_names", "grs_compile_only", "grs_render", "grs_launch_count",
           "grs_step_kernel_ms", "grs_async_begin", "grs_async_send", "grs_async_recv", "grs_async_end", "grs_async_status"]
SYMBOLS += ["grp_last_error", "grp_create", "grp_destroy", "grp_num_params", "grp_set_params", "grp_get_params", "grp_forward",
            "grp_buffer", "grp_shape", "grp_launch_count", "grp_stream"]

SYMBOLS += ["grl_last_error", "grl_gae", "grl_adam_step"]
SYMBOLS += ["grl_replay_create", "grl_replay_destroy", "grl_replay_begin", "grl_replay_add", "grl_replay_size", "grl_replay_sample",
            "grl_replay_buffer", "grl_replay_begin_indexed", "grl_replay_add_indexed", "grl_replay_status"]

_lib = None


def lib_path():
    # GRS_LIB: an alternative build of the library (development A/B runs of kernel variants); default = the in-tree build
    return os.environ.get("GRS_LIB") or _build.LIB


def load():
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise ImportError("native library %s is missing: run `python -m mujoco_rl_manipulate_unknown_objects_b200.build` "
                          "(there is no CPU fallback)" % path)
    L = C.CDLL(path)
    vp, i32, i64, u64, f32p = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.POINTER(C.c_float)
    L.grs_last_error.restype = C.c_char_p
    L.grs_default_config.argtypes = [C.POINTER(GrsConfig)]
    L.grs_create.restype = vp
    L.grs_create.argtypes = [C.c_char_p, i32, C.POINTER(GrsConfig), i32]
    L.grs_create_scenes.restype = vp
    L.grs_create_scenes.argtypes = [C.POINTER(C.c_char_p), i32, i32, C.POINTER(GrsConfig), i32]
    L.grs_num_scenes.restype = i32
    L.grs_num_scenes.argtypes = [vp]
    L.grs_compile_only.restype = vp
    L.grs_compile_only.argtypes = [C.c_char_p]
    L.grs_destroy.argtypes = [vp]
    for f in (L.grs_num_envs, L.grs_action_dim):
        f.restype = i32
        f.argtypes = [vp]
    L.grs_obs_shape.argtypes = [vp, C.POINTER(i32)]
    L.grs_stream.restype = vp
    L.grs_stream.argtypes = [vp]
    L.grs_reset.argtypes = [vp, vp, vp]
    L.grs_step.argtypes = [vp, vp, vp]
    L.grs_step_host.argtypes = [vp] + [vp] * 8
    L.grs_reset_host.argtypes = [vp, vp, vp, vp]
    L.grs_substep.argtypes = [vp, i32, vp]
    L.grs_buffer.argtypes = [vp, C.c_char_p, C.POINTER(vp), C.POINTER(u64)]
    L.grs_get_state.argtypes = [vp] + [vp] * 6
    L.grs_set_state.argtypes = [vp] + [vp] * 6
    L.grs_max_contacts.restype = i32
    L.grs_get_contacts.argtypes = [vp] + [vp] * 5
    L.grs_debug_step.argtypes = [vp]
    L.grs_model_get.restype = i64
    L.grs_model_get.argtypes = [vp, C.c_char_p, vp, i64]
    L.grs_model_get_int.restype = i64
    L.grs_model_get_int.argtypes = [vp, C.c_char_p, vp, i64]
    L.grs_model_names.restype = i64
    L.grs_model_names.argtypes = [vp, C.c_char_p, C.c_char_p, i64]
    L.grs_render.argtypes = [vp, i32, i32, i32, vp, vp, vp]
    L.grs_launch_count.restype = u64
    L.grs_launch_count.argtypes = [vp]
    L.grs_step_kernel_ms.restype = C.c_float
    L.grs_step_kernel_ms.argtypes = [vp, i32]
    L.grs_async_begin.argtypes = [vp, i32, vp]
    L.grs_async_send.argtypes = [vp, vp, vp, i32, vp]
    L.grs_async_recv.argtypes = [vp, vp, vp]
    L.grs_async_end.argtypes = [vp]
    L.grs_async_status.argtypes = [vp, C.POINTER(i64)]
    L.grp_last_error.restype = C.c_char_p
    L.grp_create.restype = vp
    L.grp_create.argtypes = [i32, i32, i32, i32, i32, i32]
    L.grp_destroy.argtypes = [vp]
    L.grp_num_params.restype = i64
    L.grp_num_params.argtypes = [vp]
    L.grp_set_params.argtypes = [vp, vp, i64]
    L.grp_get_params.argtypes = [vp, vp, i64]
    L.grp_forward.argtypes = [vp, vp, vp, vp, i32, vp]
    L.grp_buffer.argtypes = [vp, C.c_char_p, C.POINTER(vp), C.POINTER(u64)]
    L.grp_shape.argtypes = [vp, C.POINTER(i32)]
    L.grp_launch_count.restype = u64
    L.grp_launch_count.argtypes = [vp]
    L.grp_stream.restype = vp
    L.grp_stream.argtypes = [vp]
    L.grl_last_error.restype = C.c_char_p
    L.grl_gae.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, C.c_float, C.c_float, vp]
    L.grl_adam_step.argtypes = [vp, vp, vp, vp, i64, i32, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, vp]
    L.grl_replay_create.restype = vp
    L.grl_replay_create.argtypes = [i32, i32, i32, i32, i32, i32, i32, C.c_uint32, i32]
    L.grl_replay_destroy.argtypes = [vp]
    L.grl_replay_begin.argtypes = [vp, vp, vp]
    L.grl_replay_add.argtypes = [vp] + [vp] * 6 + [vp]
    L.grl_replay_size.restype = i64
    L.grl_replay_size.argtypes = [vp]
    L.grl_replay_sample.argtypes = [vp, i32, C.c_float, u64] + [vp] * 10 + [vp]
    L.grl_replay_buffer.argtypes = [vp, C.c_char_p, C.POINTER(vp), C.POINTER(u64)]
    L.grl_replay_begin_indexed.argtypes = [vp, vp]
    L.grl_replay_add_indexed.argtypes = [vp, vp, i32] + [vp] * 6 + [vp]
    L.grl_replay_status.argtypes = [vp, C.POINTER(i64)]
    _lib = L
    return L


def last_error():
    return load().grs_last_error().decode("utf-8", "replace")
