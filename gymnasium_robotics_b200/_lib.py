"""ctypes binding of the C-ABI in include/b200sim.h (the in-tree CUDA library libb200sim.so).

There is deliberately no CPU fallback: if the library or a CUDA device is missing, importing callers get a loud
error.  (The CPU restatement under oracle/ is test infrastructure and is never imported from here.)
"""
from __future__ import annotations

import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200SIM_LIB") or os.path.join(_HERE, "libb200sim.so")
_LIB = None

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "-shared", "-DB200_BLOCK_ALIGN", "-DB200_CHOL_SMEM",
              "-prec-div=false", "-prec-sqrt=false"] + \
    os.environ.get("B200SIM_NVCC_EXTRA", "").split()


class FetchTaskC(ctypes.Structure):
    """b200sim_fetch_task_t"""
    _fields_ = [(n, ctypes.c_int) for n in ("has_object", "block_gripper", "n_substeps", "reward_dense", "grip_site",
                                             "obj_site", "frame_site", "nrobot")] + \
               [("robot_qadr", ctypes.c_int * 16), ("robot_dadr", ctypes.c_int * 16), ("finger_qadr", ctypes.c_int * 2),
                ("nobs", ctypes.c_int), ("distance_threshold", ctypes.c_float), ("dt", ctypes.c_float),
                ("kind", ctypes.c_int), ("nact", ctypes.c_int), ("ngoal", ctypes.c_int), ("success_radius", ctypes.c_float),
                ("obs_qpos_start", ctypes.c_int), ("vel_clip", ctypes.c_float),
                ("obj_qadr", ctypes.c_int), ("obj_dadr", ctypes.c_int), ("goal_flags", ctypes.c_int),
                ("rotation_threshold", ctypes.c_float), ("touch_mode", ctypes.c_int), ("tip_site", ctypes.c_int * 5),
                ("penv_body", ctypes.c_int)]


class FetchResetC(ctypes.Structure):
    """b200sim_fetch_reset_t"""
    _fields_ = [("has_object", ctypes.c_int), ("target_in_the_air", ctypes.c_int), ("obj_qadr", ctypes.c_int),
                ("obj_range", ctypes.c_float), ("target_range", ctypes.c_float), ("target_offset", ctypes.c_float * 3),
                ("height_offset", ctypes.c_float), ("gripper_xpos", ctypes.c_float * 3)]


class UniformResetC(ctypes.Structure):
    """b200sim_uniform_reset_t"""
    _fields_ = [("n", ctypes.c_int), ("slot", ctypes.c_int * 16), ("lo", ctypes.c_float * 16), ("hi", ctypes.c_float * 16),
                ("quat_slot", ctypes.c_int)]


class MazeResetC(ctypes.Structure):
    """b200sim_maze_reset_t"""
    _fields_ = [("n_goal", ctypes.c_int), ("n_reset", ctypes.c_int), ("scaling", ctypes.c_float), ("noise", ctypes.c_float)]


class HandResetC(ctypes.Structure):
    """b200sim_hand_reset_t"""
    _fields_ = [(n, ctypes.c_int) for n in ("obj_qadr", "rot_mode", "randomize_rotation", "randomize_position", "goal_rot_mode",
                                             "goal_random_position")] + [("pos_lo", ctypes.c_float * 3), ("pos_hi", ctypes.c_float * 3)]


class ReachResetC(ctypes.Structure):
    """b200sim_reach_reset_t"""
    _fields_ = [("meeting", ctypes.c_float * 3), ("initial_goal", ctypes.c_float * 15)]


class KeepC(ctypes.Structure):
    """b200sim_keep_t"""
    _fields_ = [("n", ctypes.c_int), ("start", ctypes.c_int * 4), ("len", ctypes.c_int * 4)]


def build_library(force: bool = False, verbose: bool = False) -> str:
    """nvcc-compile csrc/b200sim.cu and csrc/b200sim_wide.cu for sm_100a into the in-tree libb200sim.so (cross-compiles
    without a GPU; the two translation units are compiled in parallel)."""
    names = ("b200sim", "b200sim_wide", "b200sim_kitchen", "b200sim_kitchen_groups", "b200sim_kitchen_hull")
    srcs = [os.path.join(_HERE, "csrc", n + ".cu") for n in names]
    deps = srcs + [os.path.join(_HERE, "csrc", f) for f in ("sim_core.cuh", "fetch_task.cuh", "step_kernel.cuh", "dmodel.h", "reset_sample.cuh")] + \
           [os.path.join(_HERE, "..", "include", f) for f in ("b200sim.h", "b200sim_model.h")]
    if not force and os.path.exists(LIB_PATH) and os.path.getmtime(LIB_PATH) >= max(os.path.getmtime(d) for d in deps):
        return LIB_PATH
    flags = [f for f in NVCC_FLAGS if f != "-shared"]
    objs = [os.path.join(_HERE, "csrc", n + ".o") for n in names]
    procs = [subprocess.Popen(["nvcc"] + flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", o, src]) for src, o in zip(srcs, objs)]
    rcs = [p.wait() for p in procs]
    if any(rcs):
        raise subprocess.CalledProcessError(max(rcs), "nvcc -c (b200sim)")
    subprocess.check_call(["nvcc", "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB_PATH] + objs)
    for o in objs:
        os.remove(o)
    return LIB_PATH


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(the CUDA path has no CPU fallback)")
    L = ctypes.CDLL(LIB_PATH)
    vp, ci = ctypes.c_void_p, ctypes.c_int
    L.b200sim_create.argtypes = [ctypes.c_char_p, ctypes.c_size_t, vp, vp, ctypes.POINTER(FetchTaskC), ci, ci, ctypes.POINTER(vp)]
    L.b200sim_create.restype = ci
    L.b200sim_destroy.argtypes = [vp]
    L.b200sim_destroy.restype = None
    L.b200sim_last_error.argtypes = [vp]
    L.b200sim_last_error.restype = ctypes.c_char_p
    L.b200sim_num_envs.argtypes = [vp]
    L.b200sim_layout.argtypes = [vp, ctypes.POINTER(ci)]
    L.b200sim_state.argtypes = [vp]
    L.b200sim_state.restype = vp
    L.b200sim_step.argtypes = [vp] * 11
    L.b200sim_set_time_limit.argtypes = [vp, ci, ci]
    L.b200sim_elapsed.argtypes = [vp]
    L.b200sim_elapsed.restype = vp
    L.b200sim_overflow_counter.argtypes = [vp]
    L.b200sim_overflow_counter.restype = vp
    L.b200sim_packed_width.argtypes = [vp]
    L.b200sim_set_packed.argtypes = [vp, ci]
    L.b200sim_refresh.argtypes = [vp] * 8
    L.b200sim_raw_step.argtypes = [vp, ci] + [vp] * 6
    L.b200sim_raw_step_masked.argtypes = [vp, vp, ci] + [vp] * 6
    L.b200sim_compute_reward.argtypes = [vp, vp, vp, ci, vp, vp]
    L.b200sim_reset.argtypes = [vp, vp, vp, ctypes.POINTER(FetchResetC), ctypes.c_ulonglong, ci, vp] + [vp] * 6
    L.b200sim_reset_maze.argtypes = [vp, vp, vp, ctypes.POINTER(MazeResetC), vp, vp, ctypes.c_ulonglong, ci, vp] + [vp] * 6
    L.b200sim_reset_hand_pose.argtypes = [vp, vp, vp, ctypes.POINTER(HandResetC), vp, ctypes.c_ulonglong, ci, vp, ci, vp]
    L.b200sim_reset_hand_goal.argtypes = [vp, vp, ctypes.POINTER(HandResetC), vp, ctypes.c_ulonglong, ci, vp] + [vp] * 6
    L.b200sim_reset_reach.argtypes = [vp, vp, vp, ctypes.POINTER(ReachResetC), ctypes.c_ulonglong, ci, vp] + [vp] * 6
    L.b200sim_check_state.argtypes = [vp, vp, vp, ctypes.POINTER(KeepC), vp]
    L.b200sim_reset_uniform.argtypes = [vp, vp, vp, ctypes.POINTER(UniformResetC), ctypes.c_ulonglong, ci, vp] + [vp] * 6
    L.b200sim_launch_count.argtypes = [vp]
    L.b200sim_launch_count.restype = ctypes.c_long
    L.b200sim_launch_config.argtypes = [vp, ctypes.POINTER(ci), ctypes.POINTER(ci), ctypes.POINTER(ci)]
    L.b200sim_kernel_variant.argtypes = [vp, ctypes.POINTER(ci), ctypes.POINTER(ci), ctypes.POINTER(ci)]
    _LIB = L
    return L


EXPORTED_SYMBOLS = ["b200sim_create", "b200sim_destroy", "b200sim_last_error", "b200sim_num_envs", "b200sim_layout",
                    "b200sim_state", "b200sim_step", "b200sim_refresh", "b200sim_raw_step", "b200sim_raw_step_masked", "b200sim_compute_reward", "b200sim_reset", "b200sim_reset_uniform", "b200sim_reset_maze", "b200sim_check_state", "b200sim_reset_reach", "b200sim_reset_hand_pose", "b200sim_reset_hand_goal",
                    "b200sim_launch_count", "b200sim_launch_config", "b200sim_kernel_variant", "b200sim_set_time_limit", "b200sim_elapsed", "b200sim_overflow_counter",
                    "b200sim_packed_width", "b200sim_set_packed"]
