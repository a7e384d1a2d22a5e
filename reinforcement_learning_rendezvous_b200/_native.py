"""ctypes binding of librdv_b200.so (the C ABI declared in include/rdv_b200.h).

The library is built in-tree (csrc/librdv_b200.so) by :func:`build` with
``nvcc -gencode arch=compute_100a,code=sm_100a``.  There is no CPU fallback:
:func:`lib` raises if the shared object is missing, and every entry point
returns RDV_ERR_CUDA on a machine without a usable GPU, which :func:`check`
turns into a RuntimeError.

Only raw device pointers (``tensor.data_ptr()``), sizes and the CUDA stream
handle cross this boundary; PyTorch owns every buffer.
"""
from __future__ import annotations

import ctypes as C
import importlib.util
import os
import shutil
import subprocess
import sysconfig

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC_DIR = os.path.join(PKG_DIR, "csrc")
INCLUDE_DIR = os.path.join(os.path.dirname(PKG_DIR), "include")
LIB_PATH = os.environ.get("RDV_B200_LIB") or os.path.join(CSRC_DIR, "librdv_b200.so")   # env: A/B experiments
HOST_SRC = os.path.join(CSRC_DIR, "rdv_host.c")                 # CPython helper of RendezvousVecEnv (gcc, no CUDA)
HOST_LIB = os.path.join(PKG_DIR, "_rdv_host" + (sysconfig.get_config_var("EXT_SUFFIX") or ".so"))
SOURCES = ("rdv_b200.cu",)
HEADERS = ("rdv_math.cuh", "rdv_plane_poly.h", "rdv_env.cuh", "rdv_step.cuh", "rdv_policy.cuh", "rdv_policy_tc.cuh",
           "rdv_lstm.cuh")

ABI_VERSION = 16
OBS_DIM, ACT_DIM, N_UNIFORMS = 17, 6, 24

# rows of RdvState.f64 / RdvState.i32, statistics slots, episode-record columns (rdv_b200.h)
(RCX, RCY, RCZ, VCX, VCY, VCZ, QCW, QCX, QCY, QCZ, WCX, WCY, WCZ, QTW, QTX, QTY, QTZ, WTX, WTY, WTZ,
 TDV, TDW, EPRET, NF64) = range(24)
I_STEP, I_SUCCESS, I_COLLIDED, I_EPISODE, NI32 = range(5)
STAT_NAMES = ("steps", "episodes", "return_sum", "length_sum", "succeeded", "collided", "delta_v_sum",
              "delta_w_sum", "end_obs", "end_time", "end_bubble", "end_attitude", "reward_sum",
              "rk_accepted", "rk_rejected", "failures")
NSTATS = len(STAT_NAMES)
EP_RETURN, EP_LENGTH, EP_SUCCESS, EP_COLLIDED, EP_DELTA_V, EP_DELTA_W, EP_NCOL = range(7)
INTEGRATOR_RK45, INTEGRATOR_CLOSED_FORM = 0, 1
END_REASONS = ("obs", "time", "bubble", "attitude")          # rendezvous_env.py:377


class RdvParams(C.Structure):
    _fields_ = [
        ("rc0", C.c_double * 3), ("vc0", C.c_double * 3), ("qc0", C.c_double * 4),
        ("wc0", C.c_double * 3), ("qt0", C.c_double * 4), ("wt0", C.c_double * 3),
        ("rc0_range", C.c_double), ("vc0_range", C.c_double), ("qc0_range", C.c_double),
        ("wc0_range", C.c_double), ("qt0_range", C.c_double), ("wt0_range", C.c_double),
        ("koz_radius", C.c_double), ("corridor_half_angle", C.c_double), ("h", C.c_double),
        ("dt", C.c_double), ("t_max", C.c_double),
        ("collision_coef", C.c_double), ("bonus_coef", C.c_double), ("fuel_coef", C.c_double),
        ("att_coef", C.c_double),
        ("inertia_c", C.c_double * 9), ("inertia_t", C.c_double * 9),
        ("torque_c", C.c_double * 3),
        ("integrator", C.c_int32), ("reserved0", C.c_int32),
        ("inv_inertia_c", C.c_double * 9), ("inv_inertia_t", C.c_double * 9),
        ("max_delta_v", C.c_double), ("max_delta_w", C.c_double), ("max_axial_distance", C.c_double),
        ("max_axial_speed", C.c_double), ("max_wc", C.c_double),
        ("max_attitude_error", C.c_double), ("max_rd_error", C.c_double), ("max_vd_error", C.c_double),
        ("max_qd_error", C.c_double), ("max_wd_error", C.c_double),
        ("rd", C.c_double * 3), ("capture_axis", C.c_double * 3), ("corridor_axis", C.c_double * 3),
        ("bubble0", C.c_double), ("bubble_rate", C.c_double), ("bubble_min", C.c_double), ("n", C.c_double),
        ("cw", C.c_double * 17),
        ("max_delta_v_f32", C.c_float), ("fuel_num_f32", C.c_float), ("fuel_den_f32", C.c_float),
        ("iso_c", C.c_int32), ("iso_t", C.c_int32), ("done_steps", C.c_int32),
        ("inv_max_attitude_error", C.c_double), ("inv_max_rd_error", C.c_double), ("inv_max_qd_error", C.c_double),
        ("koz_radius_sq", C.c_double), ("max_rd_error_sq", C.c_double), ("max_vd_error_sq", C.c_double),
        ("max_wd_error_sq", C.c_double),
        ("fuel_scale", C.c_double),
        ("att_scale", C.c_double), ("bonus_scale", C.c_double), ("collision_scale", C.c_double),
        ("obs_inv_r", C.c_double), ("obs_inv_v", C.c_double), ("obs_inv_w", C.c_double),
        ("near_sq", C.c_double),
        ("box_hi_r", C.c_int32), ("box_hi_v", C.c_int32), ("box_hi_w", C.c_int32), ("reserved1", C.c_int32),
    ]


class RdvState(C.Structure):
    _fields_ = [("f64", C.c_void_p), ("i32", C.c_void_p), ("ld", C.c_int64), ("param_table", C.c_void_p),
                ("param_block", C.c_void_p)]


class RdvStepIO(C.Structure):
    _fields_ = [
        ("actions", C.c_void_p), ("act_f64", C.c_int32), ("auto_reset", C.c_int32),
        ("obs", C.c_void_p), ("reward", C.c_void_p), ("done", C.c_void_p),
        ("terminal_obs", C.c_void_p), ("end_reason", C.c_void_p), ("episode_record", C.c_void_p),
        ("stats", C.c_void_p),
        ("reward_f32", C.c_void_p), ("fin_count", C.c_void_p), ("fin_rows", C.c_void_p),
        ("fin_capacity", C.c_int32), ("fin_append", C.c_int32), ("fin_env_base", C.c_int32), ("reserved", C.c_int32),
    ]


class RdvFinishedRow(C.Structure):
    _fields_ = [("env", C.c_int32), ("end_reason", C.c_int32), ("terminal_obs", C.c_float * 17), ("pad", C.c_float),
                ("record", C.c_double * 6)]


class RdvPolicy(C.Structure):
    _fields_ = [
        ("w0", C.c_void_p), ("b0", C.c_void_p), ("w1", C.c_void_p), ("b1", C.c_void_p),
        ("w2", C.c_void_p), ("b2", C.c_void_p), ("hidden", C.c_int32), ("reserved", C.c_int32),
        ("log_std", C.c_void_p),
    ]


class RdvLstmPolicy(C.Structure):
    _fields_ = [
        ("weight_ih", C.c_void_p), ("weight_hh", C.c_void_p), ("bias_ih", C.c_void_p), ("bias_hh", C.c_void_p),
        ("w0", C.c_void_p), ("b0", C.c_void_p), ("w1", C.c_void_p), ("b1", C.c_void_p),
        ("w2", C.c_void_p), ("b2", C.c_void_p), ("hidden", C.c_int32), ("reserved", C.c_int32),
    ]


LSTM_HIDDEN = 256               # the only LSTM width rdv_lstm_policy_step supports


class RdvRolloutIO(C.Structure):
    _fields_ = [
        ("steps", C.c_int32), ("action_source", C.c_int32), ("auto_reset", C.c_int32), ("reserved", C.c_int32),
        ("actions", C.c_void_p), ("action_seed", C.c_uint64), ("step_base", C.c_int64),
        ("actions_out", C.c_void_p), ("obs", C.c_void_p), ("rewards", C.c_void_p), ("dones", C.c_void_p),
        ("obs_steps", C.c_void_p), ("stats", C.c_void_p), ("policy", RdvPolicy),
        ("reset_rows", C.c_void_p), ("sm_reserve", C.c_int32), ("reserved2", C.c_int32), ("mc_out", C.c_void_p),
        ("policy_table", C.c_void_p), ("policy_tile", C.c_void_p), ("policy_count", C.c_int32),
        ("reserved3", C.c_int32),
    ]


RESET_ROWS = 23
POLICY_TILE = 128               # envs per entry of RdvRolloutIO.policy_tile
(MC_EP_LEN, MC_NUM_COLLISIONS, MC_COLLIDED, MC_TOTAL_REWARD, MC_TOTAL_DELTA_V, MC_NUM_SUCCESSES, MC_SUCCEEDED,
 MC_MIN_KOZ, MC_POS_ERR, MC_VEL_ERR, MC_ATT_ERR, MC_ROT_ERR, MC_LEVEL, MC_TAIL_COUNT, MC_END_REASON,
 MC_TOTAL_DELTA_W, MC_NCOL) = range(17)
# columns of the trajectory record of rdv_rollout_trajectory: 0 .. NF64 - 1 are the RdvState.f64 rows (RCX .. EPRET)
(TR_I_STEP, TR_I_SUCCESS, TR_I_COLLIDED, TR_I_EPISODE, TR_POS_ERR, TR_VEL_ERR, TR_ATT_ERR, TR_ROT_ERR, TR_KOZ,
 TR_COLLISION, TR_SUCCESS, TR_NCOL) = range(NF64, NF64 + 12)
TUNE_ROLLOUT_TPB, TUNE_RESET_REFILL, TUNE_ROLLOUT_PDL, TUNE_ROLLOUT_HELPERS = 0, 1, 2, 3


ACTIONS_F32, ACTIONS_F64, ACTIONS_PHILOX, ACTIONS_POLICY, ACTIONS_POLICY_SAMPLE = 0, 1, 2, 3, 4


# name -> (restype, argtypes); every symbol include/rdv_b200.h declares
PROTOTYPES = {
    "rdv_abi_version": (C.c_int, []),
    "rdv_sizeof_params": (C.c_int, []),
    "rdv_sizeof": (C.c_int, [C.c_int]),
    "rdv_strerror": (C.c_char_p, [C.c_int]),
    "rdv_tune": (C.c_int, [C.c_int, C.c_int]),
    "rdv_params_default": (None, [C.POINTER(RdvParams)]),
    "rdv_params_derive": (C.c_int, [C.POINTER(RdvParams)]),
    "rdv_step": (C.c_int, [C.POINTER(RdvParams), C.POINTER(RdvState), C.POINTER(RdvStepIO), C.c_int64,
                           C.c_uint64, C.c_int64, C.c_void_p]),
    "rdv_rollout": (C.c_int, [C.POINTER(RdvParams), C.POINTER(RdvState), C.POINTER(RdvRolloutIO), C.c_int64,
                              C.c_uint64, C.c_int64, C.c_void_p]),
    "rdv_rollout_trajectory": (C.c_int, [C.POINTER(RdvParams), C.POINTER(RdvState), C.POINTER(RdvRolloutIO),
                                         C.c_void_p, C.c_int64, C.c_uint64, C.c_int64, C.c_void_p]),
    "rdv_reset": (C.c_int, [C.POINTER(RdvParams), C.POINTER(RdvState), C.c_void_p, C.c_void_p, C.c_void_p,
                            C.c_int64, C.c_uint64, C.c_int64, C.c_int, C.c_void_p]),
    "rdv_observe": (C.c_int, [C.POINTER(RdvParams), C.POINTER(RdvState), C.c_void_p, C.c_int64, C.c_void_p]),
    "rdv_errors": (C.c_int, [C.POINTER(RdvParams), C.POINTER(RdvState), C.c_void_p, C.c_void_p, C.c_void_p,
                             C.c_void_p, C.c_int64, C.c_void_p]),
    "rdv_refresh_flags": (C.c_int, [C.POINTER(RdvParams), C.POINTER(RdvState), C.c_int64, C.c_void_p]),
    "rdv_frame_transform": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "rdv_policy_forward": (C.c_int, [C.POINTER(RdvPolicy), C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "rdv_policy_forward_ffma": (C.c_int, [C.POINTER(RdvPolicy), C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "rdv_lstm_policy_step": (C.c_int, [C.POINTER(RdvLstmPolicy), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]),
    "rdv_math_probe": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "rdv_fp64_peak_probe": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
}

_lib = None


def nvcc_command(out=LIB_PATH):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    return [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
            "-I", INCLUDE_DIR, "-shared", "-Xcompiler", "-fPIC", "-o", out] + \
           [os.path.join(CSRC_DIR, s) for s in SOURCES]


def is_stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC_DIR, f) for f in SOURCES + HEADERS] + [os.path.join(INCLUDE_DIR, "rdv_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build_host(force=False):
    """gcc -> _rdv_host*.so next to the package (the VecEnv's info-dict builder, csrc/rdv_host.c)."""
    global _host
    if force or not os.path.exists(HOST_LIB) or os.path.getmtime(HOST_LIB) < os.path.getmtime(HOST_SRC):
        cc = shutil.which("gcc") or shutil.which("cc") or "gcc"
        import numpy                                            # row views are made through the numpy C API
        subprocess.run([cc, "-O2", "-fPIC", "-shared", "-Wall", "-I", sysconfig.get_paths()["include"],
                        "-I", numpy.get_include(), "-o", HOST_LIB, HOST_SRC], check=True)
        _host = None
    return HOST_LIB


_host = None


def host():
    """The loaded _rdv_host extension module.  Raises when it has not been built."""
    global _host
    if _host is None:
        if not os.path.exists(HOST_LIB):
            raise RuntimeError(f"{HOST_LIB} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`")
        spec = importlib.util.spec_from_file_location("_rdv_host", HOST_LIB)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        _host = mod
    return _host


def build(force=False, verbose=False):
    """Compile csrc/*.cu for sm_100a into csrc/librdv_b200.so (in-tree, so it travels to the GPU box)."""
    global _lib
    build_host(force=force)
    if force or is_stale():
        cmd = nvcc_command()
        if verbose:
            cmd = cmd[:1] + ["-Xptxas", "-v"] + cmd[1:]
            print(" ".join(cmd))
        subprocess.run(cmd, check=True)
        _lib = None
    return LIB_PATH


def lib():
    """The loaded library.  Raises (no fallback) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  This package has no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        if L.rdv_abi_version() != ABI_VERSION:
            raise RuntimeError(f"librdv_b200.so ABI {L.rdv_abi_version()} != binding ABI {ABI_VERSION}; rebuild")
        for which, mirror in enumerate((RdvParams, RdvState, RdvStepIO, RdvRolloutIO, RdvPolicy, RdvFinishedRow,
                                         RdvLstmPolicy)):
            if L.rdv_sizeof(which) != C.sizeof(mirror):
                raise RuntimeError(f"{mirror.__name__} layout mismatch between include/rdv_b200.h "
                                   f"({L.rdv_sizeof(which)} B) and _native.py ({C.sizeof(mirror)} B)")
        _lib = L
    return _lib


def strerror(status: int) -> str:
    return lib().rdv_strerror(int(status)).decode()


def check(status: int, what: str):
    if status != 0:
        raise RuntimeError(f"{what} failed: {strerror(status)} (status {status})")
