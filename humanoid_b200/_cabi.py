"""ctypes binding of libphc_b200.so (include/phc_b200.h).

The library is plain C ABI — device pointers, sizes, a cudaStream_t — so the binding is
``tensor.data_ptr()`` plus the current torch stream.  There is no fallback: if the shared
object is missing or a call fails, the error is raised.
"""

from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libphc_b200.so")

ABI_VERSION = 6
NUM_BODIES = 24
SELF_OBS_DIM = 358
TASK_OBS_DIM = 576
MAX_TIME_STEPS = 16

STEP_MAPPED_HOST_IO = 1
STEP_OBS_NORM_BF16 = 2

OPT_FORCE_GENERIC_STEP = 1
OPT_STEP_EPB = 2
OPT_STEP_PDL = 3
OPT_TEST_SPEC_FAULT = 4
OPT_MULTI_GROUPS = 5
OPT_MOMENTS_BULK = 6
OPT_STEP_PERSIST = 7

STATE_INIT_START = 0
STATE_INIT_RANDOM = 1
STATE_INIT_DEFAULT = 2
STATE_INIT_HYBRID = 3

OBS_LOCAL_ROOT = 1
OBS_ROOT_HEIGHT = 2
OBS_UPRIGHT = 4
STEP_OBS_FLAGS_SET = 0x80000000


class PhcLibDesc(C.Structure):
    _fields_ = [
        ("gts", C.c_void_p), ("grs", C.c_void_p), ("lrs", C.c_void_p), ("gvs", C.c_void_p),
        ("gavs", C.c_void_p), ("dvs", C.c_void_p), ("motion_aa", C.c_void_p),
        ("motion_lengths", C.c_void_p), ("motion_num_frames", C.c_void_p), ("motion_dt", C.c_void_p),
        ("length_starts", C.c_void_p), ("motion_bodies", C.c_void_p), ("motion_limb_weights", C.c_void_p),
        ("total_frames", C.c_int64), ("num_motions", C.c_int64),
    ]  # fmt: skip


class PhcView(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("stride_env", C.c_int64), ("stride_body", C.c_int64)]


class PhcBodyState(C.Structure):
    _fields_ = [("pos", PhcView), ("rot", PhcView), ("vel", PhcView), ("ang_vel", PhcView), ("num_bodies", C.c_int32)]


class PhcMotionOut(C.Structure):
    _fields_ = [
        (k, C.c_void_p)
        for k in (
            "root_pos", "root_rot", "dof_pos", "root_vel", "root_ang_vel", "dof_vel", "motion_aa", "rg_pos",
            "rb_rot", "body_vel", "body_ang_vel", "motion_bodies", "motion_limb_weights", "frame_idx0",
            "frame_idx1", "blend",
        )
    ]  # fmt: skip


class PhcAmpArgs(C.Structure):
    _fields_ = [
        ("root_pos", C.c_void_p), ("root_pos_stride", C.c_int64),
        ("root_rot", C.c_void_p), ("root_rot_stride", C.c_int64),
        ("root_vel", C.c_void_p), ("root_vel_stride", C.c_int64),
        ("root_ang_vel", C.c_void_p), ("root_ang_vel_stride", C.c_int64),
        ("dof_pos", C.c_void_p), ("dof_pos_stride", C.c_int64), ("dof_pos_elem_stride", C.c_int64),
        ("dof_vel", C.c_void_p), ("dof_vel_stride", C.c_int64), ("dof_vel_elem_stride", C.c_int64),
        ("key_body_pos", PhcView),
        ("num_key_bodies", C.c_int32),
        ("dof_subset", C.c_void_p),
        ("num_sel", C.c_int32),
        ("flags", C.c_uint32),
    ]  # fmt: skip


class PhcRewardSpec(C.Structure):
    _fields_ = [(k, C.c_float) for k in ("k_pos", "k_rot", "k_vel", "k_ang_vel", "w_pos", "w_rot", "w_vel", "w_ang_vel")]


class PhcResetArgs(C.Structure):
    _fields_ = [
        ("body", PhcBodyState),
        ("humanoid_root_states", C.c_void_p),
        ("root_stride", C.c_int64),
        ("dof_pos", C.c_void_p),
        ("dof_vel", C.c_void_p),
        ("dof_stride", C.c_int64),
        ("dof_elem_stride", C.c_int64),
        ("progress_buf", C.c_void_p),
        ("reset_buf", C.c_void_p),
        ("terminate_buf", C.c_void_p),
        ("motion_start_times", C.c_void_p),
        ("motion_start_times_offset", C.c_void_p),
        ("global_offset", C.c_void_p),
        ("sampled_motion_ids", C.c_void_p),
        ("env_mask", C.c_void_p),
        ("phase", C.c_void_p),
        ("state_init", C.c_int32),
        ("flag_test", C.c_int32),
        ("time_steps", C.c_int32),
        ("dt", C.c_float),
        ("obs_buf", C.c_void_p),
        ("obs_stride", C.c_int64),
        ("obs_norm", C.c_void_p),
        ("obs_norm_stride", C.c_int64),
        ("norm_mean", C.c_void_p),
        ("norm_var", C.c_void_p),
        ("norm_epsilon", C.c_float),
        ("norm_clip", C.c_float),
        ("obs_norm_bf16", C.c_int32),
        ("obs_moments_mode", C.c_int32),
        ("obs_moments", C.c_void_p),
        ("obs_moments_buckets", C.c_int32),
        ("obs_flags", C.c_uint32),
        ("ref_dof_pos", C.c_void_p),
        ("ref_dof_pos_stride", C.c_int64),
        ("initial_root_states", C.c_void_p),
        ("initial_root_stride", C.c_int64),
        ("initial_dof_pos", C.c_void_p),
        ("initial_dof_vel", C.c_void_p),
        ("initial_dof_stride", C.c_int64),
        ("default_mask", C.c_void_p),
    ]


class PhcStepArgs(C.Structure):
    _fields_ = [
        ("body", PhcBodyState),
        ("progress_buf", C.c_void_p),
        ("motion_start_times", C.c_void_p),
        ("motion_start_times_offset", C.c_void_p),
        ("global_offset", C.c_void_p),
        ("sampled_motion_ids", C.c_void_p),
        ("termination_distances", C.c_void_p),
        ("reset_body_mask", C.c_uint32),
        ("use_mean", C.c_int32),
        ("enable_early_termination", C.c_int32),
        ("advance_progress", C.c_int32),
        ("time_steps", C.c_int32),
        ("dt", C.c_float),
        ("rwd", PhcRewardSpec),
        ("obs_buf", C.c_void_p),
        ("obs_stride", C.c_int64),
        ("rew_buf", C.c_void_p),
        ("reward_raw", C.c_void_p),
        ("reward_raw_stride", C.c_int64),
        ("reset_buf", C.c_void_p),
        ("terminate_buf", C.c_void_p),
        ("flags", C.c_uint32),
        ("dof_force", C.c_void_p),
        ("dof_force_stride", C.c_int64),
        ("dof_vel", C.c_void_p),
        ("dof_vel_stride", C.c_int64),
        ("dof_vel_elem_stride", C.c_int64),
        ("rew_power_coef", C.c_float),
        ("power_col", C.c_int32),
        ("obs_moments", C.c_void_p),
        ("obs_norm", C.c_void_p),
        ("obs_norm_stride", C.c_int64),
        ("norm_mean", C.c_void_p),
        ("norm_var", C.c_void_p),
        ("norm_epsilon", C.c_float),
        ("norm_clip", C.c_float),
        ("mpjpe", C.c_void_p),
        ("obs_moments_buckets", C.c_int32),
        ("ep_terminals", C.c_void_p),
        ("ep_truncations", C.c_void_p),
        ("ep_masks", C.c_void_p),
        ("ep_returns", C.c_void_p),
        ("ep_lengths", C.c_void_p),
        ("ep_sums", C.c_void_p),
        ("ep_buckets", C.c_int32),
        ("ep_raw_cols", C.c_int32),
        ("rew_out", C.c_void_p),
        ("reset_out", C.c_void_p),
        ("terminate_out", C.c_void_p),
        ("auto_reset", C.POINTER(PhcResetArgs)),
        ("ref_dof_pos", C.c_void_p),
        ("ref_dof_pos_stride", C.c_int64),
        ("obs_flags", C.c_uint32),
    ]


class PhcEpisodeArgs(C.Structure):
    _fields_ = [
        ("reset", C.c_void_p),
        ("terminate", C.c_void_p),
        ("rewards", C.c_void_p),
        ("reward_raw", C.c_void_p),
        ("reward_raw_stride", C.c_int64),
        ("reward_raw_cols", C.c_int32),
        ("_pad0", C.c_int32),
        ("terminals", C.c_void_p),
        ("truncations", C.c_void_p),
        ("masks", C.c_void_p),
        ("episode_returns", C.c_void_p),
        ("episode_lengths", C.c_void_p),
        ("stats", C.c_void_p),
        ("raw_rewards", C.c_void_p),
        ("workspace", C.c_void_p),
    ]


class PhcAmpEnvArgs(C.Structure):
    _fields_ = [
        ("body", PhcBodyState),
        ("dof_pos", C.c_void_p),
        ("dof_vel", C.c_void_p),
        ("dof_stride", C.c_int64),
        ("dof_elem_stride", C.c_int64),
        ("key_body_ids", C.c_int32 * 8),
        ("num_key_bodies", C.c_int32),
        ("num_sel", C.c_int32),
        ("dof_subset", C.c_void_p),
        ("flags", C.c_uint32),
        ("num_steps", C.c_int32),
        ("obs_per_step", C.c_int32),
        ("init_slot0", C.c_int32),
        ("amp_obs_buf", C.c_void_p),
        ("amp_obs_demo_buf", C.c_void_p),
        ("env_mask", C.c_void_p),
    ]


class PhcHostStepArgs(C.Structure):
    _fields_ = [
        (k, C.c_void_p)
        for k in (
            "state", "progress_buf", "motion_start_times", "motion_start_times_offset", "global_offset",
            "sampled_motion_ids", "obs_buf", "rew_buf", "reward_raw", "reset_buf", "terminate_buf",
        )
    ]  # fmt: skip


class PhcHostResetArgs(C.Structure):
    _fields_ = [
        ("phase", C.c_void_p),
        ("env_mask", C.c_void_p),
        ("state_init", C.c_int32),
        ("flag_test", C.c_int32),
        ("state_out", C.c_void_p),
        ("root_states", C.c_void_p),
        ("dof_pos", C.c_void_p),
        ("dof_vel", C.c_void_p),
        ("motion_start_times_out", C.c_void_p),
        ("motion_start_times_offset_out", C.c_void_p),
        ("global_offset_out", C.c_void_p),
    ]


class PhcHostDeviceOut(C.Structure):
    _fields_ = [
        ("obs", C.c_void_p),
        ("obs_norm", C.c_void_p),
        ("norm_mean", C.c_void_p),
        ("norm_var", C.c_void_p),
        ("norm_epsilon", C.c_float),
        ("norm_clip", C.c_float),
        ("flags", C.c_uint32),
        ("obs_moments", C.c_void_p),
        ("obs_moments_buckets", C.c_int32),
        ("stream", C.c_void_p),
    ]


class PhcHostEnvArgs(C.Structure):
    _fields_ = [
        ("dof_force", C.c_void_p),
        ("dof_vel", C.c_void_p),
        ("rew_power_coef", C.c_float),
        ("mpjpe", C.c_void_p),
        ("default_mask", C.c_void_p),
    ]


BUILD_FILTER_RADIUS = 8
EPISODE_SUM_COLS = 12
PEER_MAX_WORLD = 16
PEER_HANDLE_BYTES = 64
PEER_TIMEOUT = -7
PHC_ERR_BUSY = -8
HOST_SLOTS = 2


class PhcBuildArgs(C.Structure):
    _fields_ = [
        ("pose_quat_global", C.c_void_p), ("root_trans", C.c_void_p), ("pose_aa", C.c_void_p),
        ("local_translation", C.c_void_p), ("num_frames", C.c_void_p), ("length_starts", C.c_void_p),
        ("fps", C.c_void_p), ("heading_zw", C.c_void_p),
        ("parent_indices_host", C.POINTER(C.c_int32)), ("filter_weights_host", C.POINTER(C.c_double)),
        ("total_frames", C.c_int64), ("num_motions", C.c_int64),
        ("gts", C.c_void_p), ("grs", C.c_void_p), ("lrs", C.c_void_p), ("gvs", C.c_void_p), ("gavs", C.c_void_p),
        ("dvs", C.c_void_p), ("motion_aa", C.c_void_p), ("scratch", C.c_void_p),
    ]  # fmt: skip


# name -> (restype, argtypes); every symbol include/phc_b200.h declares
SIGNATURES = {
    "phc_strerror": (C.c_char_p, [C.c_int]),
    "phc_abi_version": (C.c_int, []),
    "phc_last_cuda_error": (C.c_int, []),
    "phc_lib_create": (C.c_int, [C.POINTER(PhcLibDesc), C.POINTER(C.c_void_p)]),
    "phc_lib_destroy": (None, [C.c_void_p]),
    "phc_lib_pack": (C.c_int, [C.c_void_p, C.c_void_p]),
    "phc_calc_frame_blend": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p],
    ),
    "phc_motion_state": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(PhcMotionOut), C.c_void_p],
    ),
    "phc_self_obs_smpl_max": (
        C.c_int,
        [C.POINTER(PhcBodyState), C.c_int64, C.c_uint32, C.c_void_p, C.c_int64, C.c_void_p],
    ),
    "phc_imitation_obs": (
        C.c_int,
        [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.POINTER(PhcBodyState), C.POINTER(PhcBodyState), C.c_int64,
         C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p],
    ),  # fmt: skip
    "phc_amp_obs": (C.c_int, [C.POINTER(PhcAmpArgs), C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]),
    "phc_imitation_reward": (
        C.c_int,
        [C.POINTER(PhcBodyState), C.POINTER(PhcBodyState), C.c_int64, C.POINTER(PhcRewardSpec), C.c_void_p,
         C.c_void_p, C.c_int64, C.c_void_p],
    ),  # fmt: skip
    "phc_im_reset": (
        C.c_int,
        [C.POINTER(PhcView), C.POINTER(PhcView), C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
         C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p],
    ),  # fmt: skip
    "phc_action_to_pd_targets": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_uint32,
         C.c_int64, C.c_int32, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p],
    ),  # fmt: skip
    "phc_step_fused": (C.c_int, [C.c_void_p, C.POINTER(PhcStepArgs), C.c_int64, C.c_void_p]),
    "phc_reset_envs": (C.c_int, [C.c_void_p, C.POINTER(PhcResetArgs), C.c_int64, C.c_void_p]),
    "phc_set_option": (C.c_int, [C.c_int, C.c_int]),
    "phc_set_trace_buffer": (C.c_int, [C.c_void_p, C.c_int64]),
    "phc_host_step_create": (
        C.c_int,
        [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_uint32, C.c_int32, C.c_int32, C.c_float,
         C.POINTER(PhcRewardSpec), C.POINTER(C.c_void_p)],
    ),  # fmt: skip
    "phc_host_step": (C.c_int, [C.c_void_p, C.POINTER(PhcHostStepArgs), C.c_int64]),
    "phc_host_step_destroy": (None, [C.c_void_p]),
    "phc_host_step_submit": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(PhcHostStepArgs), C.c_int64]),
    "phc_host_step_wait": (C.c_int, [C.c_void_p, C.c_int32]),
    "phc_host_step_submit_reset": (
        C.c_int,
        [C.c_void_p, C.c_int32, C.POINTER(PhcHostStepArgs), C.POINTER(PhcHostResetArgs), C.c_int64],
    ),
    "phc_host_reset_submit": (
        C.c_int,
        [C.c_void_p, C.c_int32, C.POINTER(PhcHostStepArgs), C.POINTER(PhcHostResetArgs), C.c_int64],
    ),
    "phc_host_step_submit_device": (
        C.c_int,
        [C.c_void_p, C.c_int32, C.POINTER(PhcHostStepArgs), C.POINTER(PhcHostResetArgs), C.POINTER(PhcHostDeviceOut),
         C.c_int64],
    ),  # fmt: skip
    "phc_host_reset_submit_device": (
        C.c_int,
        [C.c_void_p, C.c_int32, C.POINTER(PhcHostStepArgs), C.POINTER(PhcHostResetArgs), C.POINTER(PhcHostDeviceOut),
         C.c_int64],
    ),  # fmt: skip
    "phc_host_step_submit_env": (
        C.c_int,
        [C.c_void_p, C.c_int32, C.POINTER(PhcHostStepArgs), C.POINTER(PhcHostResetArgs), C.POINTER(PhcHostDeviceOut),
         C.POINTER(PhcHostEnvArgs), C.c_int64],
    ),  # fmt: skip
    "phc_host_reset_submit_env": (
        C.c_int,
        [C.c_void_p, C.c_int32, C.POINTER(PhcHostStepArgs), C.POINTER(PhcHostResetArgs), C.POINTER(PhcHostDeviceOut),
         C.POINTER(PhcHostEnvArgs), C.c_int64],
    ),  # fmt: skip
    "phc_host_step_set_initial_state": (
        C.c_int,
        [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64],
    ),
    "phc_host_step_path": (C.c_int, [C.c_void_p]),
    "phc_host_step_chunks": (C.c_int, [C.c_void_p]),
    "phc_host_step_tuning_calls": (C.c_int, [C.c_void_p]),
    "phc_host_step_h2d_bytes": (C.c_int64, [C.c_void_p, C.c_int64]),
    "phc_host_step_d2h_bytes": (C.c_int64, [C.c_void_p, C.c_int64]),
    "phc_obs_moments": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]),
    "phc_running_norm_update": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p],
    ),
    "phc_running_norm_forward": (
        C.c_int,
        [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_void_p,
         C.c_int64, C.c_void_p],
    ),  # fmt: skip
    "phc_episode_update": (C.c_int, [C.POINTER(PhcEpisodeArgs), C.c_int64, C.c_void_p]),
    "phc_amp_step": (C.c_int, [C.POINTER(PhcAmpEnvArgs), C.c_int64, C.c_int32, C.c_void_p]),
    "phc_amp_init_ref": (
        C.c_int,
        [C.c_void_p, C.POINTER(PhcAmpEnvArgs), C.c_void_p, C.c_void_p, C.c_float, C.c_int64, C.c_void_p],
    ),
    "phc_motion_build": (C.c_int, [C.POINTER(PhcBuildArgs), C.c_void_p]),
    "phc_episode_fold": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "phc_obs_moments_fold": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p]),
    "phc_peer_reduce_create": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, C.c_int64, C.POINTER(C.c_void_p)]),
    "phc_peer_reduce_handle": (C.c_int, [C.c_void_p, C.c_void_p]),
    "phc_peer_reduce_connect": (C.c_int, [C.c_void_p, C.c_void_p]),
    "phc_peer_reduce_connect_local": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "phc_running_norm_update_peers": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p],
    ),
    "phc_peer_reduce_status": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "phc_peer_reduce_resync": (C.c_int, [C.c_void_p]),
    "phc_peer_reduce_destroy": (None, [C.c_void_p]),
}

_lib: Optional[C.CDLL] = None


class PhcError(RuntimeError):
    pass


def load() -> C.CDLL:
    """dlopen the in-tree shared object and type every entry point.  Raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PhcError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or humanoid_b200/csrc/build.sh. There is no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    if lib.phc_abi_version() != ABI_VERSION:
        raise PhcError(f"ABI version mismatch: library {lib.phc_abi_version()}, binding {ABI_VERSION}")
    _lib = lib
    return lib


def check(code: int, what: str) -> None:
    if code != 0:
        lib = load()
        msg = lib.phc_strerror(code).decode()
        extra = f" (cudaError {lib.phc_last_cuda_error()})" if code == -5 else ""
        raise PhcError(f"{what}: {msg}{extra}")


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def stream_ptr(device) -> int:
    """The caller's current CUDA stream on ``device`` as a raw pointer (looked up on every call: the caller may switch
    streams between steps).  torch's raw accessor when it is there (0.3 us; ``torch.cuda.current_stream()`` builds a
    Stream object: 3 us, twice per env step)."""
    if _raw_stream is not None:
        idx = device.index if isinstance(device, torch.device) else torch.device(device).index
        return _raw_stream(torch.cuda.current_device() if idx is None else idx)
    return torch.cuda.current_stream(device).cuda_stream


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def require_cuda(t: torch.Tensor, name: str, dtype=None) -> None:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise PhcError(f"{name} must be a CUDA tensor (there is no CPU path)")
    if dtype is not None and t.dtype != dtype:
        raise PhcError(f"{name} must be {dtype}, got {t.dtype}")


def view3(t: torch.Tensor, name: str) -> PhcView:
    """[n, J, C] fp32 tensor -> PhcView; a copy is made only if the last dim is strided."""
    require_cuda(t, name, torch.float32)
    if t.dim() != 3:
        raise PhcError(f"{name} must be [n, J, C], got {tuple(t.shape)}")
    if t.shape[-1] > 1 and t.stride(-1) != 1:
        t = t.contiguous()
    return PhcView(t.data_ptr(), t.stride(0), t.stride(1)), t


def body_state(pos, rot, vel, ang, prefix=""):
    """Four [n,J,.] views -> PhcBodyState (+ the tensors kept alive)."""
    vp, pos = view3(pos, prefix + "body_pos")
    vr, rot = view3(rot, prefix + "body_rot")
    vv, vel = view3(vel, prefix + "body_vel")
    va, ang = view3(ang, prefix + "body_ang_vel")
    n, J = pos.shape[0], pos.shape[1]
    for t, c, nm in ((pos, 3, "pos"), (rot, 4, "rot"), (vel, 3, "vel"), (ang, 3, "ang_vel")):
        if t.shape[0] != n or t.shape[1] != J or t.shape[2] != c:
            raise PhcError(f"{prefix}body_{nm} has shape {tuple(t.shape)}, expected [{n},{J},{c}]")
    return PhcBodyState(vp, vr, vv, va, J), (pos, rot, vel, ang)


def reward_spec(rwd_specs) -> PhcRewardSpec:
    """rwd_specs = asdict(RewardConfig) (humanoid_phc.py:1307-1311); extra keys are ignored."""
    return PhcRewardSpec(*[float(rwd_specs[k]) for k in (
        "k_pos", "k_rot", "k_vel", "k_ang_vel", "w_pos", "w_rot", "w_vel", "w_ang_vel")])  # fmt: skip
