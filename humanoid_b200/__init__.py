"""humanoid_b200 — B200-native per-step environment compute of puffer-phc's PHC humanoid task.

The hot path (motion-library query, smpl_max self observation, imitation observation v6,
imitation reward, reset/termination) as hand-written sm_100a CUDA kernels behind a C ABI
(include/phc_b200.h, libphc_b200.so), with Python drop-ins that keep the reference's function
signatures and tensor layouts.  There is no CPU fallback: importing is free, every call needs
the built shared object and a CUDA device.
"""

from .common import (  # noqa: F401
    build_amp_observations_smpl,
    dof_subset_smpl,
    compute_humanoid_im_reset,
    compute_humanoid_observations_smpl_max,
    compute_imitation_observations_v6,
    compute_imitation_observations_v7,
    compute_imitation_reward,
)
from .env import HumanoidPHC, build_pd_action_offset_scale  # noqa: F401
from .host_step import HostDeviceOutputs, HostResetBuffers, HostStep, HostStepBuffers  # noqa: F401
from .motion_lib import MotionLib  # noqa: F401
from .puffer_env import PHCPufferEnv  # noqa: F401
from .running_norm import RunningNorm  # noqa: F401

__all__ = [
    "MotionLib",
    "HumanoidPHC",
    "RunningNorm",
    "PHCPufferEnv",
    "compute_humanoid_observations_smpl_max",
    "compute_imitation_observations_v6",
    "compute_imitation_observations_v7",
    "compute_imitation_reward",
    "compute_humanoid_im_reset",
    "build_amp_observations_smpl",
    "dof_subset_smpl",
    "build_pd_action_offset_scale",
    "HostStep",
    "HostStepBuffers",
    "HostResetBuffers",
    "HostDeviceOutputs",
]
