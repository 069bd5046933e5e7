"""HumanoidPHC-shaped shim around the fused step kernel.

Mirrors the buffers and method names of the reference task env
(PHC/envs/humanoid_phc.py) for the part of ``step()`` that runs after the physics step
(:138-152).  Isaac Gym / PhysX is out of scope, so the rigid-body state is a plain tensor
``_rigid_body_state_reshaped [N, bodies_per_env, 13]`` that the owner fills (synthetic data
in tests and the bench; PhysX's buffer through gymtorch in the reference, :542-549).

Two ways to run the post-physics half:

* ``step()`` / ``post_physics_step()`` — one fused kernel launch (``phc_step_fused``): clock
  advance, motion query at t, reward, reset, motion query at t+dt.., self + task obs written
  as one ``obs_buf`` row.  No host sync, graph-capturable.
* ``_compute_reward`` / ``_compute_reset`` / ``_compute_observations`` — the reference's
  own decomposition, each calling the per-function drop-ins of ``humanoid_b200.common`` and
  ``MotionLib.get_motion_state`` (used for per-op parity and for ``env_ids`` subsets).
"""

from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence

import torch

from . import _cabi
from .common import (
    compute_humanoid_im_reset,
    compute_humanoid_observations_smpl_max,
    compute_imitation_observations_v6,
    compute_imitation_observations_v7,
    compute_imitation_reward,
)
from .motion_lib import MotionLib

BODY_NAMES = (
    "Pelvis", "L_Hip", "L_Knee", "L_Ankle", "L_Toe", "R_Hip", "R_Knee", "R_Ankle", "R_Toe", "Torso", "Spine",
    "Chest", "Neck", "Head", "L_Thorax", "L_Shoulder", "L_Elbow", "L_Wrist", "L_Hand", "R_Thorax", "R_Shoulder",
    "R_Elbow", "R_Wrist", "R_Hand",
)  # PHC/body_sets.py:11-36  # fmt: skip
REMOVE_NAMES = ("L_Hand", "R_Hand", "L_Toe", "R_Toe")  # body_sets.py:42
EVAL_BODIES = tuple(n for n in BODY_NAMES if n not in REMOVE_NAMES)  # body_sets.py:57
KEY_BODIES = ("R_Ankle", "L_Ankle", "R_Wrist", "L_Wrist")  # body_sets.py:45

DEFAULT_REWARD = dict(  # asdict(RewardConfig), PHC/config.py:38-50
    k_pos=100.0, k_rot=10.0, k_vel=0.1, k_ang_vel=0.1, w_pos=0.5, w_rot=0.3, w_vel=0.1, w_ang_vel=0.1,
    imitation_reward_dim=4, full_body_reward=True, use_power_reward=True,
)  # fmt: skip


OBS_MOMENT_BUCKETS = 32  # measured: 8 -> 13.1 us per 4096-env step, 32 -> 10.9, 128..2048 -> 10.8 (1 bucket: 41.9)


def build_body_ids_tensor(body_names: Sequence[str], subset: Sequence[str], device) -> torch.Tensor:
    """PHC/body_sets.py:143-158."""
    return torch.tensor([body_names.index(n) for n in subset], dtype=torch.long, device=device)


def build_pd_action_offset_scale(dof_limits_lower, dof_limits_upper, bias_offset: bool = False,
                                 has_smpl_pd_offset: bool = False, has_upright_start: bool = True):
    """``HumanoidPHC._build_pd_action_offset_scale`` (envs/humanoid_phc.py:385-457): the ``_pd_action_offset`` /
    ``_pd_action_scale`` that ``_action_to_pd_targets`` applies, from the asset's joint limits — host logic in the
    reference too (numpy over 23 three-dof joints), run once at start-up.  Per joint the range becomes
    +-min(1.2 max|limit|, pi) (with ``bias_offset``: mid +- 0.7 (high - low)); the knees' y axis gets scale 5
    (:443-446); ``has_smpl_pd_offset`` biases the shoulders.  Returns two CPU fp32 tensors [69]."""
    import numpy as np

    lim_low = torch.as_tensor(dof_limits_lower).detach().cpu().numpy().astype(np.float32).copy()
    lim_high = torch.as_tensor(dof_limits_upper).detach().cpu().numpy().astype(np.float32).copy()
    dof_names = BODY_NAMES[1:]
    for j in range(len(dof_names)):
        sl = slice(3 * j, 3 * j + 3)
        if not bias_offset:
            scale = min(1.2 * max(np.max(np.abs(lim_low[sl])), np.max(np.abs(lim_high[sl]))), np.pi)
            lim_low[sl], lim_high[sl] = -scale, scale
        else:
            mid = 0.5 * (lim_high[sl] + lim_low[sl])
            scale = 0.7 * (lim_high[sl] - lim_low[sl])
            lim_low[sl], lim_high[sl] = mid - scale, mid + scale
    offset = torch.from_numpy(0.5 * (lim_high + lim_low)).float()
    scale = torch.from_numpy(0.5 * (lim_high - lim_low)).float()
    scale[dof_names.index("L_Knee") * 3 + 1] = 5  # "Modified SMPL to give stronger knee"
    scale[dof_names.index("R_Knee") * 3 + 1] = 5
    if has_smpl_pd_offset:
        ls, rs = dof_names.index("L_Shoulder") * 3, dof_names.index("R_Shoulder") * 3
        if has_upright_start:
            offset[ls], offset[rs] = -np.pi / 2, np.pi / 2
        else:
            offset[ls], offset[ls + 2] = -np.pi / 6, -np.pi / 2
            offset[rs], offset[rs + 2] = -np.pi / 3, np.pi / 2
    return offset, scale


class HumanoidPHC:
    def __init__(
        self,
        motion_lib: MotionLib,
        num_envs: int,
        device="cuda",
        bodies_per_env: int = 24,
        time_steps: int = 1,
        termination_distance: float = 0.25,  # config.py:100
        enable_early_termination: bool = True,  # config.py:99
        dt: float = 2 * (1.0 / 60.0),  # isaacgym_env.py:39-41
        rwd_specs: Optional[Dict[str, float]] = None,
        obs_moments: bool = False,
        use_power_reward: bool = False,  # config.py:50 (True in the reference; needs dof_force / dof_vel)
        rew_power_coef: float = 0.0005,  # config.py:112
        use_amp_obs: bool = False,  # config.py:98
        num_amp_obs_steps: int = 10,  # config.py:141
        local_root_obs: bool = True,  # config.py:121
        root_height_obs: bool = True,  # config.py:122
        has_upright_start: bool = True,  # config.py:61
        res_action: bool = False,  # config.py (False by default, humanoid_phc.py:1219)
        obs_v: int = 6,  # imitation observation version (config obs_v): 6, or 7 = the [d_pos | d_vel | l_pos] columns of v6
    ):
        if obs_v not in (6, 7):
            raise ValueError(f"obs_v must be 6 or 7, got {obs_v!r}")
        dev = torch.device(device)
        if dev.type != "cuda":
            raise _cabi.PhcError("HumanoidPHC needs a CUDA device (there is no CPU path)")
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        self.device = dev
        self.num_envs = num_envs
        self.num_bodies = 24
        self.dt = dt
        self.time_steps = int(time_steps)
        self._motion_lib = motion_lib
        self.enable_early_termination = enable_early_termination
        self.flag_im_eval = False
        self._rwd_specs = dict(rwd_specs or DEFAULT_REWARD)
        self.use_power_reward = bool(use_power_reward)
        self.rew_power_coef = float(rew_power_coef)
        self.num_dof = 69
        # self-observation flags (humanoid_phc.py:963-998); the defaults are the env's constants
        self.local_root_obs, self.root_height_obs, self.has_upright_start = bool(local_root_obs), bool(root_height_obs), bool(has_upright_start)
        self._obs_flags = (
            (_cabi.OBS_LOCAL_ROOT if self.local_root_obs else 0) | (_cabi.OBS_ROOT_HEIGHT if self.root_height_obs else 0)
            | (_cabi.OBS_UPRIGHT if self.has_upright_start else 0) | _cabi.STEP_OBS_FLAGS_SET
            | (_cabi.OBS_TASK_V7 if obs_v == 7 else 0)
        )  # fmt: skip
        self.obs_v = obs_v
        self.res_action = bool(res_action)

        N = num_envs
        # sim tensors (stand-in for the gymtorch-wrapped PhysX buffer, humanoid_phc.py:542-549)
        self._rigid_body_state_reshaped = torch.zeros((N, bodies_per_env, 13), dtype=torch.float32, device=dev)
        self._bind_body_views()

        # dof state / force tensors (humanoid_phc.py:504-506, 533-536): (pos, vel) interleaved per dof
        self._dof_state = torch.zeros((N * self.num_dof, 2), dtype=torch.float32, device=dev)
        self._dof_pos = self._dof_state.view(N, self.num_dof, 2)[..., : self.num_dof, 0]
        self._dof_vel = self._dof_state.view(N, self.num_dof, 2)[..., : self.num_dof, 1]
        self.dof_force_tensor = torch.zeros((N, self.num_dof), dtype=torch.float32, device=dev)
        self._pd_action_offset = torch.zeros(self.num_dof, dtype=torch.float32, device=dev)  # :436-451
        self._pd_action_scale = torch.ones(self.num_dof, dtype=torch.float32, device=dev)

        # env buffers (humanoid_phc.py:556-597)
        task_dim = _cabi.TASK_OBS_DIM_V7 if obs_v == 7 else _cabi.TASK_OBS_DIM
        self.num_obs = (_cabi.SELF_OBS_DIM - (0 if self.root_height_obs else 1)) + task_dim * self.time_steps  # :461-467
        self.obs_buf = torch.zeros((N, self.num_obs), dtype=torch.float32, device=dev)
        self.rew_buf = torch.zeros(N, dtype=torch.float32, device=dev)  # (:560 calls the torch module; fixed)
        self.reward_raw = torch.zeros((N, 5), dtype=torch.float32, device=dev)  # 4 + power slot (:562-569)
        self.progress_buf = torch.zeros(N, dtype=torch.short, device=dev)
        self.reset_buf = torch.ones(N, dtype=torch.bool, device=dev)
        self._terminate_buf = torch.ones(N, dtype=torch.bool, device=dev)
        self.extras = {}
        # what the reference keeps as separate tensors: extras["terminate"] = _terminate_buf.clone() (:151) and the
        # step's reset flags (the in-step reset clears reset_buf / _terminate_buf as _reset_env_tensors does, :775-778)
        self._terminate_out = torch.zeros(N, dtype=torch.bool, device=dev)
        self._reset_out = torch.zeros(N, dtype=torch.bool, device=dev)
        self.ref_dof_pos = torch.zeros((N, self.num_dof), dtype=torch.float32, device=dev) if self.res_action else None  # :1119
        self._pd_target = torch.zeros((N, self.num_dof), dtype=torch.float32, device=dev)
        self._rew_out = None  # set_reward_copy(): the wrapper's rewards.clone() written by the step itself
        self.auto_reset = False  # enable_auto_reset(): the flagged envs are reset inside the step's launch
        self._phase_pool = None
        self._phase_cursor = 0
        self._reset_args = None
        self._global_offset = torch.zeros((N, 3), dtype=torch.float32, device=dev)
        self._motion_start_times = torch.zeros(N, dtype=torch.float32, device=dev)
        self._motion_start_times_offset = torch.zeros(N, dtype=torch.float32, device=dev)
        self._sampled_motion_ids = torch.arange(N, device=dev) % motion_lib.num_motions()
        self.all_env_ids = torch.arange(N, device=dev)

        # _config_env (humanoid_phc.py:239-250)
        self._termination_distances = torch.full((24,), termination_distance, dtype=torch.float32, device=dev)
        self._termination_distances_backup = self._termination_distances.clone()
        self._track_bodies_id = build_body_ids_tensor(BODY_NAMES, BODY_NAMES, dev)
        self._reset_bodies_id = build_body_ids_tensor(BODY_NAMES, BODY_NAMES, dev)
        self._reset_bodies_id_backup = self._reset_bodies_id.clone()
        self._eval_track_bodies_id = build_body_ids_tensor(BODY_NAMES, EVAL_BODIES, dev)

        # root state of the humanoid actor (humanoid_phc.py:518-523)
        self._humanoid_root_states = torch.zeros((N, 13), dtype=torch.float32, device=dev)
        # StateInit (envs/state_init.py, config.py:110,139): "random" (the default), "start", "default", "hybrid"
        self.state_init = "random"
        self.hybrid_init_prob = 0.5
        # what _reset_default restores (:521, :543-544; the reference clones them from the simulator at start-up)
        self._initial_humanoid_root_states = torch.zeros((N, 13), dtype=torch.float32, device=dev)
        self._initial_dof_pos = torch.zeros((N, self.num_dof), dtype=torch.float32, device=dev)
        self._initial_dof_vel = torch.zeros((N, self.num_dof), dtype=torch.float32, device=dev)
        self._default_mask = None  # hybrid: [N] uint8, 1 = the env takes the default path at its next reset
        self.flag_test = False

        # AMP observation buffers (humanoid_phc.py:186-194, 245, 469-478, 596-611)
        self.use_amp_obs = bool(use_amp_obs)
        self.num_amp_obs_steps = int(num_amp_obs_steps)
        dof_names = BODY_NAMES[1:]
        self.dof_subset = torch.tensor(
            [3 * i + k for i, n in enumerate(dof_names) if n not in REMOVE_NAMES for k in range(3)],
            dtype=torch.int64, device=dev,
        )  # fmt: skip
        self._key_body_ids = build_body_ids_tensor(BODY_NAMES, KEY_BODIES, dev)
        self._key_body_ids_host = [BODY_NAMES.index(n) for n in KEY_BODIES]
        self._num_amp_obs_per_step = (
            13 + len(dof_names) * 6 + self.num_dof + 3 * len(KEY_BODIES)
            - (6 + 3) * ((self.num_dof - len(self.dof_subset)) // 3)
        )  # fmt: skip
        self.num_amp_obs = self.num_amp_obs_steps * self._num_amp_obs_per_step
        if self.use_amp_obs:
            self._amp_obs_buf = torch.zeros(
                (N, self.num_amp_obs_steps, self._num_amp_obs_per_step), dtype=torch.float32, device=dev
            )
            self._curr_amp_obs_buf = self._amp_obs_buf[:, 0]
            self._hist_amp_obs_buf = self._amp_obs_buf[:, 1:]
            self._amp_obs_demo_buf = torch.zeros_like(self._amp_obs_buf)

        # RunningNorm partials accumulated by the step's epilogue.  fp64 atomics on one address serialise (~30 ns each),
        # so the blocks spread over OBS_MOMENT_BUCKETS accumulators that obs_moments / take_obs_moments() fold.
        self._obs_moment_buckets = (
            torch.zeros((OBS_MOMENT_BUCKETS, 2 * self.num_obs), dtype=torch.float64, device=dev) if obs_moments else None
        )
        self.obs_moment_rows = 0
        self.obs_normalizer = None  # set_obs_normalizer(): RunningNorm.forward fused into the step's epilogue
        self.obs_norm_buf = None
        self._mpjpe = None
        self._step_args = None

    # ------------------------------------------------------------------------------------
    @property
    def state_init_random(self) -> bool:
        """Round-1 spelling: True = StateInit.Random, False = StateInit.Start."""
        return self.state_init == "random"

    @state_init_random.setter
    def state_init_random(self, on: bool):
        self.state_init = "random" if on else "start"

    def _state_init_code(self) -> int:
        try:
            return {"start": _cabi.STATE_INIT_START, "random": _cabi.STATE_INIT_RANDOM,
                    "default": _cabi.STATE_INIT_DEFAULT, "hybrid": _cabi.STATE_INIT_HYBRID}[self.state_init]  # fmt: skip
        except KeyError:
            raise ValueError(f"Unsupported state initialization strategy: {self.state_init}")  # humanoid_phc.py:686

    def _fill_state_init(self, a, default_mask_by_env: Optional[torch.Tensor]):
        """StateInit fields of a PhcResetArgs.  Hybrid: ``default_mask_by_env`` [N] marks the envs that take the default
        path (the reference draws ``torch.bernoulli(hybrid_init_prob) == 1`` for reference-state init, :733-737); drawn
        here when omitted."""
        a.state_init = self._state_init_code()
        if self.state_init in ("default", "hybrid"):
            if self.use_amp_obs:
                raise NotImplementedError("Not tested yet")  # the reference's own words, humanoid_phc.py:795-797
            a.initial_root_states = self._initial_humanoid_root_states.data_ptr()
            a.initial_root_stride = self._initial_humanoid_root_states.stride(0)
            a.initial_dof_pos = self._initial_dof_pos.data_ptr()
            a.initial_dof_vel = self._initial_dof_vel.data_ptr()
            a.initial_dof_stride = self._initial_dof_pos.stride(0)
        if self.state_init == "hybrid":
            if default_mask_by_env is None:
                default_mask_by_env = torch.rand(self.num_envs, device=self.device) >= self.hybrid_init_prob
            self._default_mask = default_mask_by_env.to(self.device, torch.uint8).contiguous()
            a.default_mask = self._default_mask.data_ptr()

    # ------------------------------------------------------------------------------------
    @property
    def _reset_bodies_id(self) -> torch.Tensor:
        return self.__reset_bodies_id

    @_reset_bodies_id.setter
    def _reset_bodies_id(self, ids: torch.Tensor):
        """Assigning the index tensor (as toggle_eval_mode does, :1437) also refreshes the body
        bit mask the fused kernel takes; done here, once, so step() itself never reads the device."""
        self.__reset_bodies_id = ids
        mask = 0
        for b in ids.tolist():
            mask |= 1 << int(b)
        self._reset_mask = mask
        self._step_args = None

    def _bind_body_views(self):
        s = self._rigid_body_state_reshaped
        J = self.num_bodies
        self._rigid_body_pos = s[..., :J, 0:3]
        self._rigid_body_rot = s[..., :J, 3:7]
        self._rigid_body_vel = s[..., :J, 7:10]
        self._rigid_body_ang_vel = s[..., :J, 10:13]
        self._step_args = None

    def set_sim_state(self, state: torch.Tensor, copy: bool = True):
        """Stand-in for ``_refresh_sim_tensors`` (:782): adopt or copy an AoS [N,B,13] state."""
        if copy:
            self._rigid_body_state_reshaped.copy_(state)
        else:
            _cabi.require_cuda(state, "state", torch.float32)
            self._rigid_body_state_reshaped = state
            self._bind_body_views()

    def set_clock(self, clock):
        """Load a ``synth.Clock`` into the env's motion-clock buffers."""
        self.progress_buf.copy_(clock.progress_buf)
        self._motion_start_times.copy_(clock.motion_start_times)
        self._motion_start_times_offset.copy_(clock.motion_start_times_offset)
        self._global_offset.copy_(clock.global_offset)
        self._sampled_motion_ids.copy_(clock.sampled_motion_ids)

    @property
    def rwd_specs(self) -> Dict[str, float]:
        return self._rwd_specs

    def set_termination_distances(self, termination_distances):  # :1338-1339
        self._termination_distances[:] = termination_distances

    def set_motion_libs(self, train_lib, eval_lib):
        """``_motion_train_lib`` / ``_motion_eval_lib`` of ``_load_motion`` (:612-663): two ``MotionLibSMPL`` over the
        same clips, the second with ``im_eval=True`` (longest first, no heading, no crop)."""
        self._motion_train_lib, self._motion_eval_lib = train_lib, eval_lib
        self._motion_lib = train_lib

    def toggle_eval_mode(self, phase: Optional[torch.Tensor] = None):  # :1426-1440
        self.flag_test = True
        self.flag_im_eval = True
        self.set_termination_distances(0.5)
        self._step_args = None
        if getattr(self, "_motion_eval_lib", None) is not None:
            self._motion_lib = self._motion_eval_lib
            self.begin_seq_motion_samples(phase=phase)
        if len(self._reset_bodies_id) > 15:
            self._reset_bodies_id = self._eval_track_bodies_id
        return self._motion_lib.num_motions() if not hasattr(self._motion_lib, "_num_unique_motions") else self._motion_lib._num_unique_motions

    def untoggle_eval_mode(self, failed_keys=(), auto_pmcp: bool = False, auto_pmcp_soft: bool = True):  # :1441-1455
        self.flag_test = False
        self.flag_im_eval = False
        self._termination_distances[:] = self._termination_distances_backup
        self._reset_bodies_id = self._reset_bodies_id_backup
        self._step_args = None
        if getattr(self, "_motion_train_lib", None) is not None:
            self._motion_lib = self._motion_train_lib
            if auto_pmcp:  # config.py:103-104
                self._motion_lib.update_hard_sampling_weight(failed_keys)
            elif auto_pmcp_soft:
                self._motion_lib.update_soft_sampling_weight(failed_keys)
            return self._motion_lib._termination_history.clone()

    # ------------------------------------------------------------------------------------
    # fused path
    # ------------------------------------------------------------------------------------
    def _build_step_args(self, advance: bool):
        body, keep = _cabi.body_state(
            self._rigid_body_pos, self._rigid_body_rot, self._rigid_body_vel, self._rigid_body_ang_vel
        )
        mask = self._reset_mask
        a = _cabi.PhcStepArgs()
        a.body = body
        a.progress_buf = self.progress_buf.data_ptr()
        a.motion_start_times = self._motion_start_times.data_ptr()
        a.motion_start_times_offset = self._motion_start_times_offset.data_ptr()
        a.global_offset = self._global_offset.data_ptr()
        a.sampled_motion_ids = self._sampled_motion_ids.data_ptr()
        a.termination_distances = self._termination_distances.data_ptr()
        a.reset_body_mask = mask
        a.use_mean = 1 if self.flag_im_eval else 0
        a.enable_early_termination = 1 if self.enable_early_termination else 0
        a.advance_progress = 1 if advance else 0
        a.time_steps = self.time_steps
        a.dt = self.dt
        a.rwd = _cabi.reward_spec(self._rwd_specs)
        a.obs_buf = self.obs_buf.data_ptr()
        a.obs_stride = self.obs_buf.stride(0)
        a.rew_buf = self.rew_buf.data_ptr()
        a.reward_raw = self.reward_raw.data_ptr()
        a.reward_raw_stride = self.reward_raw.stride(0)
        # torch.bool is one byte holding 0/1 — the kernel writes uint8 0/1 straight into it
        a.reset_buf = self.reset_buf.data_ptr()
        a.terminate_buf = self._terminate_buf.data_ptr()
        a.terminate_out = self._terminate_out.data_ptr()
        a.reset_out = self._reset_out.data_ptr()
        a.obs_flags = self._obs_flags
        if self._rew_out is not None:
            a.rew_out = self._rew_out.data_ptr()
        if self.res_action:
            a.ref_dof_pos = self.ref_dof_pos.data_ptr()
            a.ref_dof_pos_stride = self.ref_dof_pos.stride(0)
        if self.auto_reset:  # humanoid_phc.py:665-676 for the envs this step flags, inside the step's launch
            self._reset_args = self._fill_reset_args(None, None)
            a.auto_reset = C.pointer(self._reset_args)
        if self._obs_moment_buckets is not None:
            a.obs_moments = self._obs_moment_buckets.data_ptr()
            a.obs_moments_buckets = self._obs_moment_buckets.shape[0]
        ep = getattr(self, "_episode_buffers", None)
        if ep is not None:  # PHCPufferEnv(fused=True): the wrapper's bookkeeping rides in the step (clean_pufferl/env.py:121-159)
            a.ep_terminals, a.ep_truncations, a.ep_masks = (ep[k].data_ptr() for k in ("terminals", "truncations", "masks"))
            a.ep_returns, a.ep_lengths = ep["episode_returns"].data_ptr(), ep["episode_lengths"].data_ptr()
            a.ep_sums, a.ep_buckets = ep["sums"].data_ptr(), ep["sums"].shape[0]
            a.ep_raw_cols = self.reward_raw.shape[1]
        if self.flag_im_eval:  # extras["mpjpe"] (:159-167), from the distances the reset test computes anyway
            if self._mpjpe is None:
                self._mpjpe = torch.zeros(self.num_envs, dtype=torch.float32, device=self.device)
            a.mpjpe = self._mpjpe.data_ptr()
        if self.obs_normalizer is not None:  # policies/running_norm.py:15-20, fused
            rn = self.obs_normalizer
            a.obs_norm = self.obs_norm_buf.data_ptr()
            a.obs_norm_stride = self.obs_norm_buf.stride(0)
            a.norm_mean = rn.running_mean.data_ptr()
            a.norm_var = rn.running_var.data_ptr()
            a.norm_epsilon = rn.epsilon
            a.norm_clip = rn.clip
            if self.obs_norm_buf.dtype == torch.bfloat16:
                a.flags |= _cabi.STEP_OBS_NORM_BF16
        if self.use_power_reward:  # humanoid_phc.py:1297-1305
            a.dof_force = self.dof_force_tensor.data_ptr()
            a.dof_force_stride = self.dof_force_tensor.stride(0)
            a.dof_vel = self._dof_vel.data_ptr()
            a.dof_vel_stride = self._dof_vel.stride(0)
            a.dof_vel_elem_stride = self._dof_vel.stride(1)
            a.rew_power_coef = self.rew_power_coef
            a.power_col = self.reward_raw.shape[1] - 1
        self._step_args = (a, advance, keep, (self.flag_im_eval, self.use_power_reward, self.time_steps))
        return a

    @property
    def obs_moments(self) -> Optional[torch.Tensor]:
        """fp64 ``[sum x | sum x^2]`` over every row the step has written since the last ``take_obs_moments()``."""
        return None if self._obs_moment_buckets is None else self._obs_moment_buckets.sum(0)

    def take_obs_moments(self, sums: Optional[torch.Tensor] = None):
        """Fold the buckets into ``sums`` (+=, allocated when omitted), zero them, and return ``(sums, rows)`` — what
        ``RunningNorm.update_from_moments`` takes once per rollout (phc_train.py:331-332)."""
        if self._obs_moment_buckets is None:
            raise _cabi.PhcError("the env was built without obs_moments=True")
        b = self._obs_moment_buckets
        if sums is None:
            sums = torch.zeros(b.shape[1], dtype=torch.float64, device=self.device)
        _cabi.check(
            _cabi.load().phc_obs_moments_fold(b.data_ptr(), b.shape[0], b.shape[1], sums.data_ptr(), _cabi.stream_ptr(self.device)),
            "phc_obs_moments_fold",
        )  # fmt: skip
        rows, self.obs_moment_rows = self.obs_moment_rows, 0
        return sums, rows

    def set_episode_buffers(self, buffers: Optional[Dict[str, torch.Tensor]]):
        """Let the step do ``PHCPufferEnv.step``'s per-env episode bookkeeping: ``terminals / truncations / masks`` (bool
        [N]), ``episode_returns`` (f32 [N]), ``episode_lengths`` (i32 [N]) and ``sums`` (f64 [B, 12] accumulators)."""
        self._episode_buffers = buffers
        self._step_args = None

    def set_reward_copy(self, rew_out: Optional[torch.Tensor]):
        """``rew = self.rewards.clone()`` of ``PHCPufferEnv.step`` (clean_pufferl/env.py:121) as a second output of the
        step kernel: ``rew_out [N]`` receives what ``rew_buf`` receives."""
        if rew_out is not None:
            _cabi.require_cuda(rew_out, "rew_out", torch.float32)
        self._rew_out = rew_out
        self._step_args = None

    def enable_auto_reset(self, on: bool = True, phase_pool_steps: int = 32):
        """Reset the envs a step flags INSIDE that step's launch (``PhcStepArgs.auto_reset``): what
        ``PHCPufferEnv.step`` does with ``nonzero(reset_buf)`` + ``env.reset(indices)`` (clean_pufferl/env.py:133-135)
        with no second launch and no host sync.  After such a step ``reset_buf`` / ``_terminate_buf`` read 0 (as
        after the reference's reset, humanoid_phc.py:775-778); the step's own flags are ``extras["reset"]`` /
        ``extras["terminate"]``.  The uniform numbers of ``sample_time_interval`` come from a pool drawn
        ``phase_pool_steps`` steps at a time (one ``torch.rand`` launch per that many steps) unless ``step(phase_by_env=...)``
        supplies them.  Buffers are bit-identical to ``step()`` followed by ``reset_done(phase)``."""
        self.auto_reset = bool(on)
        self._phase_pool_steps = int(phase_pool_steps)
        self._step_args = None

    def _next_phase(self, phase_by_env: Optional[torch.Tensor]) -> torch.Tensor:
        if phase_by_env is not None:
            ph = phase_by_env.to(self.device, torch.float32).contiguous()
            self._phase_keep = ph
            return ph
        P = self._phase_pool_steps
        if self._phase_pool is None or self._phase_cursor >= P:
            if self._phase_pool is None:
                self._phase_pool = torch.empty((P, self.num_envs), dtype=torch.float32, device=self.device)
            self._phase_pool.uniform_()
            self._phase_cursor = 0
        ph = self._phase_pool[self._phase_cursor]
        self._phase_cursor += 1
        return ph

    def set_obs_normalizer(self, normalizer, dtype=torch.float32):
        """Fuse ``RunningNorm.forward`` (PHC/policies/running_norm.py:15-20) into the step: every step also
        writes ``obs_norm_buf = clamp((obs_buf - running_mean) / sqrt(running_var + eps), -clip, clip)`` —
        what the policy's first layer consumes — from the same shared-memory rows, while ``obs_buf`` keeps
        the raw rows the experience buffer and ``RunningNorm.update`` need.  The normaliser's buffers are
        read at launch time, so an ``update()`` between steps is seen by the next step.  ``None`` turns it off.
        ``dtype=torch.bfloat16`` emits the normalised rows as bf16 (each fp32 result rounded to nearest-even):
        the policy's input under autocast, at half the bytes."""
        if normalizer is not None:
            if normalizer.shape != self.num_obs or normalizer.running_mean.device != self.device:
                raise ValueError("normalizer must have shape num_obs and live on the env's device")
            if dtype not in (torch.float32, torch.bfloat16):
                raise ValueError("obs_norm_buf is float32 or bfloat16")
            if self.obs_norm_buf is None or self.obs_norm_buf.dtype != dtype:
                self.obs_norm_buf = torch.zeros_like(self.obs_buf, dtype=dtype)
        self.obs_normalizer = normalizer
        self._step_args = None

    def _refresh_step_scalars(self, a):
        """The cached ``PhcStepArgs`` keeps pointers and strides; everything a reference-style script may change by
        plain attribute assignment between steps (``env.flag_im_eval = True``, ``env.rwd_specs[...] = ...``,
        ``env.enable_early_termination``, ``env.dt``, the power-reward switches) is re-read on every step, as the
        unfused ``_compute_*`` path does."""
        a.use_mean = 1 if self.flag_im_eval else 0
        a.enable_early_termination = 1 if self.enable_early_termination else 0
        a.dt = self.dt
        r = self._rwd_specs
        a.rwd.k_pos, a.rwd.k_rot, a.rwd.k_vel, a.rwd.k_ang_vel = r["k_pos"], r["k_rot"], r["k_vel"], r["k_ang_vel"]
        a.rwd.w_pos, a.rwd.w_rot, a.rwd.w_vel, a.rwd.w_ang_vel = r["w_pos"], r["w_rot"], r["w_vel"], r["w_ang_vel"]
        a.rew_power_coef = self.rew_power_coef

    def post_physics_step(self, advance_progress: bool = True, phase_by_env: Optional[torch.Tensor] = None,
                          default_mask_by_env: Optional[torch.Tensor] = None):
        """progress += 1; reward; reset; observations (humanoid_phc.py:138-149) — one launch (with ``auto_reset`` the
        reset of the flagged envs and their new observation rows too)."""
        cached = self._step_args
        if (cached is None or cached[1] != advance_progress or cached[3] != (self.flag_im_eval, self.use_power_reward,
                                                                             self.time_steps)):  # fmt: skip
            self._build_step_args(advance_progress)  # these three change which pointers the struct carries
        a = self._step_args[0]
        self._refresh_step_scalars(a)
        if self.auto_reset:
            r = self._reset_args
            r.phase = self._next_phase(phase_by_env).data_ptr()
            self._fill_state_init(r, default_mask_by_env)
            r.flag_test = 1 if self.flag_test else 0
            r.dt = self.dt
        _cabi.check(
            _cabi.load().phc_step_fused(
                self._motion_lib.handle, C.byref(a), self.num_envs, _cabi.stream_ptr(self.device)
            ),
            "phc_step_fused",
        )
        if self._obs_moment_buckets is not None:
            self.obs_moment_rows += self.num_envs

    def pre_physics_step(self, actions: torch.Tensor, clip: float = 0.0, actions_out: Optional[torch.Tensor] = None):
        """The pre-physics half of ``step`` (:105-128): actions -> PD targets in ``self._pd_target`` (what the
        reference hands to ``gym.set_dof_position_target_tensor``), one launch.  With ``clip`` the wrapper's
        ``np.clip(actions, -clip, clip)`` (clean_pufferl/env.py:110-112) rides in the same launch and the clipped
        actions are stored in ``actions_out``."""
        return self._action_to_pd_targets(actions, res_action=self.res_action, ref_dof_pos=self.ref_dof_pos,
                                          clip=clip, actions_out=actions_out, out=self._pd_target)  # fmt: skip

    def step(self, actions=None, phase_by_env: Optional[torch.Tensor] = None,
             default_mask_by_env: Optional[torch.Tensor] = None):
        """The reference's ``step`` minus PhysX (out of scope): the caller has already written the post-physics
        rigid-body state.  ``actions`` (optional) are turned into PD targets first, as :105-128 does."""
        if actions is not None:
            self.pre_physics_step(actions)
        self.post_physics_step(True, phase_by_env, default_mask_by_env)
        self.extras["terminate"] = self._terminate_out  # = _terminate_buf.clone() (:151)
        self.extras["reset"] = self._reset_out
        self.extras["reward_raw"] = self.reward_raw
        if self.use_amp_obs:  # :153-157
            self._amp_step(roll=True)
            self.extras["amp_obs"] = self.amp_obs
            if self.auto_reset:  # _reset_envs (:675-676) for the envs the step has just reset
                self._init_amp_obs_masked(self._reset_out)
        if self.flag_im_eval:  # :159-167 (body_pos / body_pos_gt are host copies the caller can take itself)
            self.extras["mpjpe"] = self._mpjpe
        return self.obs_buf, self.rew_buf, self.reset_buf, self.extras

    # ------------------------------------------------------------------------------------
    # AMP observation buffers (humanoid_phc.py:791-843, 1125-1176, 1341-1361)
    # ------------------------------------------------------------------------------------
    @property
    def amp_obs(self):  # :1356-1358
        return self._amp_obs_buf.view(-1, self.num_amp_obs) if self.use_amp_obs else None

    def fetch_amp_obs_demo(self):  # :1360-1361
        return self._amp_obs_demo_buf.view(-1, self.num_amp_obs) if self.use_amp_obs else None

    def _amp_args(self, mask: Optional[torch.Tensor]):
        body, keep = _cabi.body_state(
            self._rigid_body_pos, self._rigid_body_rot, self._rigid_body_vel, self._rigid_body_ang_vel
        )
        a = _cabi.PhcAmpEnvArgs()
        a.body = body
        a.dof_pos, a.dof_vel = self._dof_pos.data_ptr(), self._dof_vel.data_ptr()
        a.dof_stride, a.dof_elem_stride = self._dof_pos.stride(0), self._dof_pos.stride(1)
        for i, b in enumerate(self._key_body_ids_host):
            a.key_body_ids[i] = int(b)
        a.num_key_bodies = len(self._key_body_ids_host)
        a.num_sel = int(self.dof_subset.shape[0])
        a.dof_subset = self.dof_subset.data_ptr()
        a.flags = _cabi.OBS_LOCAL_ROOT | _cabi.OBS_ROOT_HEIGHT | _cabi.OBS_UPRIGHT  # the config's constants (:1206-1211)
        a.num_steps, a.obs_per_step = self.num_amp_obs_steps, self._num_amp_obs_per_step
        a.amp_obs_buf = self._amp_obs_buf.data_ptr()
        a.amp_obs_demo_buf = self._amp_obs_demo_buf.data_ptr()
        a.env_mask = _cabi.ptr(mask)
        return a, keep

    def _amp_step(self, roll: bool, mask: Optional[torch.Tensor] = None):
        """``_update_hist_amp_obs()`` (when ``roll``) + ``_compute_amp_observations()``; one launch."""
        a, keep = self._amp_args(mask)
        _cabi.check(
            _cabi.load().phc_amp_step(C.byref(a), self.num_envs, 1 if roll else 0, _cabi.stream_ptr(self.device)),
            "phc_amp_step",
        )

    def _update_hist_amp_obs(self, env_ids=None):  # :1341-1350 (only reached through _amp_step here)
        raise NotImplementedError("fused with _compute_amp_observations: use _amp_step(roll=True)")

    def _compute_amp_observations(self, env_ids=None):  # :1125-1176
        mask = None
        if env_ids is not None:
            mask = torch.zeros(self.num_envs, dtype=torch.bool, device=self.device)
            mask[env_ids] = True
        self._amp_step(roll=False, mask=mask)

    def _init_amp_obs_masked(self, mask: torch.Tensor):
        """``_init_amp_obs(env_ids)`` (:791-799) for the envs of a byte mask, right after their reset:
        slot 0 from the freshly set sim state, the history from the motion library, the demo rows."""
        a, keep = self._amp_args(mask)
        a.init_slot0 = 1  # _compute_amp_observations(env_ids) rides in the same launch
        _cabi.check(
            _cabi.load().phc_amp_init_ref(
                self._motion_lib.handle, C.byref(a), self._sampled_motion_ids.data_ptr(),
                self._motion_start_times.data_ptr(), self.dt, self.num_envs, _cabi.stream_ptr(self.device),
            ),
            "phc_amp_init_ref",
        )  # fmt: skip

    # ------------------------------------------------------------------------------------
    # pre-physics: actions -> PD targets (humanoid_phc.py:105-128, 1218-1228)
    # ------------------------------------------------------------------------------------
    def build_pd_action_offset_scale(self, dof_limits_lower, dof_limits_upper, bias_offset: bool = False,
                                     has_smpl_pd_offset: bool = False, has_upright_start: bool = True):
        """``_build_pd_action_offset_scale`` (:385-457) into ``self._pd_action_offset`` / ``_pd_action_scale``."""
        offset, scale = build_pd_action_offset_scale(dof_limits_lower, dof_limits_upper, bias_offset, has_smpl_pd_offset,
                                                     has_upright_start)  # fmt: skip
        self._pd_action_offset, self._pd_action_scale = offset.to(self.device), scale.to(self.device)
        return self._pd_action_offset, self._pd_action_scale

    def _action_to_pd_targets(self, action: torch.Tensor, res_action: bool = False, ref_dof_pos=None,
                              freeze_hand: bool = False, freeze_toe: bool = False, clip: float = 0.0,
                              actions_out: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:  # fmt: skip
        """``pd_action_offset + pd_action_scale * action`` (or the clamped residual form), with the
        hand / toe joints zeroed as ``step()`` does when ``freeze_hand`` / ``freeze_toe`` are set.
        ``self._pd_action_offset`` / ``_pd_action_scale`` are [69] tensors the owner fills
        (built from the asset's joint limits in the reference, :385-451)."""
        _cabi.require_cuda(action, "action", torch.float32)
        action = action.contiguous()
        n, D = action.shape
        if out is None:
            out = torch.empty_like(action)
        if actions_out is not None:
            _cabi.require_cuda(actions_out, "actions_out", torch.float32)
            if actions_out.shape != action.shape or not actions_out.is_contiguous():
                raise ValueError("actions_out must be a contiguous tensor of the actions' shape")
        dof_names = BODY_NAMES[1:]
        mask = 0
        if freeze_hand:
            mask |= (1 << dof_names.index("L_Hand")) | (1 << dof_names.index("R_Hand"))
        if freeze_toe:
            mask |= (1 << dof_names.index("L_Toe")) | (1 << dof_names.index("R_Toe"))
        ref = ref_dof_pos.contiguous() if res_action else None
        _cabi.check(
            _cabi.load().phc_action_to_pd_targets(
                action.data_ptr(), self._pd_action_offset.data_ptr(), self._pd_action_scale.data_ptr(),
                1 if res_action else 0, _cabi.ptr(ref), self._dof_pos.data_ptr(), self._dof_pos.stride(0),
                self._dof_pos.stride(1), mask, n, D, float(clip), _cabi.ptr(actions_out), out.data_ptr(),
                _cabi.stream_ptr(self.device),
            ),
            "phc_action_to_pd_targets",
        )  # fmt: skip
        return out

    # ------------------------------------------------------------------------------------
    # reset (humanoid_phc.py:90-103, 665-778) — on the device, no host sync
    # ------------------------------------------------------------------------------------
    def _fill_reset_args(self, mask: Optional[torch.Tensor], phase_by_env: Optional[torch.Tensor], moments_mode: int = 0,
                         default_mask_by_env: Optional[torch.Tensor] = None):
        body, keep = _cabi.body_state(
            self._rigid_body_pos, self._rigid_body_rot, self._rigid_body_vel, self._rigid_body_ang_vel
        )
        a = _cabi.PhcResetArgs()
        a.body = body
        a.humanoid_root_states = self._humanoid_root_states.data_ptr()
        a.root_stride = self._humanoid_root_states.stride(0)
        a.dof_pos = self._dof_pos.data_ptr()
        a.dof_vel = self._dof_vel.data_ptr()
        a.dof_stride = self._dof_pos.stride(0)
        a.dof_elem_stride = self._dof_pos.stride(1)
        a.progress_buf = self.progress_buf.data_ptr()
        a.reset_buf = self.reset_buf.data_ptr()
        a.terminate_buf = self._terminate_buf.data_ptr()
        a.motion_start_times = self._motion_start_times.data_ptr()
        a.motion_start_times_offset = self._motion_start_times_offset.data_ptr()
        a.global_offset = self._global_offset.data_ptr()
        a.sampled_motion_ids = self._sampled_motion_ids.data_ptr()
        a.env_mask = _cabi.ptr(mask)
        a.phase = _cabi.ptr(phase_by_env)
        self._fill_state_init(a, default_mask_by_env)
        a.flag_test = 1 if self.flag_test else 0
        a.time_steps = self.time_steps
        a.dt = self.dt
        a.obs_buf = self.obs_buf.data_ptr()
        a.obs_stride = self.obs_buf.stride(0)
        a.obs_flags = self._obs_flags
        if self.res_action:
            a.ref_dof_pos = self.ref_dof_pos.data_ptr()
            a.ref_dof_pos_stride = self.ref_dof_pos.stride(0)
        # keep the step's fused epilogues consistent with the rows a reset rewrites: the policy reads obs_norm_buf,
        # and RunningNorm.update must see the rows the policy saw (experience.obs holds the post-reset rows)
        if self.obs_normalizer is not None:
            rn = self.obs_normalizer
            a.obs_norm = self.obs_norm_buf.data_ptr()
            a.obs_norm_stride = self.obs_norm_buf.stride(0)
            a.norm_mean, a.norm_var = rn.running_mean.data_ptr(), rn.running_var.data_ptr()
            a.norm_epsilon, a.norm_clip = rn.epsilon, rn.clip
            a.obs_norm_bf16 = 1 if self.obs_norm_buf.dtype == torch.bfloat16 else 0
        if self._obs_moment_buckets is not None and moments_mode:
            a.obs_moments_mode = moments_mode
            a.obs_moments = self._obs_moment_buckets.data_ptr()
            a.obs_moments_buckets = self._obs_moment_buckets.shape[0]
        a._keep = (keep, mask, phase_by_env)
        return a

    def _reset_masked(self, mask: torch.Tensor, phase_by_env: torch.Tensor, moments_mode: int = 0,
                      default_mask_by_env: Optional[torch.Tensor] = None):
        """``moments_mode``: 1 = the new rows are added to the step's RunningNorm partials (rows never counted: a
        ``reset()``), 2 = they replace the rows the flagging step had counted (``reset_done()``)."""
        a = self._fill_reset_args(mask, phase_by_env, moments_mode, default_mask_by_env)
        _cabi.check(
            _cabi.load().phc_reset_envs(self._motion_lib.handle, C.byref(a), self.num_envs, _cabi.stream_ptr(self.device)),
            "phc_reset_envs",
        )
        if self.use_amp_obs:  # _reset_envs (:675-676)
            self._init_amp_obs_masked(mask)

    def reset(self, env_ids=None, phase: Optional[torch.Tensor] = None, default_mask: Optional[torch.Tensor] = None):
        """``HumanoidPHC.reset(env_ids)`` (:90-103).  Reference-state init (``state_init`` "random" / "start"): sample a
        start time per env (``sample_time_interval``), pose the env from the motion library, reset its clock and
        buffers, recompute its observation.  ``phase`` are the uniform numbers the reference draws with
        ``torch.rand(len(env_ids))``; drawn here when omitted.  ``state_init`` "default": root / dof state from the
        initial buffers, clock and rigid-body state untouched (:688-692).  "hybrid": ``default_mask``
        [len(env_ids)] picks the envs that take the default path (the reference's ``torch.bernoulli(hybrid_init_prob)
        != 1``; drawn here when omitted); ``phase`` then has one number per env_id, or — as the reference draws them —
        one per reference-init env.  The second, PhysX-settling pass of ``safe_reset`` (:97-101) is out of scope."""
        if env_ids is None:
            env_ids = self.all_env_ids
        env_ids = env_ids.to(self.device)
        dmask_by_env = None
        ref_ids = env_ids
        if self.state_init == "hybrid":
            if default_mask is None:
                default_mask = torch.rand(env_ids.shape, device=self.device) >= self.hybrid_init_prob
            default_mask = default_mask.to(self.device, torch.bool)
            dmask_by_env = torch.zeros(self.num_envs, dtype=torch.bool, device=self.device)
            dmask_by_env[env_ids] = default_mask
            ref_ids = env_ids[~default_mask]
        elif self.state_init == "default":
            ref_ids = env_ids[:0]
        if phase is None:
            phase = torch.rand(ref_ids.shape, device=self.device)
        mask = torch.zeros(self.num_envs, dtype=torch.bool, device=self.device)
        mask[env_ids] = True
        by_env = torch.zeros(self.num_envs, dtype=torch.float32, device=self.device)
        by_env[ref_ids if phase.shape[0] == ref_ids.shape[0] else env_ids] = phase.to(self.device, torch.float32)
        self._reset_masked(mask, by_env, moments_mode=1, default_mask_by_env=dmask_by_env)
        if self._obs_moment_buckets is not None:
            self.obs_moment_rows += int(env_ids.numel())  # rows the policy will see and no step has counted
        return self.obs_buf

    def reset_done(self, phase_by_env: Optional[torch.Tensor] = None, default_mask_by_env: Optional[torch.Tensor] = None):
        """Reset every env whose ``reset_buf`` is set, entirely on the device: replaces the
        ``nonzero(reset_buf)`` + ``env.reset(reset_indices)`` of clean_pufferl/env.py:133-135 and its
        host sync.  ``phase_by_env [N]`` supplies one uniform number per env (used where flagged);
        ``default_mask_by_env [N]`` the hybrid-init choice per env (drawn here when omitted)."""
        if phase_by_env is None:
            phase_by_env = torch.rand(self.num_envs, device=self.device)
        # the reset kernel reads each mask byte once before it clears reset_buf, so reset_buf can be its own mask;
        # the AMP initialisation that follows needs the flags after they are cleared, hence the copy there
        mask = self.reset_buf.clone() if self.use_amp_obs else self.reset_buf
        self._reset_masked(mask, phase_by_env.to(self.device, torch.float32).contiguous(), moments_mode=2,
                           default_mask_by_env=default_mask_by_env)
        return self.obs_buf

    def set_humanoid_assets(self, skeleton_trees, humanoid_shapes, humanoid_limb_and_weights):
        """What ``_load_motion`` / ``resample_motions`` hand the loader (humanoid_phc.py:360, 418-419, 640-647):
        one skeleton tree, one [17] gender+beta row and one [10] limb-weight row per env."""
        self.skeleton_trees = list(skeleton_trees)
        self.humanoid_shapes = humanoid_shapes
        self.humanoid_limb_and_weights = humanoid_limb_and_weights

    def resample_motions(self, seq_motions: bool = False, phase: Optional[torch.Tensor] = None):
        """``resample_motions`` (:1363-1379), training branch: rebuild the library on the device from a fresh
        sample of clips (``MotionLibSMPL.load_motions``), re-anchor the xy global offset so every env's
        reference root passes through where its humanoid stands now, then reset every env."""
        if self.flag_test:
            return self.forward_motion_samples(phase=phase)
        self._motion_lib.load_motions(
            skeleton_trees=self.skeleton_trees,
            limb_weights=self.humanoid_limb_and_weights.cpu(),
            gender_betas=self.humanoid_shapes.cpu(),
            random_sample=(not self.flag_test) and (not seq_motions),
        )
        time = self.progress_buf * self.dt + self._motion_start_times + self._motion_start_times_offset
        root_res = self._motion_lib.get_root_pos_smpl(self._sampled_motion_ids, time)
        self._global_offset[:, :2] = self._humanoid_root_states[:, :2] - root_res["root_pos"][:, :2]
        return self.reset(phase=phase)

    def _load_seq(self, phase):
        self._motion_lib.load_motions(
            skeleton_trees=self.skeleton_trees,
            gender_betas=self.humanoid_shapes.cpu(),
            limb_weights=self.humanoid_limb_and_weights.cpu(),
            random_sample=False,
            start_idx=self._motion_sample_start_idx,
        )
        return self.reset(phase=phase)

    def begin_seq_motion_samples(self, phase: Optional[torch.Tensor] = None):  # :1381-1391, evaluation sweep
        self._motion_sample_start_idx = 0
        return self._load_seq(phase)

    def forward_motion_samples(self, phase: Optional[torch.Tensor] = None):  # :1393-1402
        self._motion_sample_start_idx += self.num_envs
        return self._load_seq(phase)

    @property
    def num_unique_motions(self):  # :1404-1418
        return self._motion_lib._num_unique_motions

    @property
    def current_motion_ids(self):
        return self._motion_lib._curr_motion_ids

    @property
    def motion_sample_start_idx(self):
        return self._motion_sample_start_idx

    @property
    def motion_data_keys(self):
        return self._motion_lib._motion_data_keys

    def get_motion_steps(self):  # :1420-1421
        return self._motion_lib.get_motion_num_steps()

    # ------------------------------------------------------------------------------------
    # the reference's decomposition, on the per-function kernels
    # ------------------------------------------------------------------------------------
    def _motion_times(self, env_ids=None, plus: int = 0):
        p = self.progress_buf if env_ids is None else self.progress_buf[env_ids]
        s = self._motion_start_times if env_ids is None else self._motion_start_times[env_ids]
        o = self._motion_start_times_offset if env_ids is None else self._motion_start_times_offset[env_ids]
        return (p + plus) * self.dt + s + o if plus else p * self.dt + s + o

    def _compute_reward(self):  # :1230-1271
        t = self._motion_times()
        ref = self._motion_lib.get_motion_state(self._sampled_motion_ids, t, self._global_offset)
        pos, rot, vel, ang = self._rigid_body_pos, self._rigid_body_rot, self._rigid_body_vel, self._rigid_body_ang_vel
        self.rew_buf[:], self.reward_raw[:, :4] = compute_imitation_reward(
            pos[..., 0, :], rot[..., 0, :], pos, rot, vel, ang,
            ref["rg_pos"], ref["rb_rot"], ref["body_vel"], ref["body_ang_vel"], self.rwd_specs,
        )  # fmt: skip
        if self.use_power_reward:  # :1297-1305 — plain torch ops; the fused step does this in-kernel
            power = torch.abs(torch.multiply(self.dof_force_tensor, self._dof_vel)).sum(dim=-1)
            power_reward = -self.rew_power_coef * power
            power_reward[self.progress_buf <= 3] = 0
            self.rew_buf[:] += power_reward
            self.reward_raw[:, -1] = power_reward

    def _compute_reset(self):  # :1313-1335
        t = self._motion_times()
        pass_time = t >= self._motion_lib._motion_lengths[self._sampled_motion_ids]
        ref = self._motion_lib.get_motion_state(self._sampled_motion_ids, t, self._global_offset)
        ids = self._reset_bodies_id
        self.reset_buf[:], self._terminate_buf[:] = compute_humanoid_im_reset(
            self.reset_buf, self.progress_buf, None, None,
            self._rigid_body_pos[..., ids, :].clone(), ref["rg_pos"][..., ids, :].clone(), pass_time,
            self.enable_early_termination, self._termination_distances[..., ids], self.flag_im_eval,
        )  # fmt: skip

    def _compute_humanoid_obs(self, env_ids=None):  # :963-998
        sel = (lambda x: x) if env_ids is None else (lambda x: x[env_ids])
        return compute_humanoid_observations_smpl_max(
            sel(self._rigid_body_pos), sel(self._rigid_body_rot), sel(self._rigid_body_vel),
            sel(self._rigid_body_ang_vel), None, None, self.local_root_obs, self.root_height_obs,
            self.has_upright_start, False, False,
        )  # fmt: skip

    def _compute_task_obs(self, env_ids=None):  # :1050-1123
        sel = (lambda x: x) if env_ids is None else (lambda x: x[env_ids])
        pos, rot = sel(self._rigid_body_pos), sel(self._rigid_body_rot)
        vel, ang = sel(self._rigid_body_vel), sel(self._rigid_body_ang_vel)
        ids, off = sel(self._sampled_motion_ids), sel(self._global_offset)
        refs = [self._motion_lib.get_motion_state(ids, self._motion_times(env_ids, k), off)
                for k in range(1, self.time_steps + 1)]  # fmt: skip

        def stack(key):
            if len(refs) == 1:
                return refs[0][key]
            return torch.stack([r[key] for r in refs], dim=1).flatten(0, 1)

        if self.res_action:  # :1115-1120
            if env_ids is None:
                self.ref_dof_pos[:] = refs[0]["dof_pos"]
            else:
                self.ref_dof_pos[env_ids] = refs[0]["dof_pos"]
        task_obs = compute_imitation_observations_v7 if self.obs_v == 7 else compute_imitation_observations_v6
        return task_obs(
            pos[..., 0, :], rot[..., 0, :], pos, rot, vel, ang,
            stack("rg_pos"), stack("rb_rot"), stack("body_vel"), stack("body_ang_vel"), self.time_steps,
            self.has_upright_start,
        )  # fmt: skip

    def _compute_observations(self, env_ids=None):  # :937-961
        obs = torch.cat([self._compute_humanoid_obs(env_ids), self._compute_task_obs(env_ids)], dim=-1)
        if env_ids is None:
            self.obs_buf[:] = obs
        else:
            self.obs_buf[env_ids] = obs
        return obs

    def post_physics_step_unfused(self):
        """Same result as ``post_physics_step`` through the per-function kernels."""
        self.progress_buf += 1
        self._compute_reward()
        self._compute_reset()
        self._compute_observations()
