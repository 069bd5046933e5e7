"""``PHCPufferEnv`` — the pufferlib-facing wrapper of the reference (clean_pufferl/env.py:39-204)
over the B200 ``HumanoidPHC`` shim, with the per-step episode bookkeeping (:121-159) as one
kernel (``phc_episode_update``) and the reset of flagged envs on the device (``reset_done``).

``fused=True`` is the whole wrapper step in TWO launches around the physics: (1) the action clip (:110-112) with
the PD targets of ``env.step`` (humanoid_phc.py:105-128) — ``phc_action_to_pd_targets`` — and (2) the fused step
with the episode bookkeeping, the ``rewards.clone()`` (:121) and the reset of the flagged envs (:133-135) inside it.

What changes against the reference, and why: the reference finds the flagged envs with
``torch.nonzero(reset_buf)`` and appends their returns / lengths to Python lists — two host
syncs and a device-to-host copy every step.  Here the lists are replaced by four running sums
on the device (``_stats``); ``mean_and_log`` reads them once per ``log_interval`` and reports the
same three means.  Buffers, names, return values and the order of the updates are the
reference's (including that every env, the just-reset ones too, accumulates the step's reward
after the reset — see ``phc_episode_update`` in include/phc_b200.h).
"""

from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from . import _cabi
from .env import HumanoidPHC


class PHCPufferEnv:
    def __init__(self, env: HumanoidPHC, num_actions: int = 69, clip_actions: bool = True, log_interval: int = 32,
                 use_amp_obs: bool = False, fused: bool = False):  # fmt: skip
        self.env = env
        self.clip_actions = clip_actions
        self.log_interval = log_interval
        self.use_amp_obs = use_amp_obs
        dev, N = env.device, env.num_envs
        self.device = dev
        # PufferEnvBuffers (:22-36): observations / rewards alias the env's buffers
        self.observations = env.obs_buf
        self.rewards = env.rew_buf
        self.terminals = torch.zeros(N, dtype=torch.bool, device=dev)
        self.truncations = torch.zeros(N, dtype=torch.bool, device=dev)
        self.masks = torch.ones(N, dtype=torch.bool, device=dev)
        self.actions = torch.zeros((N, num_actions), dtype=torch.float32, device=dev)
        self.episode_returns = torch.zeros(N, dtype=torch.float32, device=dev)  # :72
        self.episode_lengths = torch.zeros(N, dtype=torch.int32, device=dev)  # :73
        self.episode_count = 0
        self.raw_rewards = torch.zeros(env.reward_raw.shape[1], dtype=torch.float32, device=dev)  # :82
        self._stats = torch.zeros(4, dtype=torch.float64, device=dev)
        self._workspace = torch.zeros(16, dtype=torch.float64, device=dev)
        self.amp_obs = None
        self.tick = 0
        # fused=True: the bookkeeping below is done by the env's step kernel (PhcStepArgs.ep_*), one launch fewer per
        # step; the sums collect in per-block accumulators that mean_and_log folds
        self.fused = bool(fused)
        # one accumulator row per block of the step kernel (4 envs): fp64 atomics on one 128-byte line serialise in L2,
        # and with 32 rows the 9 sums of 32 blocks each queued on one line at the tail of every step
        buckets = max(32, min(4096, (N + 3) // 4))
        self._ep_sums = torch.zeros((buckets, _cabi.EPISODE_SUM_COLS), dtype=torch.float64, device=dev) if fused else None
        self._rew = torch.zeros(N, dtype=torch.float32, device=dev)  # `rew = self.rewards.clone()` lives here when fused
        if fused:
            env.set_episode_buffers(dict(terminals=self.terminals, truncations=self.truncations, masks=self.masks,
                                         episode_returns=self.episode_returns, episode_lengths=self.episode_lengths,
                                         sums=self._ep_sums))  # fmt: skip
            env.set_reward_copy(self._rew)
            env.enable_auto_reset(True)

    def _fold(self):
        if self.fused:
            _cabi.check(
                _cabi.load().phc_episode_fold(
                    self._ep_sums.data_ptr(), self._ep_sums.shape[0], self.raw_rewards.shape[0], self.terminals.shape[0],
                    self._stats.data_ptr(), self.raw_rewards.data_ptr(), _cabi.stream_ptr(self.device),
                ),
                "phc_episode_fold",
            )  # fmt: skip

    @property
    def num_agents(self):
        return self.env.num_envs

    def reset(self, seed=None):  # :88-107
        self.tick = 0
        self.env.reset()
        self.rewards[:] = 0
        self.terminals[:] = False
        self.truncations[:] = False
        self.masks[:] = True
        self.actions[:] = 0
        self.raw_rewards[:] = 0
        self._stats.zero_()
        if self.fused:
            self._ep_sums.zero_()
        return self.observations, []

    def update_episodes(self, reset: Optional[torch.Tensor] = None, terminate: Optional[torch.Tensor] = None,
                        rewards: Optional[torch.Tensor] = None, reward_raw: Optional[torch.Tensor] = None):  # fmt: skip
        """:121-159 for one step (the arguments default to the wrapped env's buffers)."""
        reset = self.env.reset_buf if reset is None else reset
        terminate = self.env._terminate_buf if terminate is None else terminate
        rewards = self.rewards if rewards is None else rewards
        reward_raw = self.env.reward_raw if reward_raw is None else reward_raw
        for name, t, dt in (("reset", reset, torch.bool), ("terminate", terminate, torch.bool),
                            ("rewards", rewards, torch.float32), ("reward_raw", reward_raw, torch.float32)):  # fmt: skip
            _cabi.require_cuda(t, name, dt)
        n = self.terminals.shape[0]
        if reset.shape != (n,) or terminate.shape != (n,) or rewards.shape != (n,) or reward_raw.shape[0] != n:
            raise ValueError("episode update: per-env arguments must have num_envs rows")
        if reward_raw.shape[1] != self.raw_rewards.shape[0] or reward_raw.stride(1) != 1:
            raise ValueError("reward_raw must be [num_envs, %d] with unit column stride" % self.raw_rewards.shape[0])
        reset, terminate, rewards = reset.contiguous(), terminate.contiguous(), rewards.contiguous()
        a = _cabi.PhcEpisodeArgs()
        a.reset, a.terminate, a.rewards = reset.data_ptr(), terminate.data_ptr(), rewards.data_ptr()
        a.reward_raw, a.reward_raw_stride, a.reward_raw_cols = reward_raw.data_ptr(), reward_raw.stride(0), reward_raw.shape[1]
        a.terminals, a.truncations, a.masks = self.terminals.data_ptr(), self.truncations.data_ptr(), self.masks.data_ptr()
        a.episode_returns, a.episode_lengths = self.episode_returns.data_ptr(), self.episode_lengths.data_ptr()
        a.stats, a.raw_rewards, a.workspace = self._stats.data_ptr(), self.raw_rewards.data_ptr(), self._workspace.data_ptr()
        _cabi.check(_cabi.load().phc_episode_update(a, n, _cabi.stream_ptr(self.device)), "phc_episode_update")

    def step(self, actions, phase_by_env: Optional[torch.Tensor] = None):
        """:109-183.  ``actions`` may be a numpy array (as pufferlib passes it) or a device tensor."""
        if isinstance(actions, np.ndarray):
            actions = torch.from_numpy(actions).to(self.device, non_blocking=True)
        if self.fused:
            # launch 1, before the physics: clip into self.actions + PD targets (env._pd_target)
            self.env.pre_physics_step(actions.to(torch.float32), clip=1.0 if self.clip_actions else 0.0, actions_out=self.actions)
            # (PhysX steps here in the reference; the owner of the shim writes the post-physics state)
            # launch 2: progress, reward, flags, bookkeeping, reward copy, reset of the flagged envs, observations
            self.env.step(None, phase_by_env)
            self.amp_obs = getattr(self.env, "amp_obs", None) if self.use_amp_obs else None
            rew = self._rew  # rewritten by the next step (the reference returns a fresh clone every step)
        else:
            if self.clip_actions:
                torch.clamp(actions, -1, 1, out=self.actions)
            else:
                self.actions.copy_(actions)
            self.env.step(self.actions)
            self.amp_obs = getattr(self.env, "amp_obs", None) if self.use_amp_obs else None
            rew = self.rewards.clone()
            self.update_episodes()
            self.env.reset_done(phase_by_env)  # :133-135 without the nonzero() sync
        info = []
        self.tick += 1
        if self.tick % self.log_interval == 0:
            info = self.mean_and_log()
        return self.observations, rew, self.terminals, self.truncations, info

    def mean_and_log(self):
        """:191-204 plus the reward terms of :164-176 — the one host read per ``log_interval`` steps."""
        self._fold()
        info, done = episode_info(self._stats, self.raw_rewards, self.log_interval)
        self._stats.zero_()
        self.raw_rewards.zero_()
        self.episode_count += int(done)
        return [info]


def episode_info(stats: torch.Tensor, raw_rewards: torch.Tensor, log_interval: int):
    """The dict of ``mean_and_log`` (:191-204, the reward terms of :164-176) from the folded running sums: ``stats`` f64
    [4] {episodes finished, sum of returns, sum of lengths, truncations} and ``raw_rewards`` f32 (the per-step means of
    the reward terms, summed over ``log_interval`` steps).  Returns ``(info, episodes finished)``."""
    stats = stats.tolist()
    raw = (raw_rewards / log_interval).tolist()
    done = stats[0]
    nan = float("nan")  # np.mean([]) in the reference
    info = {
        "episode_return": stats[1] / done if done else nan,
        "episode_length": stats[2] / done if done else nan,
        "truncated_rate": stats[3] / done if done else nan,
    }
    for k, v in zip(("rew_body_pos", "rew_body_rot", "rew_lin_vel", "rew_ang_vel", "rew_power"), raw):
        info[k] = v
    return info, done
