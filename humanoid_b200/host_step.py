"""Host-buffer step: the fused step on sim state and outputs that live in host memory (include/phc_b200.h,
``phc_host_step*``), for CPU-physics callers and host-side env loops.

``HostStep.step(bufs)`` returns when the outputs are in ``bufs``.  ``submit(slot, bufs)`` / ``wait(slot)`` are the
asynchronous form over two slots: submit a batch, do other work (run the policy on the other batch), collect it.
From ``submit`` until ``wait`` the library writes into the batch's tensors, so the wrapper holds them until then:
a caller that drops its own references cannot free a pinned buffer under a DMA or a posting kernel.

With ``reset=HostResetBuffers`` a step also re-poses the envs it flags (``HumanoidPHC.step()`` with auto-reset), and
``reset_submit`` / ``reset`` re-pose the envs of a mask (``HumanoidPHC.reset(env_ids, phase)``): a host env loop is
``reset`` of every env once, then ``submit(slot, bufs, reset=...)`` / ``wait(slot)`` per batch; after each ``wait`` the
caller's physics takes the root and dof state of the envs in ``bufs.reset_buf`` from the reset buffers.

With ``device_out=HostDeviceOutputs`` the observation rows (and optionally their normalised copy and the RunningNorm
moments) are written into CUDA tensors instead of ``bufs.obs_buf``: the caller whose physics runs on the CPU and whose
policy runs on the GPU gets the rows where the policy reads them, and only rewards, flags, progress and the reset rows
cross back to the host.

The reference's default configuration is available too (``phc_host_step_submit_env``): ``HostStep(...,
use_power_reward=True)`` with ``HostStepBuffers.allocate(..., power=True)`` adds the power reward (the caller's dof force
and velocity go in, ``reward_raw`` has five columns), ``allocate(..., mpjpe=True)`` the eval-mode mpjpe, and
``set_initial_state`` per slot enables ``state_init="default"`` / ``"hybrid"`` (the hybrid mask in
``HostResetBuffers.default_mask``).

Pinned buffers (``HostStepBuffers.allocate(..., pinned=True)``) take the fast paths; pageable ones work through
staging.  The CUDA device of the motion library must be current when the context is created and stepped; after
``MotionLib.repack()`` synchronise the device before the next host step (the steps run on the context's own streams).
"""

from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Any, List, Optional, Sequence, Union

import torch

from . import _cabi
from .env import DEFAULT_REWARD

_FIELDS = (  # name, dtype, trailing shape (T: the number of future steps of the task obs)
    ("state", torch.float32, lambda T: (_cabi.NUM_BODIES, 13)),
    ("progress_buf", torch.int16, lambda T: ()),
    ("motion_start_times", torch.float32, lambda T: ()),
    ("motion_start_times_offset", torch.float32, lambda T: ()),
    ("global_offset", torch.float32, lambda T: (3,)),
    ("sampled_motion_ids", torch.int64, lambda T: ()),
    ("obs_buf", torch.float32, lambda T: (_cabi.SELF_OBS_DIM + _cabi.TASK_OBS_DIM * T,)),
    ("rew_buf", torch.float32, lambda T: ()),
    ("reward_raw", torch.float32, lambda T: (4,)),
    ("reset_buf", torch.uint8, lambda T: ()),
    ("terminate_buf", torch.uint8, lambda T: ()),
)
_DOF = 69
_OPTION_FIELDS = (  # the env options (PhcHostEnvArgs): name, trailing shape
    ("dof_force", (_DOF,)),
    ("dof_vel", (_DOF,)),
    ("mpjpe", ()),
)


@dataclass(eq=False)
class HostStepBuffers:
    """The 11 CPU tensors of one batch of ``n`` envs, in the order of ``PhcHostStepArgs``.  Inputs: ``state``
    [n, 24, 13], the clock (``progress_buf`` int16, advanced in place, ``motion_start_times``,
    ``motion_start_times_offset``, ``global_offset`` [n, 3], ``sampled_motion_ids`` int64).  Outputs: ``obs_buf``
    [n, 358 + 576 T] (None when the rows go to a ``HostDeviceOutputs``), ``rew_buf``, ``reward_raw`` [n, 4] ([n, 5]
    with the power reward, its term in column 4), ``reset_buf`` / ``terminate_buf`` uint8.

    Env options (attributes, not constructor arguments), None when off: ``dof_force`` / ``dof_vel`` [n, 69] f32 (inputs of the power reward: the physics'
    dof force and the velocity half of its dof state), ``mpjpe`` [n] f32 (output, eval mode's ``extras["mpjpe"]``)."""

    state: torch.Tensor
    progress_buf: torch.Tensor
    motion_start_times: torch.Tensor
    motion_start_times_offset: torch.Tensor
    global_offset: torch.Tensor
    sampled_motion_ids: torch.Tensor
    obs_buf: Optional[torch.Tensor]
    rew_buf: torch.Tensor
    reward_raw: torch.Tensor
    reset_buf: torch.Tensor
    terminate_buf: torch.Tensor
    # the env options are attributes, not constructor fields: set by allocate(power= / mpjpe=) or assigned
    dof_force = None
    dof_vel = None
    mpjpe = None

    @classmethod
    def allocate(cls, n: int, time_steps: int = 1, pinned: bool = True, host_obs: bool = True, power: bool = False,
                 mpjpe: bool = False) -> "HostStepBuffers":  # fmt: skip
        """Zeroed buffers for ``n`` envs; ``pinned`` page-locks them (needs the CUDA driver).  ``host_obs=False``
        leaves ``obs_buf`` None, for steps whose rows go to a ``HostDeviceOutputs``.  ``power`` adds ``dof_force`` /
        ``dof_vel`` and makes ``reward_raw`` [n, 5]; ``mpjpe`` adds ``mpjpe``."""

        def make(dtype, trailing):
            t = torch.zeros((n, *trailing), dtype=dtype)
            return t.pin_memory() if pinned else t

        b = cls(**{name: make(dtype, shape(time_steps)) if host_obs or name != "obs_buf" else None
                   for name, dtype, shape in _FIELDS})  # fmt: skip
        if power:
            b.reward_raw = make(torch.float32, (5,))
            b.dof_force, b.dof_vel = make(torch.float32, (_DOF,)), make(torch.float32, (_DOF,))
        if mpjpe:
            b.mpjpe = make(torch.float32, ())
        return b

    @property
    def n(self) -> int:
        return int(self.state.shape[0])

    def validate(self, time_steps: int = 1, device_out: bool = False, power: bool = False) -> int:
        """Checks device (CPU), dtype, shape and contiguity of every tensor; returns ``n``.  ``obs_buf`` must be None
        when the rows go to device outputs (``device_out``), and a tensor otherwise.  ``power``: the step has the power
        reward, so ``dof_force`` / ``dof_vel`` are required and ``reward_raw`` is [n, 5]; without it they must be None."""
        n = self.n
        if device_out and self.obs_buf is not None:
            raise _cabi.PhcError("obs_buf must be None when the rows go to device outputs")
        if not power and (self.dof_force is not None or self.dof_vel is not None):
            raise _cabi.PhcError("dof_force / dof_vel are given but the step has no power reward (use_power_reward)")
        checks = [(name, dtype, shape(time_steps)) for name, dtype, shape in _FIELDS]
        if power:
            checks[_NAMES.index("reward_raw")] = ("reward_raw", torch.float32, (5,))
            checks += [("dof_force", torch.float32, (_DOF,)), ("dof_vel", torch.float32, (_DOF,))]
        if self.mpjpe is not None:
            checks.append(("mpjpe", torch.float32, ()))
        for name, dtype, shape in checks:
            t = getattr(self, name)
            if device_out and name == "obs_buf":
                continue
            if power and t is None and name in ("dof_force", "dof_vel"):
                raise _cabi.PhcError(f"the power reward needs {name} (HostStepBuffers.allocate(..., power=True))")
            if not isinstance(t, torch.Tensor) or t.device.type != "cpu":
                raise _cabi.PhcError(f"{name} must be a CPU tensor (the host step takes host buffers)")
            if t.dtype != dtype:
                raise _cabi.PhcError(f"{name} must be {dtype}, got {t.dtype}")
            want = (n, *shape)
            if tuple(t.shape) != want:
                raise ValueError(f"{name} has shape {tuple(t.shape)}, expected {want}")
            if not t.is_contiguous():
                raise _cabi.PhcError(f"{name} must be contiguous")
        return n

    def _args(self) -> _cabi.PhcHostStepArgs:
        """The 11 pointers of ``PhcHostStepArgs`` (the env options travel in ``PhcHostEnvArgs``)."""
        return _cabi.PhcHostStepArgs(*[_cabi.ptr(getattr(self, name)) for name in _NAMES])


_NAMES = [name for name, _, _ in _FIELDS]


_RESET_FIELDS = (  # name, dtype, trailing shape
    ("phase", torch.float32, ()),
    ("root_states", torch.float32, (13,)),
    ("dof_pos", torch.float32, (69,)),
    ("dof_vel", torch.float32, (69,)),
)
_STATE_INIT = {"start": _cabi.STATE_INIT_START, "random": _cabi.STATE_INIT_RANDOM,
               "default": _cabi.STATE_INIT_DEFAULT, "hybrid": _cabi.STATE_INIT_HYBRID}  # fmt: skip


@dataclass(eq=False)
class HostResetBuffers:
    """The CPU tensors a reset on the host path reads and writes besides a ``HostStepBuffers``.  Input: ``phase`` [n]
    f32, the uniform [0, 1) numbers of ``sample_time_interval`` (state init "random"), and for ``reset_submit`` the
    ``env_mask`` [n] (uint8 or bool, 1 = reset the env).  Outputs, written for the re-posed envs only:
    ``root_states`` [n, 13] (pos 3 | rot 4 | vel 3 | ang vel 3) and ``dof_pos`` / ``dof_vel`` [n, 69] — what the
    caller's physics sets for those envs.  The rigid-body rows and the new clock go into the ``HostStepBuffers``'
    own ``state`` and clock tensors.  ``default_mask`` [n] (uint8 or bool): state init "hybrid", 1 = the env takes the
    default path (the reference draws it with ``torch.bernoulli``; the caller supplies it, like ``phase``)."""

    phase: torch.Tensor
    root_states: torch.Tensor
    dof_pos: torch.Tensor
    dof_vel: torch.Tensor
    env_mask: Optional[torch.Tensor] = None
    default_mask: Optional[torch.Tensor] = None

    @classmethod
    def allocate(cls, n: int, pinned: bool = True, hybrid: bool = False) -> "HostResetBuffers":
        """Zeroed buffers for ``n`` envs (with a zeroed ``env_mask``); ``pinned`` page-locks them; ``hybrid`` adds a
        zeroed ``default_mask``."""

        def make(dtype, trailing):
            t = torch.zeros((n, *trailing), dtype=dtype)
            return t.pin_memory() if pinned else t

        return cls(**{name: make(dtype, shape) for name, dtype, shape in _RESET_FIELDS}, env_mask=make(torch.uint8, ()),
                   default_mask=make(torch.uint8, ()) if hybrid else None)  # fmt: skip

    @property
    def n(self) -> int:
        return int(self.phase.shape[0])

    def validate(self, n: Optional[int] = None) -> int:
        """Checks device (CPU), dtype, shape and contiguity of every tensor (``n`` rows: the batch's); returns ``n``."""
        n = self.n if n is None else int(n)
        fields_ = [(name, (dtype,), shape) for name, dtype, shape in _RESET_FIELDS]
        for name in ("env_mask", "default_mask"):
            if getattr(self, name) is not None:
                fields_.append((name, (torch.uint8, torch.bool), ()))
        for name, dtypes, shape in fields_:
            t = getattr(self, name)
            if not isinstance(t, torch.Tensor) or t.device.type != "cpu":
                raise _cabi.PhcError(f"{name} must be a CPU tensor (the host step takes host buffers)")
            if t.dtype not in dtypes:
                raise _cabi.PhcError(f"{name} must be {' or '.join(map(str, dtypes))}, got {t.dtype}")
            if tuple(t.shape) != (n, *shape):
                raise ValueError(f"{name} has shape {tuple(t.shape)}, expected {(n, *shape)}")
            if not t.is_contiguous():
                raise _cabi.PhcError(f"{name} must be contiguous")
        return n

    def _args(self, bufs: HostStepBuffers, state_init: str, flag_test: bool) -> _cabi.PhcHostResetArgs:
        """The reset's outputs alias ``bufs``' own state and clock tensors."""
        if state_init not in _STATE_INIT:
            raise ValueError(f"state_init must be one of {sorted(_STATE_INIT)}, got {state_init!r}")
        return _cabi.PhcHostResetArgs(
            self.phase.data_ptr(), _cabi.ptr(self.env_mask), _STATE_INIT[state_init], int(bool(flag_test)),
            bufs.state.data_ptr(), self.root_states.data_ptr(), self.dof_pos.data_ptr(), self.dof_vel.data_ptr(),
            bufs.motion_start_times.data_ptr(), bufs.motion_start_times_offset.data_ptr(), bufs.global_offset.data_ptr(),
        )  # fmt: skip


@dataclass(eq=False)
class HostDeviceOutputs:
    """The CUDA tensors a host step writes its rows into instead of ``HostStepBuffers.obs_buf``
    (``phc_host_step_submit_device`` / ``phc_host_reset_submit_device``).

    ``obs`` [n, 358 + 576 T] fp32: the rows ``HumanoidPHC.obs_buf`` would hold.  ``obs_norm`` (optional, fp32 or bf16,
    the same shape): ``clamp((obs - running_mean) / sqrt(running_var + epsilon), -clip, clip)`` of ``normalizer`` (a
    ``RunningNorm``, the object ``HumanoidPHC.set_obs_normalizer`` takes; its buffers are read when the kernels run).
    ``obs_moments`` (optional, fp64 [B, 2 (358 + 576 T)]): per-column sums and sums of squares of every row written
    (+=), spread over B buckets; ``take_obs_moments`` folds them, as ``HumanoidPHC.take_obs_moments`` does.  ``rows``
    counts the rows the moments hold."""

    obs: torch.Tensor
    obs_norm: Optional[torch.Tensor] = None
    normalizer: Optional[Any] = None
    obs_moments: Optional[torch.Tensor] = None
    rows: int = 0

    @classmethod
    def allocate(cls, n: int, time_steps: int = 1, device=None, norm_dtype: Optional[torch.dtype] = None,
                 normalizer=None, moments: bool = False) -> "HostDeviceOutputs":  # fmt: skip
        """Zeroed tensors for ``n`` envs on ``device`` (default: the current CUDA device); ``norm_dtype`` (float32 or
        bfloat16) adds ``obs_norm`` for ``normalizer``; ``moments`` adds 32 buckets of moments."""
        from .env import OBS_MOMENT_BUCKETS

        device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        D = _cabi.SELF_OBS_DIM + _cabi.TASK_OBS_DIM * int(time_steps)
        if norm_dtype is not None and normalizer is None:
            raise ValueError("obs_norm needs the normalizer whose running_mean / running_var it uses")
        return cls(
            obs=torch.zeros((n, D), dtype=torch.float32, device=device),
            obs_norm=None if norm_dtype is None else torch.zeros((n, D), dtype=norm_dtype, device=device),
            normalizer=normalizer,
            obs_moments=torch.zeros((OBS_MOMENT_BUCKETS, 2 * D), dtype=torch.float64, device=device) if moments else None,
        )  # fmt: skip

    def validate(self, n: int, time_steps: int = 1) -> None:
        """Checks dtype, shape and contiguity of every tensor, that all live on one CUDA device, and that ``obs_norm``
        comes with its normaliser."""
        D = _cabi.SELF_OBS_DIM + _cabi.TASK_OBS_DIM * int(time_steps)
        checks = [("obs", self.obs, (torch.float32,), (n, D))]
        if self.obs_norm is not None:
            rn = self.normalizer
            if rn is None:
                raise _cabi.PhcError("obs_norm needs the normalizer whose running_mean / running_var it uses")
            checks.append(("obs_norm", self.obs_norm, (torch.float32, torch.bfloat16), (n, D)))
            for name in ("running_mean", "running_var"):  # [D] or RunningNorm's [1, D]
                checks.append((f"normalizer.{name}", getattr(rn, name, None), (torch.float32,), (D,)))
            if not float(rn.clip) > 0.0:
                raise ValueError(f"normalizer.clip must be > 0, got {rn.clip}")
        if self.obs_moments is not None:
            m = self.obs_moments
            B = int(m.shape[0]) if isinstance(m, torch.Tensor) and m.dim() == 2 else -1
            if not 1 <= B <= 4096:
                raise ValueError(f"obs_moments must be [B, {2 * D}] with 1 <= B <= 4096")
            checks.append(("obs_moments", m, (torch.float64,), (B, 2 * D)))
        dev = self.obs.device if isinstance(self.obs, torch.Tensor) else None
        for name, t, dtypes, shape in checks:
            if not isinstance(t, torch.Tensor):
                raise _cabi.PhcError(f"{name} must be a CUDA tensor")
            if t.dtype not in dtypes:
                raise _cabi.PhcError(f"{name} must be {' or '.join(map(str, dtypes))}, got {t.dtype}")
            got = (t.numel(),) if name.startswith("normalizer") else tuple(t.shape)
            if got != shape:
                raise ValueError(f"{name} has shape {tuple(t.shape)}, expected {shape}")
            if not t.is_contiguous():
                raise _cabi.PhcError(f"{name} must be contiguous")
        for name, t, _, _ in checks:
            if t.device.type != "cuda" or t.device != dev:
                raise _cabi.PhcError(f"{name} must be a CUDA tensor on the device of obs (got {t.device})")

    def take_obs_moments(self, sums: Optional[torch.Tensor] = None):
        """Fold the buckets into ``sums`` (+=, allocated when omitted), zero them, and return ``(sums, rows)`` — what
        ``RunningNorm.update_from_moments`` takes.  Call it after ``wait``: the fold runs on the current stream."""
        b = self.obs_moments
        if b is None:
            raise _cabi.PhcError("these device outputs have no obs_moments")
        if sums is None:
            sums = torch.zeros(b.shape[1], dtype=torch.float64, device=b.device)
        _cabi.check(
            _cabi.load().phc_obs_moments_fold(b.data_ptr(), b.shape[0], b.shape[1], sums.data_ptr(), _cabi.stream_ptr(b.device)),
            "phc_obs_moments_fold",
        )  # fmt: skip
        rows, self.rows = self.rows, 0
        return sums, rows

    def _args(self) -> _cabi.PhcHostDeviceOut:
        a = _cabi.PhcHostDeviceOut()
        a.obs = self.obs.data_ptr()
        if self.obs_norm is not None:
            rn = self.normalizer
            a.obs_norm = self.obs_norm.data_ptr()
            a.norm_mean, a.norm_var = rn.running_mean.data_ptr(), rn.running_var.data_ptr()
            a.norm_epsilon, a.norm_clip = float(rn.epsilon), float(rn.clip)
            a.flags = _cabi.STEP_OBS_NORM_BF16 if self.obs_norm.dtype == torch.bfloat16 else 0
        if self.obs_moments is not None:
            a.obs_moments = self.obs_moments.data_ptr()
            a.obs_moments_buckets = self.obs_moments.shape[0]
        a.stream = _cabi.stream_ptr(self.obs.device)
        return a


class HostStep:
    """A ``phc_host_step`` context on the current CUDA device for batches of up to ``max_envs`` envs.

    ``num_chunks = 0`` lets the context tune its schedule (output path, chunk count) over its first synchronous
    ``step`` calls; ``path`` / ``chunks`` report the result (0 while undecided).  ``submit`` before that uses the
    first candidate.  One thread drives a context.

    ``use_power_reward`` adds ``-rew_power_coef * sum |dof_force * dof_vel|`` (0 while progress <= 3) to every step's
    reward, as ``reward_raw[:, 4]``; every step then needs ``HostStepBuffers.allocate(..., power=True)``."""

    def __init__(
        self,
        lib,
        max_envs: int,
        time_steps: int = 1,
        num_chunks: int = 0,
        termination_distances: Union[float, Sequence[float], torch.Tensor] = 0.25,  # config.py:100
        reset_body_mask: int = 0xFFFFFF,
        use_mean: bool = False,
        enable_early_termination: bool = True,
        dt: float = 2 * (1.0 / 60.0),
        rwd_specs: Optional[dict] = None,
        use_power_reward: bool = False,  # config.py:50 (True in the reference)
        rew_power_coef: float = 0.0005,  # config.py:112
    ):
        self._ctx = None
        self.use_power_reward = bool(use_power_reward)
        self.rew_power_coef = float(rew_power_coef)
        self._initial_rows: List[Optional[int]] = [None] * _cabi.HOST_SLOTS
        self._inflight: List[Optional[HostStepBuffers]] = [None] * _cabi.HOST_SLOTS
        self._inflight_reset: List[Optional[HostResetBuffers]] = [None] * _cabi.HOST_SLOTS
        self._inflight_dev: List[Optional[HostDeviceOutputs]] = [None] * _cabi.HOST_SLOTS
        self.time_steps = int(time_steps)
        self._capi = _cabi.load()
        term = torch.as_tensor(termination_distances, dtype=torch.float32).cpu().expand(_cabi.NUM_BODIES)
        term_host = (C.c_float * _cabi.NUM_BODIES)(*term.tolist())
        spec = _cabi.reward_spec(rwd_specs or DEFAULT_REWARD)
        ctx = C.c_void_p()
        _cabi.check(
            self._capi.phc_host_step_create(
                lib.handle, int(max_envs), self.time_steps, int(num_chunks), term_host, int(reset_body_mask),
                int(bool(use_mean)), int(bool(enable_early_termination)), float(dt), C.byref(spec), C.byref(ctx),
            ),
            "phc_host_step_create",
        )  # fmt: skip
        self._ctx = ctx
        self._lib = lib  # the context borrows the motion library

    def _live(self):
        if self._ctx is None:
            raise _cabi.PhcError("HostStep is closed")
        return self._ctx

    def step(self, bufs: HostStepBuffers, reset: Optional[HostResetBuffers] = None, state_init: str = "random",
             flag_test: bool = False, device_out: Optional[HostDeviceOutputs] = None) -> HostStepBuffers:  # fmt: skip
        """One step of ``bufs``; returns when every output is in ``bufs`` (``progress_buf`` advanced in place) and in
        ``device_out``.  With ``reset`` the envs the step flags are re-posed as well (see ``submit``); with ``reset`` or
        ``device_out`` this runs on slot 0."""
        if reset is not None or device_out is not None or self.use_power_reward or bufs.mpjpe is not None:
            self.submit(0, bufs, reset, state_init, flag_test, device_out=device_out)
            return self.wait(0)
        n = bufs.validate(self.time_steps)
        args = bufs._args()
        _cabi.check(self._capi.phc_host_step(self._live(), C.byref(args), n), "phc_host_step")
        return bufs

    def submit(self, slot: int, bufs: HostStepBuffers, reset: Optional[HostResetBuffers] = None,
               state_init: str = "random", flag_test: bool = False,
               device_out: Optional[HostDeviceOutputs] = None) -> None:  # fmt: skip
        """Enqueue one step of ``bufs`` on ``slot`` (0 or 1) and return.  ``bufs`` (and ``reset``) belong to the library
        until ``wait(slot)`` returns: do not read or write them before then.

        With ``reset`` it is ``HumanoidPHC.step()`` with auto-reset: the envs the step flags are re-posed from the
        motion library (``state_init`` "random": at ``reset.phase``; "start": at time 0; ``flag_test``: the eval
        mode's time 0).  After ``wait``, ``obs_buf`` holds the final rows, ``reset_buf`` / ``terminate_buf`` the step's
        own flags, ``progress_buf`` is 0 for re-posed envs, and for those envs only ``bufs.state``, the clock tensors
        and ``reset.root_states`` / ``dof_pos`` / ``dof_vel`` hold the new state.

        With ``device_out`` (``bufs.obs_buf`` None) the rows go to ``device_out.obs`` (and ``obs_norm`` /
        ``obs_moments``) instead; the kernels writing them wait for the work enqueued so far on the current CUDA
        stream, so the policy may still be reading the previous rows.  The tensors belong to the library until
        ``wait(slot)`` returns.

        With the power reward (``use_power_reward``) or ``bufs.mpjpe``, or ``state_init`` "default" / "hybrid" (after
        ``set_initial_state(slot, ...)``; "hybrid" takes ``reset.default_mask`` and ``reset.phase``), this is
        ``phc_host_step_submit_env``."""
        n = bufs.validate(self.time_steps, device_out=device_out is not None, power=self.use_power_reward)
        args = bufs._args()
        env = self._env_args(slot, bufs, reset, state_init, n)
        if env is not None:
            rargs = None
            if reset is not None:
                reset.validate(n)
                rargs = C.byref(reset._args(bufs, state_init, flag_test))
            dargs = None
            if device_out is not None:
                device_out.validate(n, self.time_steps)
                dargs = C.byref(device_out._args())
            _cabi.check(self._capi.phc_host_step_submit_env(self._live(), int(slot), C.byref(args), rargs, dargs,
                                                            C.byref(env), n), "phc_host_step_submit_env")  # fmt: skip
            if device_out is not None and device_out.obs_moments is not None:
                device_out.rows += n
        elif device_out is not None:
            device_out.validate(n, self.time_steps)
            rargs = None
            if reset is not None:
                reset.validate(n)
                rargs = C.byref(reset._args(bufs, state_init, flag_test))
            dargs = device_out._args()
            _cabi.check(self._capi.phc_host_step_submit_device(self._live(), int(slot), C.byref(args), rargs,
                                                               C.byref(dargs), n), "phc_host_step_submit_device")  # fmt: skip
            if device_out.obs_moments is not None:
                device_out.rows += n  # an auto-reset replaces counted rows and adds none
        elif reset is None:
            _cabi.check(self._capi.phc_host_step_submit(self._live(), int(slot), C.byref(args), n), "phc_host_step_submit")
        else:
            reset.validate(n)
            rargs = reset._args(bufs, state_init, flag_test)
            _cabi.check(self._capi.phc_host_step_submit_reset(self._live(), int(slot), C.byref(args), C.byref(rargs), n),
                        "phc_host_step_submit_reset")  # fmt: skip
        self._hold(slot, bufs, reset, device_out)

    def _env_args(self, slot, bufs: HostStepBuffers, reset: Optional[HostResetBuffers], state_init: str,
                  n: int, step: bool = True) -> Optional[_cabi.PhcHostEnvArgs]:  # fmt: skip
        """The env options of one submit, or None when it has none (the submits without options then run)."""
        power = step and self.use_power_reward
        mpjpe = step and bufs.mpjpe is not None
        init = reset is not None and state_init in ("default", "hybrid")
        if not (power or mpjpe or init):
            return None
        e = _cabi.PhcHostEnvArgs()
        if power:
            e.dof_force, e.dof_vel = bufs.dof_force.data_ptr(), bufs.dof_vel.data_ptr()
            e.rew_power_coef = self.rew_power_coef
        if mpjpe:
            e.mpjpe = bufs.mpjpe.data_ptr()
        if init:
            if not 0 <= slot < _cabi.HOST_SLOTS or self._initial_rows[slot] is None:
                raise _cabi.PhcError(f"state_init {state_init!r} is not supported on slot {slot} before "
                                     "set_initial_state(slot, ...) has given it the initial state")  # fmt: skip
            if state_init == "hybrid":
                if reset.default_mask is None:
                    raise ValueError('state_init "hybrid" needs reset.default_mask (HostResetBuffers.allocate(..., hybrid=True))')
                e.default_mask = reset.default_mask.data_ptr()
        return e

    def set_initial_state(self, slot: int, root_states: torch.Tensor, dof_pos: torch.Tensor,
                          dof_vel: torch.Tensor) -> None:  # fmt: skip
        """The reference's ``_initial_humanoid_root_states`` [n, 13] and ``_initial_dof_pos`` / ``_initial_dof_vel``
        [n, 69] (f32 CPU tensors) of the envs submitted on ``slot``: row i is env i of every batch on that slot.  Copied
        once, synchronously, to the device; the tensors may be freed afterwards.  Needed for state init "default" /
        "hybrid"; the slot must be idle."""
        n = None
        for name, t, width in (("root_states", root_states, 13), ("dof_pos", dof_pos, _DOF), ("dof_vel", dof_vel, _DOF)):
            if not isinstance(t, torch.Tensor) or t.device.type != "cpu":
                raise _cabi.PhcError(f"{name} must be a CPU tensor (the host step takes host buffers)")
            if t.dtype != torch.float32:
                raise _cabi.PhcError(f"{name} must be torch.float32, got {t.dtype}")
            n = int(t.shape[0]) if n is None and t.dim() == 2 else n
            if t.dim() != 2 or tuple(t.shape) != (n, width):
                raise ValueError(f"{name} has shape {tuple(t.shape)}, expected {(n, width)}")
            if not t.is_contiguous():
                raise _cabi.PhcError(f"{name} must be contiguous")
        _cabi.check(self._capi.phc_host_step_set_initial_state(self._live(), int(slot), root_states.data_ptr(),
                                                               dof_pos.data_ptr(), dof_vel.data_ptr(), n),
                    "phc_host_step_set_initial_state")  # fmt: skip
        self._initial_rows[slot] = n

    def _hold(self, slot, bufs, reset, device_out):
        """Keep a batch's tensors alive until its ``wait``."""
        self._inflight[slot] = bufs
        self._inflight_reset[slot] = reset
        self._inflight_dev[slot] = device_out

    def reset_submit(self, slot: int, bufs: HostStepBuffers, reset: HostResetBuffers, state_init: str = "random",
                     flag_test: bool = False, device_out: Optional[HostDeviceOutputs] = None) -> None:  # fmt: skip
        """Enqueue ``HumanoidPHC.reset(env_ids, phase)`` for the envs of ``reset.env_mask`` on ``slot`` and return:
        reads the clock and ids of ``bufs``; after ``wait``, for the masked envs only, ``obs_buf`` rows, ``state``,
        the clock, ``progress_buf`` = 0, ``reset_buf`` = ``terminate_buf`` = 0 and ``reset``'s root / dof rows hold
        the re-posed envs.  How a host loop gets its first observation.  With ``device_out`` the masked envs' rows go
        to ``device_out.obs`` / ``obs_norm`` and are added to ``obs_moments`` (rows no step has counted).  State init
        "default" / "hybrid" as in ``submit`` (``phc_host_reset_submit_env``); the power inputs are not read."""
        n = bufs.validate(self.time_steps, device_out=device_out is not None, power=self.use_power_reward)
        reset.validate(n)
        if reset.env_mask is None:
            raise ValueError("reset_submit needs reset.env_mask")
        args, rargs = bufs._args(), reset._args(bufs, state_init, flag_test)
        env = self._env_args(slot, bufs, reset, state_init, n, step=False)
        if env is not None:
            dargs = None
            if device_out is not None:
                device_out.validate(n, self.time_steps)
                dargs = C.byref(device_out._args())
            _cabi.check(self._capi.phc_host_reset_submit_env(self._live(), int(slot), C.byref(args), C.byref(rargs),
                                                             dargs, C.byref(env), n), "phc_host_reset_submit_env")  # fmt: skip
            if device_out is not None and device_out.obs_moments is not None:
                device_out.rows += int(reset.env_mask.count_nonzero())
        elif device_out is None:
            _cabi.check(self._capi.phc_host_reset_submit(self._live(), int(slot), C.byref(args), C.byref(rargs), n),
                        "phc_host_reset_submit")  # fmt: skip
        else:
            device_out.validate(n, self.time_steps)
            dargs = device_out._args()
            _cabi.check(self._capi.phc_host_reset_submit_device(self._live(), int(slot), C.byref(args), C.byref(rargs),
                                                                C.byref(dargs), n), "phc_host_reset_submit_device")  # fmt: skip
            if device_out.obs_moments is not None:
                device_out.rows += int(reset.env_mask.count_nonzero())
        self._hold(slot, bufs, reset, device_out)

    def reset(self, bufs: HostStepBuffers, reset: HostResetBuffers, state_init: str = "random",
              flag_test: bool = False, device_out: Optional[HostDeviceOutputs] = None) -> HostStepBuffers:  # fmt: skip
        """``reset_submit`` on slot 0 + ``wait(0)``."""
        self.reset_submit(0, bufs, reset, state_init, flag_test, device_out)
        return self.wait(0)

    def wait(self, slot: int) -> Optional[HostStepBuffers]:
        """Block until ``slot``'s step has finished; returns its buffers (None if the slot was idle)."""
        rc = self._capi.phc_host_step_wait(self._live(), int(slot))
        bufs = None
        if 0 <= slot < _cabi.HOST_SLOTS:  # the slot is idle after wait, also when it reports an error
            bufs = self._inflight[slot]
            self._hold(slot, None, None, None)
        _cabi.check(rc, "phc_host_step_wait")
        return bufs

    @property
    def path(self) -> int:
        """1 = direct (kernels post into the pinned host buffers), 2 = staged (copy-engine D2H), 0 = undecided."""
        return int(self._capi.phc_host_step_path(self._live()))

    @property
    def chunks(self) -> int:
        return int(self._capi.phc_host_step_chunks(self._live()))

    def close(self) -> None:
        """Wait for both slots, then free the context.  Idempotent."""
        ctx, self._ctx = self._ctx, None
        if ctx is not None:
            self._capi.phc_host_step_destroy(ctx)  # finishes every slot in flight before freeing
        self._inflight = [None] * _cabi.HOST_SLOTS
        self._inflight_reset = [None] * _cabi.HOST_SLOTS
        self._inflight_dev = [None] * _cabi.HOST_SLOTS

    def __enter__(self) -> "HostStep":
        return self

    def __exit__(self, *exc) -> None:
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
