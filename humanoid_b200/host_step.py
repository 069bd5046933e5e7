"""Host-buffer step: the fused step on sim state and outputs that live in host memory (include/phc_b200.h,
``phc_host_step*``), for CPU-physics callers and host-side env loops.

``HostStep.step(bufs)`` returns when the outputs are in ``bufs``.  ``submit(slot, bufs)`` / ``wait(slot)`` are the
asynchronous form over two slots: submit a batch, do other work (run the policy on the other batch), collect it.
From ``submit`` until ``wait`` the library writes into the batch's tensors, so the wrapper holds them until then:
a caller that drops its own references cannot free a pinned buffer under a DMA or a posting kernel.

Pinned buffers (``HostStepBuffers.allocate(..., pinned=True)``) take the fast paths; pageable ones work through
staging.  The CUDA device of the motion library must be current when the context is created and stepped; after
``MotionLib.repack()`` synchronise the device before the next host step (the steps run on the context's own streams).
"""

from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, fields
from typing import List, Optional, Sequence, Union

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


@dataclass(eq=False)
class HostStepBuffers:
    """The 11 CPU tensors of one batch of ``n`` envs, in the order of ``PhcHostStepArgs``.  Inputs: ``state``
    [n, 24, 13], the clock (``progress_buf`` int16, advanced in place, ``motion_start_times``,
    ``motion_start_times_offset``, ``global_offset`` [n, 3], ``sampled_motion_ids`` int64).  Outputs: ``obs_buf``
    [n, 358 + 576 T], ``rew_buf``, ``reward_raw`` [n, 4], ``reset_buf`` / ``terminate_buf`` uint8."""

    state: torch.Tensor
    progress_buf: torch.Tensor
    motion_start_times: torch.Tensor
    motion_start_times_offset: torch.Tensor
    global_offset: torch.Tensor
    sampled_motion_ids: torch.Tensor
    obs_buf: torch.Tensor
    rew_buf: torch.Tensor
    reward_raw: torch.Tensor
    reset_buf: torch.Tensor
    terminate_buf: torch.Tensor

    @classmethod
    def allocate(cls, n: int, time_steps: int = 1, pinned: bool = True) -> "HostStepBuffers":
        """Zeroed buffers for ``n`` envs; ``pinned`` page-locks them (needs the CUDA driver)."""

        def make(dtype, trailing):
            t = torch.zeros((n, *trailing), dtype=dtype)
            return t.pin_memory() if pinned else t

        return cls(**{name: make(dtype, shape(time_steps)) for name, dtype, shape in _FIELDS})

    @property
    def n(self) -> int:
        return int(self.state.shape[0])

    def validate(self, time_steps: int = 1) -> int:
        """Checks device (CPU), dtype, shape and contiguity of every tensor; returns ``n``."""
        n = self.n
        for name, dtype, shape in _FIELDS:
            t = getattr(self, name)
            if not isinstance(t, torch.Tensor) or t.device.type != "cpu":
                raise _cabi.PhcError(f"{name} must be a CPU tensor (the host step takes host buffers)")
            if t.dtype != dtype:
                raise _cabi.PhcError(f"{name} must be {dtype}, got {t.dtype}")
            want = (n, *shape(time_steps))
            if tuple(t.shape) != want:
                raise ValueError(f"{name} has shape {tuple(t.shape)}, expected {want}")
            if not t.is_contiguous():
                raise _cabi.PhcError(f"{name} must be contiguous")
        return n

    def _args(self) -> _cabi.PhcHostStepArgs:
        return _cabi.PhcHostStepArgs(*[getattr(self, f.name).data_ptr() for f in fields(self)])


class HostStep:
    """A ``phc_host_step`` context on the current CUDA device for batches of up to ``max_envs`` envs.

    ``num_chunks = 0`` lets the context tune its schedule (output path, chunk count) over its first synchronous
    ``step`` calls; ``path`` / ``chunks`` report the result (0 while undecided).  ``submit`` before that uses the
    first candidate.  One thread drives a context."""

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
    ):
        self._ctx = None
        self._inflight: List[Optional[HostStepBuffers]] = [None] * _cabi.HOST_SLOTS
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

    def step(self, bufs: HostStepBuffers) -> HostStepBuffers:
        """One step of ``bufs``; returns when every output is in ``bufs`` (``progress_buf`` advanced in place)."""
        n = bufs.validate(self.time_steps)
        args = bufs._args()
        _cabi.check(self._capi.phc_host_step(self._live(), C.byref(args), n), "phc_host_step")
        return bufs

    def submit(self, slot: int, bufs: HostStepBuffers) -> None:
        """Enqueue one step of ``bufs`` on ``slot`` (0 or 1) and return.  ``bufs`` belongs to the library until
        ``wait(slot)`` returns: do not read or write it before then."""
        n = bufs.validate(self.time_steps)
        args = bufs._args()
        _cabi.check(self._capi.phc_host_step_submit(self._live(), int(slot), C.byref(args), n), "phc_host_step_submit")
        self._inflight[slot] = bufs

    def wait(self, slot: int) -> Optional[HostStepBuffers]:
        """Block until ``slot``'s step has finished; returns its buffers (None if the slot was idle)."""
        rc = self._capi.phc_host_step_wait(self._live(), int(slot))
        bufs = None
        if 0 <= slot < _cabi.HOST_SLOTS:  # the slot is idle after wait, also when it reports an error
            bufs, self._inflight[slot] = self._inflight[slot], None
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

    def __enter__(self) -> "HostStep":
        return self

    def __exit__(self, *exc) -> None:
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
