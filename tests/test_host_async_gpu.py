"""GPU: the asynchronous host step (phc_host_step_submit / phc_host_step_wait, HostStep) equals the device path
(HumanoidPHC.step on the same inputs) bit for bit: obs, reward, reward_raw[:, :4], reset, terminate and the advanced
progress, on every output path, on each slot alone and with both slots in flight over different batches."""

import ctypes as C
import gc

import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from humanoid_b200 import HostStep, HostStepBuffers, HumanoidPHC, MotionLib, _cabi, synth
    from util_gpu import DEV

OK, NULL, SHAPE, UNSUPPORTED, BUSY = 0, -1, -2, -4, -8


def _motion_lib(M=96, seed=501):
    data = synth.make_motion_lib(M, 60, 300, seed=seed, device=DEV)
    return data, MotionLib(data, device=DEV)


class Batch:
    """One env batch: host buffers for the host step, and a HumanoidPHC on the same inputs for the expected outputs."""

    def __init__(self, data, mlib, n, seed, pinned=True, ids="mod", aligned=True):
        clock = synth.make_clock(data, n, seed=seed, ids=ids, aligned=aligned, max_progress=40)
        ref = mlib.get_motion_state(clock.sampled_motion_ids, synth.reward_time(clock, extra_steps=1), clock.global_offset)
        state = synth.make_sim_state(ref, seed=seed + 1)
        self.env = HumanoidPHC(mlib, n, device=DEV)
        self.env.set_sim_state(state)
        self.env.set_clock(clock)
        self.progress0 = clock.progress_buf.cpu()
        b = HostStepBuffers.allocate(n, 1, pinned=pinned)
        b.state.copy_(state.cpu())
        b.progress_buf.copy_(self.progress0)
        b.motion_start_times.copy_(clock.motion_start_times.cpu())
        b.motion_start_times_offset.copy_(clock.motion_start_times_offset.cpu())
        b.global_offset.copy_(clock.global_offset.cpu())
        b.sampled_motion_ids.copy_(clock.sampled_motion_ids.cpu())
        self.bufs = b
        self.n = n
        self.poison()

    def poison(self):
        b = self.bufs
        for t in (b.obs_buf, b.rew_buf, b.reward_raw):
            t.fill_(float("nan"))
        b.reset_buf.fill_(7)
        b.terminate_buf.fill_(7)

    def advance(self):
        """One step of the device path; returns its outputs on the host."""
        e = self.env
        e.step()
        torch.cuda.synchronize()
        return dict(obs=e.obs_buf.cpu(), rew=e.rew_buf.cpu(), raw=e.reward_raw[:, :4].cpu(), reset=e.reset_buf.cpu(),
                    term=e._terminate_buf.cpu(), prog=e.progress_buf.cpu())  # fmt: skip

    def check(self, want, what=""):
        b = self.bufs
        assert torch.equal(b.obs_buf, want["obs"]), f"obs {what}"
        assert torch.equal(b.rew_buf, want["rew"]), f"rew {what}"
        assert torch.equal(b.reward_raw, want["raw"]), f"reward_raw {what}"
        assert torch.equal(b.reset_buf.bool(), want["reset"]) and int(b.reset_buf.max()) <= 1, f"reset {what}"
        assert torch.equal(b.terminate_buf.bool(), want["term"]) and int(b.terminate_buf.max()) <= 1, f"term {what}"
        assert torch.equal(b.progress_buf, want["prog"]), f"progress {what}"


def _ctx(hs):
    return hs._ctx


def _set_path(monkeypatch, mode):
    if mode in ("direct", "staged"):
        monkeypatch.setenv("PHC_HOST_PATH", mode)
    else:
        monkeypatch.delenv("PHC_HOST_PATH", raising=False)
    monkeypatch.delenv("PHC_HOST_STAGED", raising=False)


@pytest.mark.parametrize("slot", [0, 1])
@pytest.mark.parametrize("mode", ["direct", "staged", "pageable"])
def test_each_slot_alone_three_steps_deep(slot, mode, monkeypatch):
    """A ragged batch (not a multiple of 8 envs), three steps with the progress carried in the host buffer."""
    _set_path(monkeypatch, mode)
    data, mlib = _motion_lib()
    bat = Batch(data, mlib, 2005, 11, pinned=mode != "pageable")
    with HostStep(mlib, 2005, num_chunks=3) as hs:
        for i in range(3):
            want = bat.advance()
            bat.poison()
            hs.submit(slot, bat.bufs)
            assert hs.wait(slot) is bat.bufs
            bat.check(want, f"step {i}")
        assert hs.path == (2 if mode == "pageable" else {"direct": 1, "staged": 2}[mode])
        assert hs.chunks == 3


@pytest.mark.parametrize("mode", ["direct", "staged"])
def test_two_slots_in_flight_over_different_batches(mode, monkeypatch):
    """Different sizes, clips and clocks on the two slots; B is waited before A; six rounds.  The first steps of both
    slots follow a phc_lib_pack (the first fused step after a pack runs without speculation)."""
    _set_path(monkeypatch, mode)
    data, mlib = _motion_lib()
    a = Batch(data, mlib, 3001, 21)
    b = Batch(data, mlib, 5003, 31, ids="random", aligned=False)
    mlib.repack()
    torch.cuda.synchronize()
    with HostStep(mlib, 6000, num_chunks=3) as hs:
        for r in range(6):
            wa, wb = a.advance(), b.advance()
            a.poison(), b.poison()
            hs.submit(0, a.bufs)
            hs.submit(1, b.bufs)
            hs.wait(1)
            hs.wait(0)
            a.check(wa, f"A round {r}")
            b.check(wb, f"B round {r}")


def test_two_persistent_kernel_launches_in_flight(monkeypatch):
    """Staged chunks of >= 10240 envs take the persistent step kernel; with both slots in flight two such launches run
    at once and must draw different tile counters.  Each result equals the device path's."""
    _set_path(monkeypatch, "staged")
    data, mlib = _motion_lib(256, 502)
    a = Batch(data, mlib, 45000, 41)  # three doubling chunks: 11256 / 11256 / 22488 envs
    b = Batch(data, mlib, 41000, 51, ids="random")
    with HostStep(mlib, 45000, num_chunks=3) as hs:
        for r in range(2):
            wa, wb = a.advance(), b.advance()
            a.poison(), b.poison()
            hs.submit(0, a.bufs)
            hs.submit(1, b.bufs)
            hs.wait(0)
            hs.wait(1)
            a.check(wa, f"A round {r}")
            b.check(wb, f"B round {r}")


def test_busy_slot_is_refused_and_the_step_in_flight_finishes(monkeypatch):
    _set_path(monkeypatch, "auto")
    data, mlib = _motion_lib()
    a = Batch(data, mlib, 2005, 61)
    b = Batch(data, mlib, 2005, 71)
    capi = _cabi.load()
    with HostStep(mlib, 2005, num_chunks=3) as hs:
        assert capi.phc_host_step_wait(_ctx(hs), 0) == OK  # idle slot
        assert capi.phc_host_step_wait(_ctx(hs), 1) == OK
        wa, wb = a.advance(), b.advance()
        a.poison(), b.poison()
        args_a, args_b = a.bufs._args(), b.bufs._args()
        assert capi.phc_host_step_submit(_ctx(hs), 0, C.byref(args_a), a.n) == OK
        assert capi.phc_host_step_submit(_ctx(hs), 0, C.byref(args_b), b.n) == BUSY
        assert capi.phc_host_step(_ctx(hs), C.byref(args_b), b.n) == BUSY  # the synchronous call runs on slot 0
        assert capi.phc_host_step_wait(_ctx(hs), 0) == OK
        a.check(wa)
        assert torch.isnan(b.bufs.obs_buf).all() and int(b.bufs.reset_buf.min()) == 7  # nothing was enqueued for B
        # while slot 1 is in flight the synchronous call runs normally
        a.bufs.progress_buf.copy_(a.progress0)
        b.poison()
        assert capi.phc_host_step_submit(_ctx(hs), 1, C.byref(args_b), b.n) == OK
        assert capi.phc_host_step_submit(_ctx(hs), 1, C.byref(args_a), a.n) == BUSY
        a.poison()
        assert capi.phc_host_step(_ctx(hs), C.byref(args_a), a.n) == OK
        a.check(wa, "synchronous call beside slot 1")
        assert capi.phc_host_step_wait(_ctx(hs), 1) == OK
        b.check(wb)
        assert capi.phc_host_step_wait(_ctx(hs), 1) == OK


def test_bad_slot_and_device_pointer_leave_the_slot_idle(monkeypatch):
    _set_path(monkeypatch, "direct")
    data, mlib = _motion_lib()
    a = Batch(data, mlib, 1003, 81)
    capi = _cabi.load()
    with HostStep(mlib, 1003, num_chunks=3) as hs:
        args = a.bufs._args()
        for bad in (-1, 2):
            assert capi.phc_host_step_submit(_ctx(hs), bad, C.byref(args), a.n) == SHAPE
            assert capi.phc_host_step_wait(_ctx(hs), bad) == SHAPE
        assert capi.phc_host_step_submit(_ctx(hs), 0, None, a.n) == NULL
        assert capi.phc_host_step_submit(_ctx(hs), 0, C.byref(args), 1004) == SHAPE  # n > max_envs
        dev_args = a.bufs._args()
        dev_args.state = a.env._rigid_body_state_reshaped.data_ptr()
        for slot in (0, 1):
            assert capi.phc_host_step_submit(_ctx(hs), slot, C.byref(dev_args), a.n) == UNSUPPORTED
            assert capi.phc_host_step_wait(_ctx(hs), slot) == OK
        assert torch.isnan(a.bufs.obs_buf).all()
        for slot in (0, 1):
            a.bufs.progress_buf.copy_(a.progress0)
            want = a.advance() if slot == 0 else want
            a.poison()
            assert capi.phc_host_step_submit(_ctx(hs), slot, C.byref(args), a.n) == OK
            assert capi.phc_host_step_wait(_ctx(hs), slot) == OK
            a.check(want, f"slot {slot}")


def test_destroy_waits_for_both_slots(monkeypatch):
    """Slot 0 on pinned buffers (the kernels post into them), slot 1 on pageable ones (staged: the scalar outputs are
    unpacked when the step is finished).  Destroy returns after both; the buffers then hold the outputs."""
    _set_path(monkeypatch, "direct")
    data, mlib = _motion_lib()
    a = Batch(data, mlib, 4003, 91)
    b = Batch(data, mlib, 2999, 95, pinned=False)
    wa, wb = a.advance(), b.advance()
    a.poison(), b.poison()
    capi = _cabi.load()
    hs = HostStep(mlib, 4003, num_chunks=3)
    args_a, args_b = a.bufs._args(), b.bufs._args()
    assert capi.phc_host_step_submit(_ctx(hs), 0, C.byref(args_a), a.n) == OK
    assert capi.phc_host_step_submit(_ctx(hs), 1, C.byref(args_b), b.n) == OK
    ctx, hs._ctx = hs._ctx, None
    capi.phc_host_step_destroy(ctx)
    a.check(wa, "direct slot")
    b.check(wb, "staged slot")


def test_submit_before_tuning_uses_the_first_candidate_and_tuning_still_settles(monkeypatch):
    _set_path(monkeypatch, "auto")
    data, mlib = _motion_lib()
    a = Batch(data, mlib, 4096, 101)
    b = Batch(data, mlib, 4096, 111)
    want_a, want_b = a.advance(), b.advance()
    with HostStep(mlib, 4096, num_chunks=0) as hs:
        capi = hs._capi
        tuning = capi.phc_host_step_tuning_calls(_ctx(hs))
        assert tuning == 2 + 6 * 5
        # async submits and a synchronous call made while slot 1 is in flight: untimed, on the first candidate
        for r in range(3):
            b.bufs.progress_buf.copy_(b.progress0)
            b.poison()
            hs.submit(1, b.bufs)
            a.bufs.progress_buf.copy_(a.progress0)
            a.poison()
            hs.step(a.bufs)
            hs.wait(1)
            a.check(want_a, f"sync beside slot 1, round {r}")
            b.check(want_b, f"slot 1, round {r}")
            assert hs.path == 0
        # none of those counted: tuning takes its full number of synchronous calls, every one of them right
        for i in range(tuning):
            assert hs.path == 0, f"settled early, after {i} calls"
            a.bufs.progress_buf.copy_(a.progress0)
            a.poison()
            hs.step(a.bufs)
            a.check(want_a, f"tuning call {i}")
        assert hs.path in (1, 2) and hs.chunks in (2, 3, 4, 6)
        b.bufs.progress_buf.copy_(b.progress0)
        b.poison()
        hs.submit(0, b.bufs)
        hs.wait(0)
        b.check(want_b, "after tuning")


def test_host_step_class_matches_and_guards_lifetimes(monkeypatch):
    _set_path(monkeypatch, "direct")
    data, mlib = _motion_lib()
    a = Batch(data, mlib, 3000, 121)
    hs = HostStep(mlib, 3000, num_chunks=3, termination_distances=[0.25] * 24, rwd_specs=a.env.rwd_specs)
    want = a.advance()
    a.poison()
    assert hs.step(a.bufs) is a.bufs
    a.check(want, "step")
    assert hs.path == 1 and hs.chunks == 3  # one candidate: nothing to tune
    assert hs.wait(0) is None and hs.wait(1) is None

    # a submit whose tensors the caller drops before wait: the wrapper holds them
    want2 = a.advance()

    def submit_dropped(slot):
        b = HostStepBuffers(**{k: v.clone().pin_memory() for k, v in vars(a.bufs).items()})
        for t in (b.obs_buf, b.rew_buf):
            t.fill_(float("nan"))
        hs.submit(slot, b)
        return id(b)

    ident = submit_dropped(1)
    gc.collect()
    scratch = [torch.full((3000, 934), 3.0).pin_memory() for _ in range(4)]  # reuse of freed pinned blocks, if any
    back = hs.wait(1)
    assert back is not None and id(back) == ident
    a.bufs, saved = back, a.bufs
    a.check(want2, "dropped buffers")
    a.bufs = saved
    del scratch

    # close with both slots in flight: it waits for them, the buffers hold the outputs
    x = Batch(data, mlib, 3000, 131)
    y = Batch(data, mlib, 2000, 141, pinned=False)
    wx, wy = x.advance(), y.advance()
    x.poison(), y.poison()
    hs.submit(0, x.bufs)
    hs.submit(1, y.bufs)
    hs.close()
    hs.close()
    x.check(wx, "close, slot 0")
    y.check(wy, "close, slot 1")
    with pytest.raises(_cabi.PhcError, match="closed"):
        hs.step(x.bufs)
