"""GPU: the host step with device outputs equals the device path bit for bit.

``HostStep.submit(slot, bufs, device_out=...)`` (phc_host_step_submit_device) and ``reset_submit(..., device_out=...)``
(phc_host_reset_submit_device) against ``HumanoidPHC.step`` / ``HumanoidPHC.reset(env_ids, phase)`` on the same inputs:
the device ``obs`` rows equal ``obs_buf``, ``obs_norm`` equals ``obs_norm_buf`` of ``set_obs_normalizer(rn, dtype)``,
and rewards, reward_raw[:, :4], flags, progress and the reset rows on the host are as on the device path.  The folded
moments equal the fp64 column sums and sums of squares of every row written.  Short clips and clocks near clip ends,
so that every auto-reset step flags envs by clip end and by termination; a few envs are pushed away from their
reference each step (the stand-in for physics)."""

import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from humanoid_b200 import (HostDeviceOutputs, HostResetBuffers, HostStep, HostStepBuffers, HumanoidPHC, MotionLib,
                               RunningNorm, _cabi, synth)  # fmt: skip
    from util_gpu import DEV

OK, NULL, SHAPE, ALIGN, UNSUPPORTED, BUSY = 0, -1, -2, -3, -4, -8
SENTINEL = 12345.0


def _motion_lib(M=48, seed=701):
    data = synth.make_motion_lib(M, 60, 90, seed=seed, device=DEV)
    return data, MotionLib(data, device=DEV)


def _normalizer(D, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    rn = RunningNorm(D, device=DEV)
    rn.running_mean.copy_(torch.randn(1, D, generator=g, device=DEV) * 0.3)
    rn.running_var.copy_(torch.rand(1, D, generator=g, device=DEV) * 2 + 0.05)
    return rn


class Case:
    """One batch on both paths: host inputs and device outputs for the host step, a HumanoidPHC on the same inputs."""

    def __init__(self, data, mlib, n, seed, T=1, pinned=True, pinned_reset=None, auto_reset=False, norm=None,
                 moments=False, ids="mod", aligned=True, state_init="random", eval_mode=False, flag_test=False):  # fmt: skip
        clock = synth.make_clock(data, n, seed=seed, ids=ids, aligned=aligned, max_progress=30)
        ref = mlib.get_motion_state(clock.sampled_motion_ids, synth.reward_time(clock, extra_steps=1), clock.global_offset)
        state = synth.make_sim_state(ref, seed=seed + 1)
        env = HumanoidPHC(mlib, n, device=DEV, time_steps=T, obs_moments=moments)
        env.set_sim_state(state)
        env.set_clock(clock)
        env.enable_auto_reset(auto_reset)
        env.state_init, env.flag_test = state_init, flag_test
        if eval_mode:
            env.flag_im_eval = True
            env.set_termination_distances(0.1)
        D = _cabi.SELF_OBS_DIM + _cabi.TASK_OBS_DIM * T
        self.rn = _normalizer(D, seed + 3) if norm is not None else None
        if norm is not None:
            env.set_obs_normalizer(self.rn, norm)
        self.env, self.n, self.T, self.auto_reset = env, n, T, auto_reset
        self.state_init, self.flag_test = state_init, flag_test
        b = HostStepBuffers.allocate(n, T, pinned=pinned, host_obs=False)
        for name, v in (("state", state), ("progress_buf", clock.progress_buf), ("motion_start_times", clock.motion_start_times),
                        ("motion_start_times_offset", clock.motion_start_times_offset),
                        ("global_offset", clock.global_offset), ("sampled_motion_ids", clock.sampled_motion_ids)):  # fmt: skip
            getattr(b, name).copy_(v.cpu())
        self.bufs = b
        self.rb = HostResetBuffers.allocate(n, pinned=pinned if pinned_reset is None else pinned_reset)
        self.dev = HostDeviceOutputs.allocate(n, T, DEV, norm_dtype=norm, normalizer=self.rn, moments=moments)
        self.want_sums = torch.zeros(2 * D, dtype=torch.float64, device=DEV)
        self.abs_sums = torch.zeros(D, dtype=torch.float64, device=DEV)  # error bound of the reordered sums
        self.gen = torch.Generator().manual_seed(seed + 2)
        self.k = 0

    def kw(self):
        return dict(state_init=self.state_init, flag_test=self.flag_test)

    def poison(self):
        b, r, d = self.bufs, self.rb, self.dev
        for t in (b.rew_buf, b.reward_raw):
            t.fill_(float("nan"))
        b.reset_buf.fill_(7)
        b.terminate_buf.fill_(7)
        for t in (r.root_states, r.dof_pos, r.dof_vel, d.obs):
            t.fill_(SENTINEL)
        if d.obs_norm is not None:
            d.obs_norm.fill_(SENTINEL)

    def physics(self):
        """The same push on both paths: ~3 % of the envs move 0.5 m (they terminate), the others a little."""
        n, k = self.n, self.k
        d = torch.randn(n, 24, 3, generator=self.gen) * 0.01
        d[(torch.arange(n) * 7 + k) % 29 == 0, :, 0] += 0.5
        self.bufs.state[..., 0:3] += d
        self.env._rigid_body_state_reshaped[..., 0:3] += d.to(DEV)
        self.k += 1

    def count(self, rows):
        x = rows.double()
        D = x.shape[1]
        self.want_sums[:D] += x.sum(0)
        self.want_sums[D:] += (x * x).sum(0)
        self.abs_sums += x.abs().sum(0)

    def advance(self):
        """Physics, a fresh phase, poisoned outputs, one step of the device path; returns its outputs."""
        self.physics()
        self.rb.phase.copy_(torch.rand(self.n, generator=self.gen))
        self.poison()
        e = self.env
        if self.auto_reset:
            e.step(phase_by_env=self.rb.phase.to(DEV))
            flags = (e.extras["reset"].clone(), e.extras["terminate"].clone())
        else:
            e.step()
            flags = (e.reset_buf.clone(), e._terminate_buf.clone())
        torch.cuda.synchronize()
        self.count(e.obs_buf)
        return self.snapshot(dict(reset=flags[0].cpu(), term=flags[1].cpu()))

    def snapshot(self, out):
        e = self.env
        out.update(obs=e.obs_buf.clone(), rew=e.rew_buf.cpu(), raw=e.reward_raw[:, :4].cpu(), prog=e.progress_buf.cpu(),
                   root=e._humanoid_root_states.cpu(), dofp=e._dof_pos.cpu(), dofv=e._dof_vel.cpu(),
                   norm=None if e.obs_norm_buf is None else e.obs_norm_buf.clone())  # fmt: skip
        return out

    def submit(self, hs, slot):
        hs.submit(slot, self.bufs, self.rb if self.auto_reset else None, device_out=self.dev, **self.kw())

    def check_step(self, want, what=""):
        b, d = self.bufs, self.dev
        f = want["reset"]
        if self.auto_reset:
            assert 0 < int(f.sum()) < self.n, f"the case should flag some envs and spare others {what}"
        assert torch.equal(d.obs, want["obs"]), f"obs {what}"
        if d.obs_norm is not None:
            assert torch.equal(d.obs_norm, want["norm"]), f"obs_norm {what}"
        assert torch.equal(b.rew_buf, want["rew"]), f"rew {what}"
        assert torch.equal(b.reward_raw, want["raw"]), f"reward_raw {what}"
        assert torch.equal(b.reset_buf.bool(), f) and int(b.reset_buf.max()) <= 1, f"reset {what}"
        assert torch.equal(b.terminate_buf.bool(), want["term"]), f"term {what}"
        assert torch.equal(b.progress_buf, want["prog"]), f"progress {what}"
        if self.auto_reset:
            r = self.rb
            for name, got in (("root", r.root_states), ("dofp", r.dof_pos), ("dofv", r.dof_vel)):
                assert torch.equal(got[f], want[name][f]), f"{name} of re-posed envs {what}"
                assert bool((got[~f] == SENTINEL).all()), f"{name} of other envs written {what}"

    def check_moments(self, expect_rows):
        sums, rows = self.dev.take_obs_moments()
        torch.cuda.synchronize()
        assert rows == expect_rows
        D = self.abs_sums.shape[0]
        bound = 1e-12 * torch.cat([self.abs_sums, self.want_sums[D:]]) + 1e-300
        assert bool(((sums - self.want_sums).abs() <= bound).all()), "moments"
        assert float(self.dev.obs_moments.abs().max()) == 0.0  # folded buckets are zeroed
        self.want_sums.zero_()
        self.abs_sums.zero_()


def _set_path(monkeypatch, mode):
    if mode in ("direct", "staged"):
        monkeypatch.setenv("PHC_HOST_PATH", mode)
    else:
        monkeypatch.delenv("PHC_HOST_PATH", raising=False)


def _steps(hs, case, slot, steps, what=""):
    for i in range(steps):
        want = case.advance()
        case.submit(hs, slot)
        assert hs.wait(slot) is case.bufs
        case.check_step(want, f"{what} step {i}")


@pytest.mark.parametrize("slot", [0, 1])
@pytest.mark.parametrize("mode", ["direct", "staged"])
def test_plain_step_each_slot_eight_steps_deep(slot, mode, monkeypatch):
    """direct: pinned scalars posted by the kernels; staged: pageable buffers through the copy engines."""
    _set_path(monkeypatch, mode)
    data, mlib = _motion_lib()
    case = Case(data, mlib, 2005, 11, pinned=mode == "direct")
    with HostStep(mlib, 2005, num_chunks=3) as hs:
        _steps(hs, case, slot, 8, mode)
        assert hs.path == (1 if mode == "direct" else 2)


@pytest.mark.parametrize("mode", ["direct", "staged"])
def test_two_slots_in_flight_waited_out_of_order(mode, monkeypatch):
    _set_path(monkeypatch, mode)
    data, mlib = _motion_lib()
    a = Case(data, mlib, 3001, 21, auto_reset=True)
    b = Case(data, mlib, 5003, 31, ids="random", aligned=False)
    with HostStep(mlib, 6000, num_chunks=3) as hs:
        for r in range(4):
            wa, wb = a.advance(), b.advance()
            a.submit(hs, 0)
            b.submit(hs, 1)
            hs.wait(1)
            hs.wait(0)
            a.check_step(wa, f"A round {r}")
            b.check_step(wb, f"B round {r}")


@pytest.mark.parametrize("variant", ["T3", "generic"])
@pytest.mark.parametrize("mode", ["direct", "staged"])
def test_kernel_variants_with_auto_reset_norm_and_moments(variant, mode, monkeypatch):
    """T = 3 and the generic kernel: the step is followed by a separate reset launch, which must keep the normalised
    rows and the moments consistent with the final rows."""
    _set_path(monkeypatch, mode)
    data, mlib = _motion_lib()
    T = 3 if variant == "T3" else 1
    case = Case(data, mlib, 1003, 41, T=T, auto_reset=True, norm=torch.float32, moments=True)
    capi = _cabi.load()
    if variant == "generic":
        capi.phc_set_option(_cabi.OPT_FORCE_GENERIC_STEP, 1)
    try:
        with HostStep(mlib, 1003, time_steps=T, num_chunks=3) as hs:
            _steps(hs, case, 0, 3, variant)
            case.check_moments(3 * 1003)
    finally:
        capi.phc_set_option(_cabi.OPT_FORCE_GENERIC_STEP, 0)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("mode", ["direct", "staged"])
def test_normaliser(dtype, mode, monkeypatch):
    _set_path(monkeypatch, mode)
    data, mlib = _motion_lib()
    case = Case(data, mlib, 2005, 51, pinned=mode == "direct", norm=dtype)
    with HostStep(mlib, 2005, num_chunks=3) as hs:
        _steps(hs, case, 1, 3, f"norm {dtype}")


@pytest.mark.parametrize("mode", ["direct", "staged"])
def test_moments_of_steps_resets_and_both_slots(mode, monkeypatch):
    """Plain steps on both slots adding into one accumulator, then steps with auto-reset (the final rows are counted),
    then a masked host reset (the new rows are added); fp64 sums equal torch's to the reordering bound."""
    _set_path(monkeypatch, mode)
    data, mlib = _motion_lib()
    n = 2005
    case = Case(data, mlib, n, 61, pinned=mode == "direct", norm=torch.bfloat16, moments=True)
    with HostStep(mlib, n, num_chunks=3) as hs:
        for i in range(4):
            want = case.advance()
            case.submit(hs, i % 2)
            hs.wait(i % 2)
            case.check_step(want, f"plain {i}")
        case.check_moments(4 * n)
        case.auto_reset = True
        case.env.enable_auto_reset(True)
        case.bufs.progress_buf.copy_(case.env.progress_buf.cpu())
        for i in range(3):
            want = case.advance()
            case.submit(hs, 1 - i % 2)
            hs.wait(1 - i % 2)
            case.check_step(want, f"auto-reset {i}")
        case.check_moments(3 * n)
        mask = torch.rand(n, generator=case.gen) < 0.3
        ids = mask.nonzero().squeeze(1)
        case.rb.env_mask.copy_(mask)
        case.poison()
        case.env.reset(ids.to(DEV), case.rb.phase[ids].to(DEV))
        torch.cuda.synchronize()
        case.count(case.env.obs_buf[ids.to(DEV)])
        hs.reset(case.bufs, case.rb, device_out=case.dev)
        case.check_moments(int(mask.sum()))


@pytest.mark.parametrize("variant", ["random", "start", "eval"])
def test_auto_reset_state_init_and_eval_mode(variant, monkeypatch):
    _set_path(monkeypatch, "direct")
    data, mlib = _motion_lib()
    case = Case(data, mlib, 2005, 71, auto_reset=True, state_init="start" if variant == "start" else "random",
                eval_mode=variant == "eval", pinned_reset=variant != "random")  # fmt: skip
    kw = dict(use_mean=True, termination_distances=0.1) if variant == "eval" else {}
    with HostStep(mlib, 2005, num_chunks=3, **kw) as hs:
        _steps(hs, case, 1, 4, variant)


@pytest.mark.parametrize("pinned", [True, False], ids=["pinned", "pageable"])
def test_masked_host_reset(pinned, monkeypatch):
    """Masked envs' obs and normalised rows equal HumanoidPHC.reset(env_ids, phase); other rows keep the sentinel.  The
    pageable case takes the reset rows through the slot's staging (unpacked by wait, with no obs rows)."""
    _set_path(monkeypatch, "direct")
    data, mlib = _motion_lib()
    n = 2005
    case = Case(data, mlib, n, 81, pinned=pinned, norm=torch.bfloat16)
    b, r, d = case.bufs, case.rb, case.dev
    with HostStep(mlib, n, num_chunks=3) as hs:
        case.rb.phase.copy_(torch.rand(n, generator=case.gen))
        mask = torch.rand(n, generator=case.gen) < 0.4
        ids = mask.nonzero().squeeze(1)
        r.env_mask.copy_(mask)
        case.poison()
        prog = b.progress_buf.clone()
        case.env.reset(ids.to(DEV), r.phase[ids].to(DEV))
        torch.cuda.synchronize()
        want = case.snapshot({})
        hs.reset_submit(1, b, r, device_out=d)
        assert hs.wait(1) is b
        m = mask.to(DEV)
        assert torch.equal(d.obs[m], want["obs"][m]) and bool((d.obs[~m] == SENTINEL).all())
        assert torch.equal(d.obs_norm[m], want["norm"][m]) and bool((d.obs_norm[~m] == SENTINEL).all())
        assert int(b.progress_buf[mask].abs().max()) == 0 and torch.equal(b.progress_buf[~mask], prog[~mask])
        assert int(b.reset_buf[mask].max()) == 0 and int(b.reset_buf[~mask].min()) == 7
        for name, got in (("root", r.root_states), ("dofp", r.dof_pos), ("dofv", r.dof_vel)):
            assert torch.equal(got[mask], want[name][mask]), name
            assert bool((got[~mask] == SENTINEL).all()), name


@pytest.mark.parametrize("mode", ["direct", "staged"])
def test_rows_wait_for_the_callers_stream(mode, monkeypatch):
    """A fill of obs enqueued on the current stream behind a long sleep lands before the step's rows: after wait the
    rows are the step's, not the fill's."""
    _set_path(monkeypatch, mode)
    data, mlib = _motion_lib()
    case = Case(data, mlib, 2005, 91, pinned=mode == "direct", norm=torch.float32)
    with HostStep(mlib, 2005, num_chunks=3) as hs:
        for i in range(2):
            want = case.advance()
            torch.cuda._sleep(200_000_000)  # ~0.1 s on the current stream
            case.dev.obs.fill_(-1.0)
            case.dev.obs_norm.fill_(-1.0)
            case.submit(hs, i)
            hs.wait(i)
            case.check_step(want, f"ordered {i}")


def test_error_codes_enqueue_nothing(monkeypatch):
    _set_path(monkeypatch, "direct")
    data, mlib = _motion_lib()
    n = 1003
    case = Case(data, mlib, n, 101, auto_reset=True, norm=torch.float32, moments=True)
    capi = _cabi.load()
    host_rows = torch.zeros(n, 934).pin_memory()
    host_moments = torch.zeros(32, 2 * 934, dtype=torch.float64).pin_memory()
    with HostStep(mlib, n, num_chunks=3) as hs:
        ctx = hs._ctx
        case.poison()
        args = case.bufs._args()
        rargs = case.rb._args(case.bufs, "random", False)
        fns = ((capi.phc_host_step_submit_device, None), (capi.phc_host_step_submit_device, C.byref(rargs)),
               (capi.phc_host_reset_submit_device, C.byref(rargs)))  # fmt: skip

        def bad(**fields):
            d = case.dev._args()
            for k, v in fields.items():
                setattr(d, k, v)
            return d

        cases = [
            (NULL, None), (NULL, bad(obs=None)), (NULL, bad(norm_mean=None)), (NULL, bad(norm_var=None)),
            (UNSUPPORTED, bad(obs=host_rows.data_ptr())), (UNSUPPORTED, bad(obs_moments=host_moments.data_ptr())),
            (UNSUPPORTED, bad(norm_var=host_rows.data_ptr())), (UNSUPPORTED, bad(flags=4)),
            (ALIGN, bad(obs=case.dev.obs.data_ptr() + 4)), (ALIGN, bad(obs_norm=case.dev.obs_norm.data_ptr() + 8)),
            (SHAPE, bad(obs_moments_buckets=4097)), (SHAPE, bad(obs_moments_buckets=-1)), (SHAPE, bad(norm_clip=0.0)),
        ]  # fmt: skip
        for slot in (0, 1):
            for fn, r in fns:
                for code, d in cases:
                    assert fn(ctx, slot, C.byref(args), r, None if d is None else C.byref(d), n) == code, (code, fn)
                host_args = case.bufs._args()
                host_args.obs_buf = host_rows.data_ptr()  # the rows go to one place only
                assert fn(ctx, slot, C.byref(host_args), r, C.byref(case.dev._args()), n) == UNSUPPORTED
                nophase = case.rb._args(case.bufs, "random", False)
                nophase.phase = None
                assert fn(ctx, slot, C.byref(args), C.byref(nophase), C.byref(case.dev._args()), n) == NULL
                assert capi.phc_host_step_wait(ctx, slot) == OK
        torch.cuda.synchronize()
        assert bool((case.dev.obs == SENTINEL).all()) and bool((case.dev.obs_norm == SENTINEL).all())
        assert float(case.dev.obs_moments.abs().max()) == 0.0
        assert bool(torch.isnan(case.bufs.rew_buf).all()) and bool((case.rb.root_states == SENTINEL).all())
        # busy: a device-output step in flight refuses both submits, then the slot works as before
        want = case.advance()
        case.submit(hs, 0)
        for fn, r in fns:
            assert fn(ctx, 0, C.byref(args), r, C.byref(case.dev._args()), n) == BUSY
        hs.wait(0)
        case.check_step(want, "after the errors")
        case.check_moments(n)


def test_close_with_device_out_batches_in_flight(monkeypatch):
    _set_path(monkeypatch, "direct")
    data, mlib = _motion_lib()
    a = Case(data, mlib, 2005, 111, auto_reset=True, norm=torch.bfloat16)
    b = Case(data, mlib, 1999, 121, pinned=False, moments=True)
    hs = HostStep(mlib, 2005, num_chunks=3)
    wa, wb = a.advance(), b.advance()
    a.submit(hs, 0)
    b.submit(hs, 1)
    hs.close()
    a.check_step(wa, "close, slot 0")
    b.check_step(wb, "close, slot 1")
    b.check_moments(1999)
