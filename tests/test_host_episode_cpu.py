"""CPU: the episode bookkeeping of the host step (phc_host_step_submit_episode): the NULL-context code, the
PhcHostEpisodeOut layout, and the Python validation of HostEpisodeBuffers.  No GPU needed: every call here fails before
the library touches a device, and the buffers are built on the meta device where CUDA ones would be."""

import ctypes as C

import pytest
import torch

from humanoid_b200 import HostEpisodeBuffers, _cabi


def test_null_context_is_refused():
    lib = _cabi.load()
    args, rargs, dev = _cabi.PhcHostStepArgs(), _cabi.PhcHostResetArgs(), _cabi.PhcHostDeviceOut()
    env, ep = _cabi.PhcHostEnvArgs(), _cabi.PhcHostEpisodeOut()
    fn = lib.phc_host_step_submit_episode
    assert fn(None, 0, C.byref(args), C.byref(rargs), C.byref(dev), C.byref(env), C.byref(ep), 8) == -1
    assert fn(None, 0, C.byref(args), None, None, None, C.byref(ep), 8) == -1
    assert fn(None, 0, None, None, None, None, None, 8) == -1


def test_episode_out_layout():
    # terminals, truncations, masks, episode_returns, episode_lengths, rewards, sums | buckets + pad | stream
    E = _cabi.PhcHostEpisodeOut
    assert C.sizeof(E) == 9 * 8
    offs = tuple(getattr(E, f).offset for f in ("terminals", "truncations", "masks", "episode_returns",
                                                "episode_lengths", "rewards", "sums", "buckets", "stream"))  # fmt: skip
    assert offs == (0, 8, 16, 24, 32, 40, 48, 56, 64)
    assert _cabi.EPISODE_SUM_COLS == 12


def _buffers(n=10, raw_cols=4, buckets=None, rewards=True):
    """HostEpisodeBuffers.allocate's tensors, on the meta device (validate checks the device type separately)."""
    return HostEpisodeBuffers.allocate(n, raw_cols, device="meta", buckets=buckets, rewards=rewards)


def test_allocate_shapes_and_default_buckets():
    e = _buffers(10)
    assert e.terminals.dtype == torch.bool and tuple(e.terminals.shape) == (10,)
    assert e.episode_lengths.dtype == torch.int32 and e.episode_returns.dtype == torch.float32
    assert e.rewards is not None and tuple(e.sums.shape) == (32, _cabi.EPISODE_SUM_COLS)
    assert e.sums.dtype == torch.float64 and e.raw_cols == 4 and e.n == 10
    # one row per block of four envs, within 32..4096 (as PHCPufferEnv)
    assert _buffers(4096).sums.shape[0] == 1024
    assert _buffers(1000).sums.shape[0] == 250
    assert _buffers(100000).sums.shape[0] == 4096
    assert _buffers(100, buckets=7).sums.shape[0] == 7
    assert _buffers(10, rewards=False).rewards is None


def test_validate_refuses_cpu_tensors_and_wrong_raw_cols():
    e = HostEpisodeBuffers(
        terminals=torch.zeros(6, dtype=torch.bool), truncations=torch.zeros(6, dtype=torch.bool),
        masks=torch.ones(6, dtype=torch.bool), episode_returns=torch.zeros(6), episode_lengths=torch.zeros(6, dtype=torch.int32),
        sums=torch.zeros(32, 12, dtype=torch.float64), raw_cols=4, rewards=torch.zeros(6),
    )  # fmt: skip
    with pytest.raises(_cabi.PhcError, match="CUDA tensor"):
        e.validate(6, 4)
    with pytest.raises(ValueError, match="reward terms"):
        e.validate(6, 5)  # the power reward writes five columns


class _FakeCuda:
    """Patches torch.Tensor so meta tensors pass the CUDA-device check: what follows it is dtype / shape / contiguity."""

    def __enter__(self):
        self.saved = torch.Tensor.device
        meta = torch.device("meta")

        def device(t):
            d = self.saved.__get__(t)
            return torch.device("cuda", 0) if d == meta else d

        torch.Tensor.device = property(device)
        return self

    def __exit__(self, *exc):
        torch.Tensor.device = self.saved


@pytest.mark.parametrize(
    "field, bad, err",
    [
        ("terminals", lambda n: torch.zeros(n, dtype=torch.int32, device="meta"), _cabi.PhcError),  # dtype
        ("masks", lambda n: torch.ones(n + 1, dtype=torch.bool, device="meta"), ValueError),  # shape
        ("episode_returns", lambda n: torch.zeros(n, dtype=torch.float64, device="meta"), _cabi.PhcError),
        ("episode_lengths", lambda n: torch.zeros(n, dtype=torch.int64, device="meta"), _cabi.PhcError),
        ("rewards", lambda n: torch.zeros(2 * n, device="meta")[::2], _cabi.PhcError),  # not contiguous
        ("sums", lambda n: torch.zeros(32, 8, dtype=torch.float64, device="meta"), ValueError),
        ("sums", lambda n: torch.zeros(4097, 12, dtype=torch.float64, device="meta"), ValueError),
        ("sums", lambda n: torch.zeros(32, 12, dtype=torch.float32, device="meta"), _cabi.PhcError),
        ("truncations", lambda n: torch.zeros(n, dtype=torch.bool), _cabi.PhcError),  # CPU, not CUDA
    ],
)
def test_validate_refuses_bad_tensors(field, bad, err):
    n = 10
    with _FakeCuda():
        e = _buffers(n)
        e.validate(n, 4)  # the allocated buffers pass
        setattr(e, field, bad(n))
        with pytest.raises(err):
            e.validate(n, 4)


def test_validate_takes_uint8_flags_and_no_rewards():
    with _FakeCuda():
        e = _buffers(10, raw_cols=5, rewards=False)
        e.terminals = torch.zeros(10, dtype=torch.uint8, device="meta")
        e.validate(10, 5)
        with pytest.raises(ValueError, match="shape"):
            e.validate(11, 5)


def test_log_needs_batches_of_one_kind():
    with pytest.raises(ValueError, match="at least one"):
        HostEpisodeBuffers.log([], 32)
    a, b = _buffers(8, 4), _buffers(8, 5)
    with pytest.raises(ValueError, match="same reward terms"):
        HostEpisodeBuffers.log([a, b], 32)
