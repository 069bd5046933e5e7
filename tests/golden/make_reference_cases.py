"""Record ``reference_cases.npz``: the reference's outputs on the seeded inputs of tests/test_oracle_vs_reference.py,
which those tests compare with where the reference cannot be imported.

    python tests/golden/make_reference_cases.py

With the reference importable (``oracle.ref_loader``) its own functions are recorded.  Without it, the same numbers
come from ``oracle/phc_oracle.py`` and ``humanoid_b200.motion_build.ClipSampler``, which those tests hold equal to the
reference bit for bit (``torch.equal``) on exactly these inputs.  The recording in this directory was made that way:
nothing on the oracle side of those tests (oracle, synthetic inputs, ClipSampler) had changed since they last passed
against the live reference.  Obs and motion-state rows are kept for a fixed seeded sample of envs, and the fp64
sum of every obs row.
"""

from __future__ import annotations

import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from conftest import Golden  # noqa: E402
from oracle import ref_loader  # noqa: E402

import test_oracle_vs_reference as T  # noqa: E402

OBS_ROWS = 8
MOTION_STATE_ROWS = 16


def sample_rows(n, k, seed):
    return torch.randperm(n, generator=torch.Generator().manual_seed(seed))[:k].sort().values


def main():
    live = ref_loader.available()
    golden = Golden
    arrays = {}

    def put(prefix, d, rows=None):
        for k, v in d.items():
            v = v[rows] if rows is not None and k in T.ROW_KEYS else v
            arrays[f"{prefix}.{k}"] = v.detach().cpu().numpy()
        if rows is not None:
            arrays[f"{prefix}.rows"] = rows.numpy()

    for c, kw in enumerate(T.STEP_CASES):
        out = T.reference_step(kw) if live else T.oracle_step(kw)
        out["obs_row_sum"] = out["obs"].double().sum(1)  # every env's row, beside the sampled ones
        put(f"step{c}", out, sample_rows(kw["num_envs"], OBS_ROWS, seed=100 + c))
    ms = T.reference_motion_state() if live else T.oracle_motion_state()
    put("motion_state", ms, sample_rows(ms["root_pos"].shape[0], MOTION_STATE_ROWS, seed=200))
    put("sampler", T.reference_sampler_trace(golden) if live else T.sampler_trace(golden))

    path = os.path.join(HERE, T.RECORDED + ".npz")
    np.savez_compressed(path, **arrays)
    print(f"{T.RECORDED}: {os.path.getsize(path) / 1024:.0f} KiB, {len(arrays)} arrays, "
          f"from {'the reference' if live else 'the oracle side'}")  # fmt: skip


if __name__ == "__main__":
    main()
