"""CPU test: the oracle restatement is bit-identical to the reference's own code, run on the same cases
through ParticleSet.execute with its own kernels and a user DeleteParticle handler.  The reference's
outputs are stored in tests/golden/ref_cases.npz (oracle/make_golden.py)."""

import os

import numpy as np
import pytest

from oracle_run import load_case, run_oracle


@pytest.mark.parametrize("name", ["c2_small", "all_f32", "delayed_partial", "diffusion", "raise_oob"])
def test_live_reference_equals_oracle(name, golden_dir):
    ref = np.load(os.path.join(golden_dir, "ref_cases.npz"))
    pd, _ = run_oracle(load_case(name))
    for key in ("particle_id", "state", "ei", "t", "x", "y", "z"):
        np.testing.assert_array_equal(ref[f"{name}/{key}"], pd[key], err_msg=key)
