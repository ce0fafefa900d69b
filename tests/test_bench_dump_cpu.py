"""CPU test of bench.py --dump-outputs: what a caller of ParticleSet.execute receives (deleted particles dropped), float32 /
float64 files only, within the byte budget, and the same seeded sample of particles from run to run."""

import os

import numpy as np

import bench
from parcels_b200.particle import create_particle_data
from parcels_b200.statuscodes import StatusCode


def _particles(n):
    d = create_particle_data(nparticles=n, ngrids=2, initial=dict(x=np.arange(n) * 1e-3, y=np.ones(n), z=np.ones(n), t=np.zeros(n),
                                                                    particle_id=np.arange(n)))  # fmt: skip
    d["state"][::7] = StatusCode.Delete
    return d


def _load(path):
    return {f[len("w_"):-len(".npy")]: np.load(os.path.join(path, f)) for f in sorted(os.listdir(path))}


def test_whole_set_below_the_budget(tmp_path):
    d = _particles(1000)
    bench.dump_outputs(tmp_path, "w", d, d["particle_id"], 1 << 20)
    out = _load(tmp_path)
    assert set(out) == set(d)
    assert all(v.dtype in (np.float32, np.float64) for v in out.values())
    keep = d["state"] != StatusCode.Delete
    np.testing.assert_array_equal(out["particle_id"], d["particle_id"][keep])
    np.testing.assert_array_equal(out["x"], d["x"][keep])
    assert out["ei"].shape == (keep.sum(), 2)


def test_fixed_sample_within_the_budget(tmp_path):
    d = _particles(200_000)
    budget = 1 << 20
    for run in ("a", "b"):
        bench.dump_outputs(tmp_path / run, "w", d, d["particle_id"], budget)
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= budget
    assert 0 < len(a["particle_id"]) < 200_000
    for k in a:
        np.testing.assert_array_equal(a[k], b[k])
    assert not np.isin(a["particle_id"], d["particle_id"][d["state"] == StatusCode.Delete]).any()
