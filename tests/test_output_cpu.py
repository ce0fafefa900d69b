"""Output path, host side (no GPU): the selection rule against the reference's own outputs, ParticleFile's
constructor checks and Parquet round trip (reference _core/particlefile.py:54-221)."""

import os

import numpy as np
import pytest

import parcels_b200 as pb
from oracle import parcels_oracle as po
from parcels_b200.particlefile import to_write_particles


def _rule_vectors(golden_dir):
    g = np.load(os.path.join(golden_dir, "output_rows.npz"))
    d = {"t": g["rule/t"], "dt": g["rule/dt"], "particle_id": np.arange(len(g["rule/t"]), dtype=np.int64)}
    return g, d


def test_selection_rule_matches_reference_outputs(golden_dir):
    g, d = _rule_vectors(golden_dir)
    k = 0
    while f"rule/tout{k}" in g:
        tout = float(g[f"rule/tout{k}"])
        np.testing.assert_array_equal(po.to_write_particles(d, tout), g[f"rule/rows{k}"])  # oracle restatement
        np.testing.assert_array_equal(to_write_particles(d, tout), g[f"rule/rows{k}"])  # host form of the product
        k += 1
    assert k == 6


def test_selection_rule_matches_reference_code(golden_dir):
    """20 random draws and the rows the reference's own _to_write_particles selected for them (oracle/make_golden.py)."""
    g = np.load(os.path.join(golden_dir, "output_rule_random.npz"))
    for k in range(20):
        d = {"t": g[f"t{k}"], "dt": g[f"dt{k}"], "particle_id": np.arange(len(g[f"t{k}"]))}
        tout = float(g[f"tout{k}"])
        np.testing.assert_array_equal(po.to_write_particles(d, tout), g[f"rows{k}"])
        np.testing.assert_array_equal(to_write_particles(d, tout), g[f"rows{k}"])


def _tiny_pset(n=50, pclass=pb.Particle, **kw):
    lon, lat = np.linspace(0, 10, 6), np.linspace(0, 5, 4)
    U = np.ones((1, 1, 4, 6), dtype=np.float32)
    fs = pb.FieldSet.from_arrays(lon=lon, lat=lat, U=U, V=U, mesh="flat")
    rng = np.random.default_rng(1)
    return pb.ParticleSet(fs, pclass=pclass, x=rng.uniform(1, 9, n), y=rng.uniform(1, 4, n), t=np.arange(n, dtype=float), **kw)


def test_particlefile_constructor_checks(tmp_path):
    with pytest.raises(ValueError, match="extension must be '.parquet'"):
        pb.ParticleFile(tmp_path / "out.zarr", outputdt=1.0)
    with pytest.raises(ValueError, match="positive/non-zero"):
        pb.ParticleFile(tmp_path / "a.parquet", outputdt=0.0)
    with pytest.raises(ValueError, match="Expected outputdt"):
        pb.ParticleFile(tmp_path / "a.parquet", outputdt=1)
    with pytest.raises(ValueError, match="Invalid mode"):
        pb.ParticleFile(tmp_path / "a.parquet", outputdt=1.0, mode="a")
    with pytest.raises(ValueError, match="does not exist"):
        pb.ParticleFile(tmp_path / "nodir" / "a.parquet", outputdt=1.0)
    (tmp_path / "b.parquet").write_bytes(b"x")
    with pytest.raises(ValueError, match="already exists"):
        pb.ParticleFile(tmp_path / "b.parquet", outputdt=1.0)
    pf = pb.ParticleFile(tmp_path / "b.parquet", outputdt=np.timedelta64(90, "s"), mode="w")
    assert pf.outputdt == 90.0 and not (tmp_path / "b.parquet").exists()


def test_particlefile_host_round_trip(tmp_path):
    import pyarrow.parquet as pq

    P = pb.Particle.add_variable([pb.Variable("age", np.float32, initial=2.5, attrs={"units": "s"}),
                                  pb.Variable("scratch", np.int32, to_write=False)])  # fmt: skip
    ps = _tiny_pset(pclass=P)
    ps._data["dt"][:] = 4.0
    with pb.ParticleFile(tmp_path / "traj.parquet", outputdt=10.0) as pf:
        pf.set_metadata("flat")
        pf.write(ps, 10.0)  # rows with 8 <= t <= 12
        pf.write(ps, np.timedelta64(30, "s"))
    tab = pq.read_table(tmp_path / "traj.parquet")
    assert tab.column_names == ["t", "z", "y", "x", "particle_id", "age"]  # declaration order, to_write only
    assert tab.schema.field("x").metadata[b"units"] == b"degrees_east"
    assert tab.schema.field("age").metadata[b"units"] == b"s"
    assert tab.schema.metadata[b"feature_type"] == b"trajectory"
    d = pb.read_particlefile(tmp_path / "traj.parquet")
    np.testing.assert_array_equal(d["particle_id"], [8, 9, 10, 11, 12, 28, 29, 30, 31, 32])
    np.testing.assert_array_equal(d["x"], ps._data["x"][d["particle_id"]])
    assert d["x"].dtype == np.float32 and d["t"].dtype == np.float64 and d["particle_id"].dtype == np.int64
    assert pf.rows_written == 10 and pf.device_writes == 0


def test_time_units_follow_the_time_axis(tmp_path):
    import pyarrow.parquet as pq

    lon, lat = np.linspace(0, 10, 6), np.linspace(0, 5, 4)
    U = np.ones((3, 1, 4, 6), dtype=np.float32)
    for k, (time, units) in enumerate((
        (np.array([0.0, 10.0, 20.0]), b"seconds"),
        (np.array([0, 10, 20], dtype="timedelta64[s]"), b"seconds"),
        (np.datetime64("2000-01-02T03:00:00") + np.array([0, 10, 20], dtype="timedelta64[s]"), b"seconds since 2000-01-02 03:00:00"),
    )):  # fmt: skip
        fs = pb.FieldSet.from_arrays(lon=lon, lat=lat, U=U, V=U, time=time, mesh="flat")
        ps = pb.ParticleSet(fs, x=[1.0, 2.0], y=[1.0, 2.0], t=[0.0, 0.0])
        with pb.ParticleFile(tmp_path / f"t{k}.parquet", outputdt=10.0) as pf:
            pf.write(ps, 0.0)
        assert pq.read_table(tmp_path / f"t{k}.parquet").schema.field("t").metadata[b"units"] == units


def test_variable_validation():
    with pytest.raises(ValueError, match="to_write must be one of"):
        pb.Variable("a", to_write="once")
    with pytest.raises(ValueError, match="Attributes cannot be set"):
        pb.Variable("a", to_write=False, attrs={"units": "m"})
    with pytest.raises(TypeError, match="valid numpy dtype"):
        pb.Variable("a", dtype="not-a-dtype")
