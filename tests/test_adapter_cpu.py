"""CPU test: the adapter reads a reference FieldSet correctly.  The reference objects are rebuilt from
tests/golden/adapter_reference.npz (what ``adapter.from_parcels`` reads of them, recorded from the reference
itself by oracle/make_golden.py) around the inputs of tests/cases.py."""

import json
import os
from types import SimpleNamespace as NS

import numpy as np
import pytest

from oracle_run import load_case


@pytest.fixture(scope="module")
def golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "adapter_reference.npz"))
    return json.loads(str(g["record"])), g


def _ref_fieldset(rec, arrays, constants=None):
    """A reference FieldSet as recorded: grids, fields with their interpolator class names, vector fields, context."""
    gr = rec["grid"]

    def mesh(spherical, radius=None):
        return NS(is_spherical=lambda: spherical, **({} if radius is None else {"radius": radius}))

    def padding(values):
        return tuple(NS(padding=NS(value=v)) for v in values)

    md = NS(face_dimensions=padding(gr["padding"]), vertical_dimensions=gr["vertical_padding"] and padding(gr["vertical_padding"]))
    grid = NS(lon=arrays["lon"], lat=arrays["lat"], depth=arrays["depth"], axes=gr["axes"], xdim=gr["xdim"], ydim=gr["ydim"],
              zdim=gr["zdim"], deg2m=gr["deg2m"], _mesh=mesh(gr["spherical"], gr["radius"]), sgrid_metadata=md)  # fmt: skip
    time = None if rec["time_ns"] is None else NS(values=np.array(rec["time_ns"], dtype="timedelta64[ns]"))
    const_grid = NS(_mesh=mesh(gr["spherical"]))
    fields = {}
    for name, f in rec["fields"].items():
        value = arrays.get(name)
        if f["interp"] == "XConstantField":
            value = np.full((1, 1, 1, 1), (constants or {})[name])
        fields[name] = NS(data=NS(values=value, time=time), grid=grid if f["on_grid"] else const_grid,
                          interp_method=type(f["interp"], (), {})(), time_interval=None if time is None else True)  # fmt: skip
    assert type(fields["UV"].interp_method).__name__ == rec["vector"]
    return NS(fields=fields, gridset=[grid] * rec["gridset"], context=dict(rec["context"]), **fields)


def test_from_parcels_reads_reference_fieldset(golden):
    from parcels_b200 import adapter

    rec, g = golden
    c = load_case("diffusion")
    ref = _ref_fieldset(rec["diffusion"], c, constants=c["constants"])
    fs = adapter.from_parcels(ref)
    np.testing.assert_array_equal(fs.grid.lon, c["lon"])
    np.testing.assert_array_equal(fs.grid.depth, c["depth"])
    assert fs.grid.is_spherical() and fs.grid.deg2m == ref.U.grid.deg2m
    assert (fs.grid.xdim, fs.grid.ydim, fs.grid.zdim) == (ref.U.grid.xdim, ref.U.grid.ydim, ref.U.grid.zdim)
    np.testing.assert_array_equal(fs._time_s, c["times"])
    np.testing.assert_array_equal(fs.W.data, c["W"])
    assert fs.constants == {"Kh_zonal": 100.0, "Kh_meridional": 50.0}
    assert len(fs.gridset) == len(ref.gridset) == 2
    rp = NS(_data={k.split("/")[-1]: g[k].copy() for k in g.files if k.startswith("diffusion/pset/")})
    ps = adapter.pset_from_parcels(rp, fs)
    assert ps._data is rp._data and ps._data["ei"].shape == (len(c["x"]), 2)


def test_from_parcels_curvilinear_cgrid_scalars_and_context(golden):
    from parcels_b200 import adapter
    from parcels_b200.particleset import KernelPlan
    import parcels_b200 as pb

    rec, _ = golden
    c = load_case("curv_sph_2d")
    ref = _ref_fieldset(rec["curv_sph_2d"], c)
    fs = adapter.from_parcels(ref)
    assert fs.grid.curvilinear and fs.interp_method == "cgrid_velocity" and fs.offsets == (1, 1, 0)
    assert (fs.grid.xdim, fs.grid.ydim) == (ref.U.grid.xdim, ref.U.grid.ydim)
    np.testing.assert_array_equal(fs.grid.lon, c["lon"])

    c = load_case("flat_f32c_f64d")
    kz = np.abs(c["U"]) + 1
    ref = _ref_fieldset(rec["flat_f32c_f64d"], {**c, "Kh_zonal": kz, "Kh_meridional": kz[:1]})
    fs = adapter.from_parcels(ref)
    assert fs.context == {"dres": 12.5} and fs.Kh_zonal._slot == 3 and fs.Kh_meridional.data.shape[0] == 1

    def reference_kernel(name):  # stands for the reference's own kernel function: same name, same module
        f = lambda particles, fieldset: None  # noqa: E731
        f.__name__, f.__module__ = name, rec["kernel_modules"][name]
        return f

    with pytest.raises(NotImplementedError, match="share dtype and time dimension"):
        KernelPlan([reference_kernel("AdvectionDiffusionM1")], fs)  # the reference's own kernel function is recognised as the built-in
    assert KernelPlan([reference_kernel("AdvectionRK4"), pb.DeleteParticle], fs).scheme == 4
