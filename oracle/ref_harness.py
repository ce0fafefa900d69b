"""TEST INFRASTRUCTURE ONLY -- reference-code harness (never imported by the product path).

Runs the *reference's own* hot-path modules (``/root/reference/src/parcels``) in this
build container, where ``xarray``/``dask``/``zarr``/``cftime``/... are not installed, by
registering permissive stub modules and a NumPy duck type for ``xarray.DataArray``
(recipe: SURVEY.md Appendix A).  It is used for two things only:

* ``oracle/make_golden.py`` -- generate the committed fixtures under ``tests/golden/``
  (outputs of the reference itself on seeded inputs);
* ``tests/test_install_cpu.py`` -- where the reference package is present, run its own
  ``ParticleSet.execute`` with and without ``parcels_b200.install()``.

``/root/reference`` does not exist on the GPU box: nothing reachable from ``-m gpu`` tests,
``smoke()`` or ``bench.py`` imports this file.
"""

from __future__ import annotations

import os
import sys
import types

import numpy as np

REFERENCE_SRC = os.environ.get("PARCELS_REFERENCE_SRC", "/root/reference/src/parcels")


def reference_available() -> bool:
    return os.path.isdir(REFERENCE_SRC)


class _Stub(types.ModuleType):
    """Module whose every attribute is a fresh empty class (satisfies isinstance / annotations)."""

    __path__: list = []

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        cls = type(name, (), {})
        setattr(self, name, cls)
        return cls


class DataArray:
    """~40-line duck type for ``xarray.DataArray`` backed by a NumPy array."""

    def __init__(self, data, dims=None, coords=None, attrs=None, name=None):
        self._v = np.asarray(data)
        if dims is None:
            dims = tuple(f"dim_{i}" for i in range(self._v.ndim))
        if isinstance(dims, str):
            dims = (dims,)
        self.dims = tuple(dims)
        self._coords = dict(coords or {})
        self.attrs = dict(attrs or {})
        self.name = name

    values = property(lambda self: self._v)
    data = property(lambda self: self._v)
    shape = property(lambda self: self._v.shape)
    ndim = property(lambda self: self._v.ndim)
    dtype = property(lambda self: self._v.dtype)
    sizes = property(lambda self: dict(zip(self.dims, self._v.shape, strict=True)))

    def __getattr__(self, name):
        coords = self.__dict__.get("_coords", {})
        if name in coords:
            c = coords[name]
            return c if isinstance(c, DataArray) else DataArray(c, dims=(name,))
        raise AttributeError(name)

    def __getitem__(self, key):
        out = self._v[key]
        return DataArray(out, dims=tuple(f"d{i}" for i in range(np.ndim(out))))

    def __len__(self):
        return len(self._v)

    def load(self):
        return self

    def isel(self, indexers):
        """Pointwise (vectorised) selection: every indexed dim carries a flat 'points' index."""
        key = []
        for d, n in zip(self.dims, self._v.shape, strict=True):
            if d in indexers:
                idx = indexers[d]
                key.append(np.asarray(idx.values if isinstance(idx, DataArray) else idx))
            else:
                assert n == 1, f"un-indexed dim {d!r} must have size 1"
                key.append(0)
        return DataArray(self._v[tuple(key)], dims=("points",))


class Dataset:
    """Minimal duck ``xr.Dataset`` for XGrid: named variables + dims/sizes."""

    def __init__(self, variables: dict[str, DataArray], extra_dims: dict[str, int] | None = None):
        self._vars = variables
        self.sizes = dict(extra_dims or {})
        for v in variables.values():
            self.sizes.update(v.sizes)
        self.dims = set(self.sizes)

    def __getitem__(self, k):
        return self._vars[k]

    def __contains__(self, k):
        return k in self._vars

    def __getattr__(self, k):
        v = self.__dict__.get("_vars", {})
        if k in v:
            return v[k]
        raise AttributeError(k)

    def set_coords(self, *_):
        return self


_INSTALLED = False


def install():
    """Register the bare ``parcels`` package + third-party stubs (idempotent)."""
    global _INSTALLED
    if _INSTALLED:
        return
    if not reference_available():
        raise RuntimeError(f"reference sources not found at {REFERENCE_SRC}")
    for name in [
        "cftime", "zarr", "zarr.storage", "uxarray", "cf_xarray", "netCDF4", "pooch", "polars",
        "dask", "dask.array", "dask.base", "xarray", "xgcm",
    ]:  # fmt: skip
        if name not in sys.modules:
            try:
                __import__(name)
            except Exception:
                sys.modules[name] = _Stub(name)
    dask = sys.modules["dask"]
    if isinstance(dask, _Stub):
        dask.is_dask_collection = lambda x: False
        sys.modules["dask.base"].is_dask_collection = lambda x: False
        dask.base = sys.modules["dask.base"]
        dask.array = sys.modules["dask.array"]
    xr = sys.modules["xarray"]
    if isinstance(xr, _Stub):
        xr.register_dataset_accessor = lambda name: (lambda cls: cls)
        xr.DataArray = DataArray
        xr.Dataset = Dataset
    if "tqdm" not in sys.modules:
        try:
            import tqdm  # noqa: F401
        except Exception:
            m = _Stub("tqdm")
            m.tqdm = lambda *a, **k: None
            sys.modules["tqdm"] = m
    pkg = types.ModuleType("parcels")
    pkg.__path__ = [REFERENCE_SRC]
    sys.modules["parcels"] = pkg
    _INSTALLED = True


# ----------------------------------------------------------------------------------------------
# Builders: hand-built XGrid / model / fieldset around the reference's real classes.
# ----------------------------------------------------------------------------------------------


class _Model:
    def __init__(self, grid, data: dict[str, DataArray], time_interval):
        self.grid = grid
        self.data = data
        self.field_to_interpolator = {}
        self.time_interval = time_interval

    def field_data(self, name):
        return self.data[name]


class _FieldSet:
    def __init__(self, fields: dict, gridset: list, time_interval, context=None):
        self.fields = fields
        self.gridset = gridset
        self.time_interval = time_interval
        self.context = dict(context or {})
        for k, v in fields.items():
            setattr(self, k, v)

    def add_context(self, name, value):  # _core/fieldset.py:207-222
        if name in self.context:
            raise ValueError(f"FieldSet already has a context with name '{name}'")
        self.context[name] = value

    def __getattr__(self, name):
        ctx = self.__dict__.get("context", {})
        if name in ctx:
            return ctx[name]
        raise AttributeError(name)


def _padding(name):
    from parcels._sgrid import Padding

    return {"low": Padding.LOW, "high": Padding.HIGH, "none": Padding.NONE, "both": Padding.BOTH}[name]


def build_xgrid(*, lon, lat, depth=None, mesh="flat", padding=("low", "low", "high"), radius=None):
    """Reference ``XGrid`` (``_core/xgrid.py:107``) around duck datasets.

    ``lon``/``lat`` 1-D (rectilinear) or 2-D (curvilinear, shape (ny, nx)); ``depth`` 1-D or None.
    Dimension names: XG/YG nodes, XC/YC faces (absent from the dataset => cell count = nodes-1
    for LOW/HIGH padding, ``xgrid.py:21-24``).
    """
    install()
    from parcels._core.mesh import SphericalMesh, get_mesh
    from parcels._core.xgrid import XGrid
    from parcels._sgrid import FaceNodePadding, SGrid2DMetadata

    lon = np.asarray(lon)
    lat = np.asarray(lat)
    variables = {}
    if lon.ndim == 1:
        variables["lon"] = DataArray(lon, dims=("XG",))
        variables["lat"] = DataArray(lat, dims=("YG",))
    else:
        variables["lon"] = DataArray(lon, dims=("YG", "XG"))
        variables["lat"] = DataArray(lat, dims=("YG", "XG"))
    vertical = None
    if depth is not None:
        variables["depth"] = DataArray(np.asarray(depth), dims=("depth",))
        vertical = (FaceNodePadding("ZC", "depth", _padding(padding[2])),)
    g = object.__new__(XGrid)
    g._ds = Dataset(variables)
    g._mesh = SphericalMesh(radius) if radius is not None else get_mesh(mesh)
    g._spatialhash = None
    g.sgrid_metadata = SGrid2DMetadata(
        cf_role="grid_topology",
        topology_dimension=2,
        node_dimensions=("XG", "YG"),
        node_coordinates=("lon", "lat"),
        face_dimensions=(
            FaceNodePadding("XC", "XG", _padding(padding[0])),
            FaceNodePadding("YC", "YG", _padding(padding[1])),
        ),
        vertical_dimensions=vertical,
    )
    return g


def build_fieldset(
    *,
    lon,
    lat,
    depth=None,
    times=None,
    U,
    V,
    W=None,
    mesh="flat",
    padding=("low", "low", "high"),
    interp="linear",
    constants: dict[str, float] | None = None,
    radius=None,
    scalars: dict | None = None,
):
    """Duck FieldSet around the reference's real ``Field``/``VectorField``/``XGrid``/interpolators.

    U, V, W: arrays (T, Z, Y, X) (T == 1 with ``times=None`` => no time dimension).
    ``times``: float seconds (first must be 0).  ``constants``: name -> value, added as constant
    fields on a 0-D grid (mirrors ``FieldSet.add_constant_field``, ``fieldset.py:175-205``).
    """
    install()
    from parcels._core.field import Field, VectorField
    from parcels._core.utils.time import TimeInterval
    from parcels.interpolators._xinterpolators import CGrid_Velocity, XConstantField, XLinear, XLinear_Velocity

    grid = build_xgrid(lon=lon, lat=lat, depth=depth, mesh=mesh, padding=padding, radius=radius)
    zname = "depth" if depth is not None else "mockZ"
    if times is not None:
        times = np.asarray(times, dtype=np.float64)
        tcoord = (times * 1e9).astype("timedelta64[ns]")
        dims = ("time", zname, "YG", "XG")
        ti = TimeInterval(tcoord[0], tcoord[-1])
        coords = {"time": DataArray(tcoord, dims=("time",))}
    else:
        dims = ("mockT", zname, "YG", "XG")
        ti = None
        coords = {}
    data = {"U": DataArray(U, dims=dims, coords=coords), "V": DataArray(V, dims=dims, coords=coords)}
    if W is not None:
        data["W"] = DataArray(W, dims=dims, coords=coords)
    # scalar fields on the same grid: name -> (array (T, Z, Y, X), "linear" | "nearest" | "cgrid_tracer")
    smethod = {}
    for sname, (sarr, how) in (scalars or {}).items():
        sarr = np.asarray(sarr)
        if sarr.shape[0] > 1:
            data[sname] = DataArray(sarr, dims=("time", zname, "YG", "XG"), coords=coords)
        else:
            data[sname] = DataArray(sarr, dims=("mockT", zname, "YG", "XG"))
        smethod[sname] = how
    model = _Model(grid, data, ti)
    fields = {}
    from parcels.interpolators._xinterpolators import CGrid_Tracer, XLinearInvdistLandTracer
    from parcels.interpolators._xinterpolators import XNearest as _XNearest

    for name in data:
        f = Field(name, model)
        f.interp_method = {"linear": XLinear, "nearest": _XNearest, "cgrid_tracer": CGrid_Tracer,
                           "linear_invdist_land": XLinearInvdistLandTracer}[smethod.get(name, "linear")]()  # fmt: skip
        fields[name] = f
    from parcels.interpolators._base import VectorInterpolator
    from parcels.interpolators._xinterpolators import XFreeslip, XNearest, XPartialslip

    class XNearest_Velocity(VectorInterpolator):  # noqa: N801 -- as defined in the reference's tests/test_interpolation.py:279-294
        def interp(self, particle_positions, grid_positions, vectorfield):
            n = XNearest()
            return tuple(n.interp(particle_positions, grid_positions, f) for f in (vectorfield.U, vectorfield.V, vectorfield.W))

    vi = {"linear": XLinear_Velocity, "cgrid_velocity": CGrid_Velocity, "freeslip": XFreeslip, "partialslip": XPartialslip,
          "nearest": XNearest_Velocity}[interp]()  # fmt: skip
    fields["UV"] = VectorField("UV", fields["U"], fields["V"], interp_method=vi)
    if W is not None:
        fields["UVW"] = VectorField("UVW", fields["U"], fields["V"], fields["W"], interp_method=vi)
    gridset = [grid]
    if constants:
        # one shared model/grid per mesh, as CONSTANT_FIELD_MODELS (model.py:292-318)
        cgrid = build_const_grid(mesh=mesh, radius=radius)
        cmodel = _Model(cgrid, {}, None)
        for cname, cval in constants.items():
            cmodel.data[cname] = DataArray(np.full((1, 1, 1, 1), cval), dims=("mockT", "mockZ", "lat", "lon"))
            cf = Field(cname, cmodel)
            cf.interp_method = XConstantField()
            fields[cname] = cf
        gridset.append(cgrid)
    return _FieldSet(fields, gridset, ti)


def build_const_grid(mesh="flat", radius=None):
    """Grid of a constant field (``model.py:292-318``): lon=[0], lat=[0] (X, Y axes of size 1), no Z axis."""
    install()
    from parcels._core.mesh import SphericalMesh, get_mesh
    from parcels._core.xgrid import XGrid
    from parcels._sgrid import FaceNodePadding, Padding, SGrid2DMetadata

    g = object.__new__(XGrid)
    g._ds = Dataset({"lon": DataArray(np.array([0]), dims=("lon",)), "lat": DataArray(np.array([0]), dims=("lat",))})
    g._mesh = SphericalMesh(radius) if radius is not None else get_mesh(mesh)
    g._spatialhash = None
    g.sgrid_metadata = SGrid2DMetadata(
        cf_role="grid_topology",
        topology_dimension=2,
        node_dimensions=("lon", "lat"),
        face_dimensions=(FaceNodePadding("XC", "lon", Padding.LOW), FaceNodePadding("YC", "lat", Padding.LOW)),
        vertical_dimensions=None,
    )
    return g


def make_pset(fieldset, *, x, y, z, t=None, extra_variables=(), **kwargs):
    """``extra_variables``: (name, dtype, initial) tuples added to the default Particle (e.g. next_dt for RK45)."""
    install()
    from parcels._core.particle import Particle, Variable
    from parcels._core.particleset import ParticleSet

    n = np.size(x)
    if t is None:
        t = np.repeat(np.timedelta64(0, "s"), n)
    elif not isinstance(np.asarray(t).flat[0], np.timedelta64):
        t = (np.asarray(t, dtype=np.float64) * 1e9).astype("timedelta64[ns]")
    if extra_variables:
        pclass = Particle.add_variable([Variable(n_, dtype=d_, initial=i_) for n_, d_, i_ in extra_variables])
        return ParticleSet(fieldset, pclass=pclass, x=x, y=y, z=z, t=t, **kwargs)
    return ParticleSet(fieldset, x=x, y=y, z=z, t=t)


def kernels():
    install()
    import parcels.kernels as k

    return k
