"""TEST INFRASTRUCTURE ONLY -- generates the committed fixtures under ``tests/golden/``.

Run in the build container (needs ``/root/reference``):  ``python -m oracle.make_golden``

Fixtures produced
-----------------
``tests/golden/v3_jit_linear.npz``
    The reference's strongest pin on this path (reference ``tests/test_interpolation.py:297-378``,
    ``test_interp_regression_v3``): inputs decoded from
    ``tests/test_data/test_interpolation_data_random_linear.nc`` and the Parcels-v3 JIT golden
    trajectories decoded from ``tests/test_data/test_interpolation_jit_linear.zarr``.
    (``.nc`` = NetCDF-4/HDF5 with contiguous little-endian f64 datasets; ``.zarr`` = zarr-v2 with
    blosc-1/lz4/byte-shuffle chunks -- both decoded here without h5py/zarr, SURVEY.md 8c-11.)
``tests/golden/v3_jit_cgrid.npz``
    Same for ``..._cgrid_velocity`` (CGrid_Velocity on a rectilinear C-grid).
``tests/golden/ref_cases.npz``
    Outputs of the reference's OWN code (run through ``oracle/ref_harness.py``) on seeded
    synthetic inputs covering dtype / mesh / 2-D-3-D / static-time-varying / out-of-bounds /
    delayed-release / backward-in-time / partial-last-step cases.  Inputs are regenerated from
    the seeds by ``tests/cases.py``; only the reference's outputs are stored.
"""

from __future__ import annotations

import json
import os
import struct
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(ROOT, "tests", "golden")
REF_TESTDATA = "/root/reference/tests/test_data"


# ----------------------------------------------------------------------------------------------
# minimal HDF5 (superblock v2/3, v2 object headers, contiguous layout) dataset locator
# ----------------------------------------------------------------------------------------------
def _h5_datasets(buf: bytes) -> dict[str, tuple[int, tuple[int, ...]]]:
    """Return {name: (byte offset, shape)} for contiguous datasets linked from the root group."""
    assert buf[:8] == b"\x89HDF\r\n\x1a\n"
    ver = buf[8]
    assert ver in (2, 3), ver
    off_sz, len_sz = buf[9], buf[10]
    assert off_sz == 8 and len_sz == 8
    root = struct.unpack_from("<Q", buf, 12 + 8 * 3)[0]

    def messages(addr):
        assert buf[addr : addr + 4] == b"OHDR", buf[addr : addr + 4]
        flags = buf[addr + 5]
        p = addr + 6
        if flags & 0x20:
            p += 16
        if flags & 0x10:
            p += 4
        szf = 1 << (flags & 3)
        chunk0 = int.from_bytes(buf[p : p + szf], "little")
        p += szf
        track = bool(flags & 0x04)
        blocks = [(p, p + chunk0)]
        out = []
        while blocks:
            s, e = blocks.pop(0)
            q = s
            while q + 4 <= e - 0:  # (gap/checksum at the end is shorter than a message header)
                mtype = buf[q]
                msize = struct.unpack_from("<H", buf, q + 1)[0]
                q += 4 + (2 if track else 0)
                if q + msize > e:
                    break
                body = buf[q : q + msize]
                if mtype == 0x10:  # continuation
                    caddr, clen = struct.unpack_from("<QQ", body, 0)
                    assert buf[caddr : caddr + 4] == b"OCHK"
                    blocks.append((caddr + 4, caddr + clen - 4))
                else:
                    out.append((mtype, body))
                q += msize
        return out

    found = {}
    for mtype, body in messages(root):
        if mtype != 6:  # link message
            continue
        ver_l, fl = body[0], body[1]
        p = 2
        ltype = 0
        if fl & 0x08:
            ltype = body[p]
            p += 1
        if fl & 0x04:
            p += 8
        if fl & 0x10:
            p += 1
        lsz = 1 << (fl & 3)
        nlen = int.from_bytes(body[p : p + lsz], "little")
        p += lsz
        name = body[p : p + nlen].decode()
        p += nlen
        if ltype != 0:
            continue
        oaddr = struct.unpack_from("<Q", body, p)[0]
        shape, daddr = None, None
        for mt, b in messages(oaddr):
            if mt == 1:  # dataspace
                v, rank, f = b[0], b[1], b[2]
                q = 4 if v == 2 else 8
                shape = tuple(struct.unpack_from("<Q", b, q + 8 * i)[0] for i in range(rank))
            elif mt == 8 and b[0] == 3 and b[1] == 1:  # layout v3, contiguous
                daddr = struct.unpack_from("<Q", b, 2)[0]
        if shape is not None and daddr is not None:
            found[name] = (daddr, shape)
    return found


def read_nc_f64(path: str, names: list[str]) -> dict[str, np.ndarray]:
    buf = open(path, "rb").read()
    ds = _h5_datasets(buf)
    out = {}
    for n in names:
        off, shape = ds[n]
        cnt = int(np.prod(shape))
        out[n] = np.frombuffer(buf, dtype="<f8", count=cnt, offset=off).reshape(shape).copy()
    return out


# ----------------------------------------------------------------------------------------------
# blosc-1 (lz4, byte shuffle) chunk decoder for zarr-v2
# ----------------------------------------------------------------------------------------------
def _lz4_raw(src: bytes, n_out: int) -> bytes:
    import pyarrow as pa

    return pa.Codec("lz4_raw").decompress(src, decompressed_size=n_out).to_pybytes()


def blosc_decode(raw: bytes) -> bytes:
    _ver, _verlz, flags, typesize, nbytes, blocksize, _cbytes = struct.unpack_from("<BBBBIII", raw, 0)
    if flags & 0x02:  # memcpyed
        return raw[16 : 16 + nbytes]
    shuffled = bool(flags & 0x01)
    dont_split = bool(flags & 0x10)
    nblocks = (nbytes + blocksize - 1) // blocksize
    bstarts = struct.unpack_from(f"<{nblocks}I", raw, 16)
    out = bytearray()
    for b in range(nblocks):
        bsize = min(blocksize, nbytes - b * blocksize)
        leftover = bsize != blocksize
        nsplit = typesize if (not dont_split and typesize <= 16 and bsize // typesize >= 128 and not leftover) else 1
        # blosc-1 splits a full block into `typesize` streams when it is large enough
        if not dont_split and typesize <= 16 and bsize >= typesize * 128 and not leftover:
            nsplit = typesize
        p = bstarts[b]
        seg = bsize // nsplit
        blk = bytearray()
        for _ in range(nsplit):
            csize = struct.unpack_from("<i", raw, p)[0]
            p += 4
            blk += raw[p : p + csize] if csize == seg else _lz4_raw(raw[p : p + csize], seg)
            p += csize
        if shuffled and typesize > 1:
            n = bsize // typesize
            a = np.frombuffer(bytes(blk[: n * typesize]), dtype=np.uint8).reshape(typesize, n).T.copy()
            blk = bytearray(a.tobytes()) + blk[n * typesize :]
        out += blk
    return bytes(out)


def read_zarr_v2(path: str, var: str) -> np.ndarray:
    meta = json.load(open(os.path.join(path, var, ".zarray")))
    shape, chunks, dtype = meta["shape"], meta["chunks"], np.dtype(meta["dtype"])
    fill = meta["fill_value"]
    out = np.full(shape, np.nan if fill == "NaN" else (0 if fill is None else fill), dtype=dtype)
    grid = [(s + c - 1) // c for s, c in zip(shape, chunks, strict=True)]
    for idx in np.ndindex(*grid):
        f = os.path.join(path, var, ".".join(str(i) for i in idx))
        if not os.path.exists(f):
            continue
        arr = np.frombuffer(blosc_decode(open(f, "rb").read()), dtype=dtype).reshape(chunks)
        sl = tuple(slice(i * c, min((i + 1) * c, s)) for i, c, s in zip(idx, chunks, shape, strict=True))
        out[sl] = arr[tuple(slice(0, s.stop - s.start) for s in sl)]
    return out


def make_v3(interp_name: str, out_name: str):
    nc = read_nc_f64(
        os.path.join(REF_TESTDATA, f"test_interpolation_data_random_{interp_name}.nc"),
        ["U", "V", "W", "time", "depth", "lat", "lon"],
    )
    z = os.path.join(REF_TESTDATA, f"test_interpolation_jit_{interp_name}.zarr")
    traj = read_zarr_v2(z, "trajectory")
    order = np.argsort(traj, kind="stable")  # reference test sorts v3 rows by trajectory (:372)
    gold = {k: read_zarr_v2(z, k)[order] for k in ("lon", "lat", "z")}
    np.savez_compressed(
        os.path.join(GOLDEN, out_name),
        U=nc["U"], V=nc["V"], W=nc["W"], time=nc["time"], depth=nc["depth"], lat=nc["lat"], lon=nc["lon"],
        gold_lon=gold["lon"], gold_lat=gold["lat"], gold_z=gold["z"], trajectory=traj[order],
    )  # fmt: skip
    print(out_name, {k: v.shape for k, v in nc.items()}, gold["lon"].shape, "NaN frac", np.isnan(gold["lon"]).mean())


def make_ref_cases(only=None):
    """only: names to (re)generate, merged into the existing file (``python -m oracle.make_golden ref_cases name ...``)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import cases  # tests/cases.py: seeded input generators shared by tests and this script

    from . import ref_harness as rh

    out = {}
    if only:
        with np.load(os.path.join(GOLDEN, "ref_cases.npz")) as old:
            out = {k: old[k] for k in old.files if k.split("/")[0] not in only}
    for name, spec in cases.CASES.items():
        if only and name not in only:
            continue
        c = cases.build(spec)
        fs = rh.build_fieldset(
            lon=c["lon"], lat=c["lat"], depth=c["depth"], times=c["times"], U=c["U"], V=c["V"], W=c["W"],
            mesh=c["mesh"], constants=c["constants"], interp=c.get("interp", "linear"),
            padding=c.get("padding", ("low", "low", "high")),
        )  # fmt: skip
        ps = rh.make_pset(fs, x=c["x"], y=c["y"], z=c["z"], t=c["t"])
        k = rh.kernels()

        def DeleteParticle(particles, fieldset):
            particles[particles.state >= 50].state = 30

        kern = [getattr(k, kn) for kn in c["kernels"]]
        if c["delete_on_error"]:
            kern.append(DeleteParticle)
        err = ""
        if c["rng_seed"] is not None:
            np.random.seed(c["rng_seed"])
        try:
            for seg in c["segments"]:
                ps.execute(kern, dt=c["dt"], verbose_progress=False, **seg)
        except Exception as e:  # the reference raised: store which error
            err = type(e).__name__
        for key in ("x", "y", "z", "t", "state", "ei", "particle_id", "dt"):
            out[f"{name}/{key}"] = ps._data[key]
        out[f"{name}/error"] = np.array(err)
        print(f"{name}: n_out={len(ps._data['x'])} err={err!r} states={np.unique(ps._data['state'])}")
    np.savez_compressed(os.path.join(GOLDEN, "ref_cases.npz"), **out)


OUTPUT_CASES = {"delayed_partial": 300.0, "flat_f32c_f64d": 30.0, "backward": None}


def make_output_golden():
    """ParticleFile.write's row selection (reference _core/particlefile.py:198-221), run by the reference itself:
    (1) the rule on seeded vectors, (2) the rows an execute() with an output file writes, per output time."""
    import cases as tc
    from oracle import ref_harness as rh

    rh.install()
    from parcels._core.particlefile import _to_write_particles

    out = {}
    rng = np.random.default_rng(77)
    n = 4000
    t = np.round(rng.uniform(-50, 250, n), 1)
    t[rng.uniform(size=n) < 0.05] = np.nan
    t[rng.uniform(size=n) < 0.02] = np.inf
    dt = np.where(rng.uniform(size=n) < 0.5, 10.0, -10.0)
    pid = np.arange(n, dtype=np.int64)
    out["rule/t"], out["rule/dt"] = t, dt
    for k, tout in enumerate((0.0, 95.0, 100.0, 104.9, 105.0, 250.0)):
        out[f"rule/tout{k}"] = np.array(tout)
        out[f"rule/rows{k}"] = _to_write_particles({"t": t, "dt": dt, "particle_id": pid}, tout)

    class Recorder:
        path = "memory"

        def __init__(self, outputdt):
            self.outputdt, self.metadata, self.rows = outputdt, {}, []

        def set_metadata(self, mesh):
            pass

        def write(self, pset, time):
            d = pset._data
            rows = _to_write_particles(d, time)
            self.rows.append((time, {k: d[k][rows].copy() for k in ("particle_id", "t", "x", "y", "z")}))

        def __enter__(self):
            return self

        def __exit__(self, *a):
            pass

    k = rh.kernels()

    def DeleteParticle(particles, fieldset):
        particles[particles.state >= 50].state = 30

    for name, outputdt in OUTPUT_CASES.items():
        c = tc.build(tc.CASES[name])
        if outputdt is None:
            outputdt = 3 * abs(c["dt"])
        fs = rh.build_fieldset(lon=c["lon"], lat=c["lat"], depth=c["depth"], times=c["times"], U=c["U"], V=c["V"], W=c["W"],
                               mesh=c["mesh"], constants=c["constants"], interp=c.get("interp", "linear"),
                               padding=c.get("padding", ("low", "low", "high")))  # fmt: skip
        ps = rh.make_pset(fs, x=c["x"], y=c["y"], z=c["z"], t=c["t"])
        kern = [getattr(k, kn) for kn in c["kernels"]] + ([DeleteParticle] if c["delete_on_error"] else [])
        rec = Recorder(outputdt)
        seg = c["segments"][0]
        ps.execute(kern, dt=c["dt"], output_file=rec, verbose_progress=False, **seg)
        out[f"{name}/outputdt"] = np.array(outputdt)
        out[f"{name}/times"] = np.array([r[0] for r in rec.rows])
        for i, (_, cols) in enumerate(rec.rows):
            for key, v in cols.items():
                out[f"{name}/{i}/{key}"] = v
        print(f"output {name}: {len(rec.rows)} writes, rows {[len(r[1]['t']) for r in rec.rows]}")
    np.savez_compressed(os.path.join(GOLDEN, "output_rows.npz"), **out)


def make_output_rule_random_golden():
    """The reference's ``_to_write_particles`` on 20 seeded random draws (tests/test_output_cpu.py)."""
    from oracle import ref_harness as rh

    rh.install()
    from parcels._core.particlefile import _to_write_particles

    out = {}
    rng = np.random.default_rng(5)
    for k in range(20):
        n = 500
        t = np.round(rng.uniform(0, 100, n))
        t[rng.uniform(size=n) < 0.1] = np.nan
        dt = np.full(n, rng.choice([-7.0, 3.0, 10.0]))
        tout = float(np.round(rng.uniform(0, 100)))
        out[f"t{k}"], out[f"dt{k}"], out[f"tout{k}"] = t, dt, np.array(tout)
        out[f"rows{k}"] = _to_write_particles({"t": t, "dt": dt, "particle_id": np.arange(n)}, tout)
    np.savez_compressed(os.path.join(GOLDEN, "output_rule_random.npz"), **out)


def _fieldset_record(fs):
    """What ``parcels_b200.adapter.from_parcels`` reads from a reference FieldSet, as plain values (tests/test_adapter_cpu.py
    rebuilds the object from it)."""
    g = fs.U.grid
    md = g.sgrid_metadata

    def pad(p):
        return str(getattr(p, "value", p))

    axes = list(g.axes)
    return {
        "grid": {"axes": axes, "xdim": int(g.xdim), "ydim": int(g.ydim), "zdim": int(g.zdim) if "Z" in axes else None,
                 "deg2m": float(g.deg2m), "spherical": bool(g._mesh.is_spherical()), "radius": getattr(g._mesh, "radius", None),
                 "padding": [pad(f.padding) for f in md.face_dimensions],
                 "vertical_padding": [pad(v.padding) for v in md.vertical_dimensions] if md.vertical_dimensions else None},
        "time_ns": None if fs.U.time_interval is None else np.asarray(fs.U.data.time.values).astype(np.int64).tolist(),
        "fields": {name: {"interp": type(getattr(f, "interp_method", None)).__name__, "on_grid": getattr(f, "grid", None) is g,
                          "spherical": bool(f.grid._mesh.is_spherical()) if hasattr(f, "grid") else None}
                   for name, f in fs.fields.items()},
        "vector": type((getattr(fs, "UVW", None) or fs.UV).interp_method).__name__,
        "gridset": len(fs.gridset),
        "context": dict(fs.context),
    }  # fmt: skip


def make_adapter_golden():
    """Reference FieldSets / a ParticleSet as ``parcels_b200.adapter`` sees them (tests/test_adapter_cpu.py)."""
    import cases as tc
    from oracle import ref_harness as rh

    def fieldset(c, **kw):
        return rh.build_fieldset(lon=c["lon"], lat=c["lat"], depth=c["depth"], times=c["times"], U=c["U"], V=c["V"], W=c["W"],
                                 mesh=c["mesh"], **kw)  # fmt: skip

    rec, out = {}, {}
    c = tc.build(tc.CASES["diffusion"])
    ref = fieldset(c, constants=c["constants"])
    rec["diffusion"] = _fieldset_record(ref)
    for k, v in rh.make_pset(ref, x=c["x"], y=c["y"], z=c["z"], t=c["t"])._data.items():
        out[f"diffusion/pset/{k}"] = v
    c = tc.build(tc.CASES["curv_sph_2d"])
    rec["curv_sph_2d"] = _fieldset_record(fieldset(c, interp="cgrid_velocity", padding=c["padding"]))
    c = tc.build(tc.CASES["flat_f32c_f64d"])
    kz = np.abs(c["U"]) + 1
    c["W"] = None
    ref = fieldset(c, scalars={"Kh_zonal": (kz, "linear"), "Kh_meridional": (kz[:1], "linear")})
    ref.add_context("dres", 12.5)
    rec["flat_f32c_f64d"] = _fieldset_record(ref)
    k = rh.kernels()
    rec["kernel_modules"] = {name: getattr(k, name).__module__ for name in ("AdvectionDiffusionM1", "AdvectionRK4")}
    out["record"] = np.array(json.dumps(rec))
    np.savez_compressed(os.path.join(GOLDEN, "adapter_reference.npz"), **out)


SCALAR_CASES = ("c2_small", "flat_f32c_f64d", "all_f32", "cgrid_rect_3d")


def scalar_inputs(c, T, seed=3):
    """The scalar field + sample times used by the scalar-eval fixtures (shared with the tests)."""
    rng = np.random.default_rng(seed)
    P = rng.uniform(-1, 1, (T,) + c["U"].shape[1:]).astype(c["U"].dtype)
    tq = np.asarray(c["t"], dtype=np.float64) + (0.37 * c["times"][-1] if c["times"] is not None else 0.0)
    return P, tq


def land_tracer_inputs(c, T, seed=4):
    """Tracer field with blocks of land (exact zeros, growing with depth) for the XLinearInvdistLandTracer fixtures, and
    sample points that include ocean nodes of partly-land cells (the exact-node branch)."""
    rng = np.random.default_rng(seed)
    shape = (T,) + c["U"].shape[1:]
    P = (1.0 + rng.uniform(0, 1, shape)).astype(c["U"].dtype)
    ny, nx = shape[2], shape[3]
    r = rng.uniform(0, 1, (ny // 2 + 1, nx // 2 + 1))
    for k in range(shape[1]):
        land = np.kron(r < 0.3 + 0.05 * k, np.ones((2, 2), dtype=bool))[:ny, :nx]
        P[:, k][..., land] = 0
    x, y = np.array(c["x"], dtype=np.float64), np.array(c["y"], dtype=np.float64)
    n = min(40, len(x))
    jj, ii = rng.integers(0, ny, n), rng.integers(0, nx, n)
    x[:n], y[:n] = np.asarray(c["lon"], dtype=np.float64)[ii], np.asarray(c["lat"], dtype=np.float64)[jj]  # exactly on nodes
    tq = np.asarray(c["t"], dtype=np.float64) + (0.37 * c["times"][-1] if c["times"] is not None else 0.0)
    return P, tq, x, y


def make_scalar_golden():
    """Field.eval of the reference (XLinear / XNearest / CGrid_Tracer, with and without a time dimension)."""
    import warnings

    import cases as tc
    from oracle import ref_harness as rh

    out = {}
    for name in SCALAR_CASES:
        c = tc.build(tc.CASES[name])
        for T in (c["U"].shape[0], 1):
            P, tq = scalar_inputs(c, T)
            for how in ("linear", "nearest", "cgrid_tracer"):
                fs = rh.build_fieldset(lon=c["lon"], lat=c["lat"], depth=c["depth"], times=c["times"], U=c["U"], V=c["V"],
                                       W=c["W"], mesh=c["mesh"], padding=c.get("padding", ("low", "low", "high")),
                                       interp=c.get("interp", "linear"), scalars={"P": (P, how)})  # fmt: skip
                ps = rh.make_pset(fs, x=c["x"], y=c["y"], z=c["z"], t=c["t"])
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    val = fs.P.eval(tq, ps._data["z"], ps._data["y"], ps._data["x"], ps)
                key = f"{name}/T{T}/{how}"
                out[f"{key}/value"], out[f"{key}/state"], out[f"{key}/ei"] = val, ps._data["state"].copy(), ps._data["ei"].copy()
        for T in (c["U"].shape[0], 1):  # XLinearInvdistLandTracer on a field with land
            P, tq, x, y = land_tracer_inputs(c, T)
            fs = rh.build_fieldset(lon=c["lon"], lat=c["lat"], depth=c["depth"], times=c["times"], U=c["U"], V=c["V"], W=c["W"],
                                   mesh=c["mesh"], padding=c.get("padding", ("low", "low", "high")),
                                   interp=c.get("interp", "linear"), scalars={"P": (P, "linear_invdist_land")})  # fmt: skip
            ps = rh.make_pset(fs, x=x, y=y, z=c["z"], t=c["t"])
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                val = fs.P.eval(tq, ps._data["z"], ps._data["y"], ps._data["x"], ps)
            key = f"{name}/T{T}/linear_invdist_land"
            out[f"{key}/value"], out[f"{key}/state"], out[f"{key}/ei"] = val, ps._data["state"].copy(), ps._data["ei"].copy()
        print(f"scalar {name}: done")
    np.savez_compressed(os.path.join(GOLDEN, "scalar_eval.npz"), **out)


SCALAR_CURV_CASES = ("curv_sph_2d", "curv_flat_2d", "curv_sph_3d", "curv_sph_f32")


def make_scalar_curv_golden(methods=("nearest", "cgrid_tracer"), out_name="scalar_eval_curv.npz"):
    """Field.eval on CURVILINEAR grids (CGrid_Tracer / XNearest; XLinear in its own file, ``python -m oracle.make_golden
    scalar_curv_linear``): a fresh set (every hinted xi is 0: the whole batch goes through the spatial hash) and a second,
    displaced evaluation hinted by the cells just found."""
    import warnings

    import cases as tc
    from oracle import ref_harness as rh

    out = {}
    for name in SCALAR_CURV_CASES:
        c = tc.build(tc.CASES[name])
        for T in (c["U"].shape[0], 1):
            P, tq = scalar_inputs(c, T)
            for how in methods:
                fs = rh.build_fieldset(lon=c["lon"], lat=c["lat"], depth=c["depth"], times=c["times"], U=c["U"], V=c["V"], W=c["W"],
                                       mesh=c["mesh"], padding=c.get("padding", ("low", "low", "high")), interp="cgrid_velocity",
                                       scalars={"P": (P, how)})  # fmt: skip
                ps = rh.make_pset(fs, x=c["x"], y=c["y"], z=c["z"], t=c["t"])
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    val = fs.P.eval(tq, ps._data["z"], ps._data["y"], ps._data["x"], ps)
                    ei1 = ps._data["ei"].copy()
                    x2 = np.asarray(ps._data["x"], dtype=np.float64) + 0.3 * float(np.abs(np.diff(np.asarray(c["lon"], dtype=np.float64), axis=1)).mean())
                    val2 = fs.P.eval(tq, ps._data["z"], np.asarray(ps._data["y"], dtype=np.float64), x2, ps)
                key = f"{name}/T{T}/{how}"
                out[f"{key}/value"], out[f"{key}/ei"] = val, ei1
                out[f"{key}/value2"], out[f"{key}/ei2"], out[f"{key}/state2"] = val2, ps._data["ei"].copy(), ps._data["state"].copy()
        print(f"scalar curv {name}: done")
    np.savez_compressed(os.path.join(GOLDEN, out_name), **out)


# name -> (RK45_tol in metres, RK45_min_dt, RK45_max_dt factor of |dt|, runtime, dt)
RK45_CASES = {
    "flat_f32c_f64d": (1e-4, 0.5, 4, 140.0, 10.0),
    "c2_small": (0.5, 1.0, 4, 7200.0, 300.0),  # runs stay inside the fields' time axis (see DESIGN.md, RK45 waiver)
    "all_f32": (0.2, 1.0, 4, 3600.0, 150.0),
    "backward": (0.002, 7.0, 4, 5000.0, -600.0),
    "c1_peninsula": (1e-6, 1.0, 8, 3600.0, 300.0),
    # CGrid_Velocity: rectilinear (flat, spherical) and curvilinear (flat, spherical, float32 node coordinates) C-grids
    "cgrid_rect_3d": (2e-4, 1.0, 4, 500.0, 25.0),
    "cgrid_rect_sph": (2.0, 5.0, 4, 6000.0, 600.0),
    "curv_flat_2d": (1e-4, 1.0, 4, 600.0, 60.0),
    "curv_sph_2d": (20.0, 10.0, 4, 10800.0, 900.0),
    "curv_sph_f32": (20.0, 10.0, 4, 6000.0, 600.0),
    # XFreeslip / XPartialslip (land = nodes with U = V = 0)
    "freeslip_3d": (2e-4, 1.0, 4, 500.0, 25.0),
    "freeslip_surface": (1e-3, 1.0, 4, 700.0, 60.0),
    "partialslip_sph": (2.0, 5.0, 4, 6000.0, 600.0),
}


def make_rk45_golden():
    """AdvectionRK45 under the reference's own Kernel.execute (Repeat loop, next_dt, per-particle dt)."""
    import warnings

    import cases as tc
    from oracle import ref_harness as rh

    out = {}
    for name, (tol, min_dt, fmax, runtime, dt) in RK45_CASES.items():
        c = tc.build(tc.CASES[name])
        fs = rh.build_fieldset(lon=c["lon"], lat=c["lat"], depth=c["depth"], times=c["times"], U=c["U"], V=c["V"], W=c["W"],
                               mesh=c["mesh"], interp=c.get("interp", "linear"), padding=c.get("padding", ("low", "low", "high")))  # fmt: skip
        fs.add_context("RK45_tol", tol)
        fs.add_context("RK45_min_dt", min_dt)
        fs.add_context("RK45_max_dt", fmax * abs(dt))
        z = np.abs(np.asarray(c["z"]))
        ps = rh.make_pset(fs, x=c["x"], y=c["y"], z=z, t=c["t"], extra_variables=[("next_dt", np.float32, 0)])
        k = rh.kernels()
        attempts = [0]
        real = k.AdvectionRK45

        def Counted(particles, fieldset, real=real, attempts=attempts):
            attempts[0] += int(np.size(np.asarray(particles.state)))
            real(particles, fieldset)

        Counted.__name__ = "AdvectionRK45"
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ps.execute(real, dt=dt, runtime=runtime, verbose_progress=False)
        for key in ("x", "y", "z", "t", "dt", "next_dt", "state", "ei"):
            out[f"{name}/{key}"] = ps._data[key]
        out[f"{name}/tol_used"] = np.array(fs.context["RK45_tol"])  # after the reference's in-place unit conversion
        print(f"rk45 {name}: states {np.unique(ps._data['state'])} dt {np.unique(ps._data['dt'])[:5]} "
              f"next_dt {np.unique(ps._data['next_dt'])[:6]}")
    np.savez_compressed(os.path.join(GOLDEN, "rk45.npz"), **out)


# name -> (base case of tests/cases.py, kernel, Kh dtype, Kh fields have a time dimension, dt, runtime, delete-on-error, np.random seed)
ADVDIFF_CASES = {
    "m1_flat": ("flat_f32c_f64d", "AdvectionDiffusionM1", "f8", True, 10.0, 140.0, True, 1636),
    "em_sph": ("c2_small", "AdvectionDiffusionEM", "f4", True, 600.0, 6000.0, True, 1234),
    "m1_all_f32_static": ("all_f32", "AdvectionDiffusionM1", "f4", False, 300.0, 3300.0, True, 7),
    "em_f64_static": ("rk2_3d", "AdvectionDiffusionEM", "f8", False, 50.0, 700.0, True, 8),
    "m1_backward": ("backward", "AdvectionDiffusionM1", "f4", True, -600.0, 5400.0, True, 9),
    "em_raise": ("raise_oob", "AdvectionDiffusionEM", "f8", True, 100.0, 1500.0, False, 10),
    # fieldset.UV with CGrid_Velocity on rectilinear C-grids (the kernels are grid-agnostic, _advectiondiffusion.py:21-117)
    "m1_cgrid_flat": ("cgrid_rect_3d", "AdvectionDiffusionM1", "f8", True, 50.0, 550.0, True, 11),
    "em_cgrid_sph": ("cgrid_rect_sph", "AdvectionDiffusionEM", "f4", True, 600.0, 6000.0, True, 12),
}


def advdiff_inputs(c, kdtype, ktime, seed=5):
    """Kh_zonal / Kh_meridional (positive, smooth + noise, (T or 1, Z, Y, X)) and dres for an advection-diffusion case."""
    rng = np.random.default_rng(seed)
    T = c["U"].shape[0] if ktime else 1
    shape = (T,) + c["U"].shape[1:]
    ny, nx = shape[2], shape[3]
    X = np.linspace(0, 1, nx)[None, None, None, :]
    Y = np.linspace(0, 1, ny)[None, None, :, None]
    scale = 40.0 if c["mesh"] == "flat" else 4000.0
    kz = scale * (1.5 + np.tanh(6 * (X - 0.5)) + 0.3 * np.sin(5 * Y) + 0.2 * rng.uniform(-1, 1, shape))
    km = scale * (1.5 + np.tanh(4 * (Y - 0.4)) + 0.3 * np.cos(7 * X) + 0.2 * rng.uniform(-1, 1, shape))
    dres = float(np.float64(c["lon"][1]) - np.float64(c["lon"][0]))
    return kz.astype(kdtype), km.astype(kdtype), dres


def make_advdiff_golden(only=None):
    """AdvectionDiffusionM1 / EM under the reference's own Kernel.execute; the Wiener increments are the reference's
    (np.random.normal after np.random.seed): the oracle restatement draws the same stream.
    only: names to (re)generate, merged into the existing file (``python -m oracle.make_golden advdiff name ...``)."""
    import warnings

    import cases as tc
    from oracle import ref_harness as rh

    out = {}
    if only:
        with np.load(os.path.join(GOLDEN, "advdiff.npz")) as old:
            out = {k: old[k] for k in old.files if k.split("/")[0] not in only}
    for name, (base, kern, kd, ktime, dt, runtime, delete, rseed) in ADVDIFF_CASES.items():
        if only and name not in only:
            continue
        c = tc.build(tc.CASES[base])
        kz, km, dres = advdiff_inputs(c, kd, ktime)
        fs = rh.build_fieldset(lon=c["lon"], lat=c["lat"], depth=c["depth"], times=c["times"], U=c["U"], V=c["V"], W=None,
                               mesh=c["mesh"], interp=c.get("interp", "linear"), padding=c.get("padding", ("low", "low", "high")),
                               scalars={"Kh_zonal": (kz, "linear"), "Kh_meridional": (km, "linear")})  # fmt: skip
        fs.add_context("dres", dres)
        z = np.abs(np.asarray(c["z"]))
        ps = rh.make_pset(fs, x=c["x"], y=c["y"], z=z, t=c["t"])
        k = rh.kernels()
        kl = [getattr(k, kern)]
        if delete:
            def DeleteParticle(particles, fieldset):
                particles.state = np.where(particles.state >= 50, 30, particles.state)

            kl.append(DeleteParticle)
        err = ""
        np.random.seed(rseed)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            try:
                ps.execute(kl, dt=dt, runtime=runtime, verbose_progress=False)
            except Exception as e:  # noqa: BLE001 -- the reference's error classes
                err = type(e).__name__
        for key in ("particle_id", "x", "y", "z", "t", "dt", "state", "ei", "dx", "dy"):
            out[f"{name}/{key}"] = ps._data[key]
        out[f"{name}/error"] = np.array(err)
        print(f"advdiff {name}: {len(ps._data['x'])} of {len(c['x'])} particles left, states {np.unique(ps._data['state'])}, error {err!r}")
    np.savez_compressed(os.path.join(GOLDEN, "advdiff.npz"), **out)


if __name__ == "__main__":
    os.makedirs(GOLDEN, exist_ok=True)
    if len(sys.argv) > 1 and sys.argv[1] == "scalar_curv_linear":
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        make_scalar_curv_golden(methods=("linear",), out_name="scalar_eval_curv_linear.npz")
        sys.exit(0)
    if len(sys.argv) > 2 and sys.argv[1] == "advdiff":
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        make_advdiff_golden(only=set(sys.argv[2:]))
        sys.exit(0)
    if len(sys.argv) > 2 and sys.argv[1] == "ref_cases":
        make_ref_cases(only=set(sys.argv[2:]))
        sys.exit(0)
    make_v3("linear", "v3_jit_linear.npz")
    make_v3("cgrid_velocity", "v3_jit_cgrid.npz")
    make_v3("freeslip", "v3_jit_freeslip.npz")
    make_v3("nearest", "v3_jit_nearest.npz")
    make_ref_cases()
    make_output_golden()
    make_output_rule_random_golden()
    make_adapter_golden()
    make_scalar_golden()
    make_scalar_curv_golden()
    make_rk45_golden()
    make_advdiff_golden()
