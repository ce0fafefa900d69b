#!/usr/bin/env python
"""bench.py -- particle-RK4-steps/s of the hot path on N B200s (contract: see the task statement).

One bench "step" = one pass of the hot path over one batch: ``Kernel.execute`` of the workload's kernel list over the
whole particle set for one output interval (e.g. 144 dt-steps of 600 s = one day), i.e. dt_steps x N_particles
particle-RK4-steps.

  value         whole-job particle-RK4-steps/s, particles + field already resident in HBM (CUDA events, max over ranks)
  e2e           same metric through the public API ``ParticleSet.execute`` with HOST particle arrays: host->device upload
                and device->host download of the particle SoA inside the timed region
  roofline      algorithmic bytes per particle-RK4-step (SURVEY.md 8d / DESIGN.md) x steps per launch / CUDA-event duration
                of the advection kernel, against the measured HBM peak
  parity_sample the GPU and the CPU oracle advect the SAME bounded sample of the workload: ids / states / times / cells
                compared bit for bit, positions in float32 ulp (N = 1, rank 0)
  cpu_baseline  the time the oracle took for that sample (NumPy restatement of the reference path, one core)

Default (the driver's ``--gpus 1``): the north-star workload ``ns`` (BASELINE.json: 1e7 particles, 1/12 deg 3-D rectilinear
field) as value / e2e / roofline, and BASELINE configs[1..3] (``c2``, ``c3``, ``c4``) as compact blocks under ``extra``.
``--gpus N`` > 1 (torchrun): mode R (field replicated, particles sharded, no data-path collective) as value, plus a
``mode_d`` block: BASELINE configs[4] (``c5``: the 1/12 deg field cut into N X-slabs, NCCL all-to-all particle migration)
with a bit-exactness check of the decomposed run against a single GPU.

``--impl reference`` times the reference arm: the reference's own algorithm (oracle port; the reference is pure Python and
cannot travel to the GPU box) on all host cores, same ``config``.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "particle-RK4-steps/sec"
DUMP_BYTES = 60 << 20  # --dump-outputs: all files of one run together stay below 64 MB
_G = {}


# ------------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------------
def c2_field(nx=1440, ny=720, nz=50, nt=3, seed=1):
    """config 2 (SURVEY.md 8d): rectilinear 1/4 deg x 50 levels, T=3 daily snapshots, f32 U,V,W, spherical."""
    rng = np.random.default_rng(seed)
    lon = np.linspace(-180.0, 180.0, nx)
    lat = np.linspace(-80.0, 80.0, ny)
    depth = 5500.0 * (np.linspace(0.0, 1.0, nz) ** 1.8)
    times = np.arange(nt) * 86400.0
    X = (2 * np.pi * np.linspace(0, 1, nx)).astype(np.float32)[None, None, None, :]
    Y = (2 * np.pi * np.linspace(0, 1, ny)).astype(np.float32)[None, None, :, None]
    Z = np.linspace(0, 1, nz).astype(np.float32)[None, :, None, None]
    T = np.arange(nt, dtype=np.float32)[:, None, None, None]
    shape = (nt, nz, ny, nx)

    def noise():
        return rng.random(shape, dtype=np.float32) * np.float32(0.1) - np.float32(0.05)

    U = (np.sin(3 * X + 0.3 * T) * np.cos(2 * Y) * (1 - 0.5 * Z) * np.float32(0.6)
         + np.cos(5 * Y + T) * np.float32(0.3) + noise()).astype(np.float32)  # fmt: skip
    V = (np.cos(2 * X + 0.2 * T) * np.sin(4 * Y) * (1 - 0.3 * Z) * np.float32(0.6)
         + np.sin(3 * X) * np.float32(0.25) + noise()).astype(np.float32)  # fmt: skip
    W = ((np.sin(2 * X) * np.sin(3 * Y) * np.sin(np.float32(np.pi) * Z) * np.cos(0.5 * T) * np.float32(0.9)
          + noise()) * np.float32(1e-3)).astype(np.float32)  # fmt: skip
    return dict(lon=lon, lat=lat, depth=depth, times=times, U=U, V=V, W=W, mesh="spherical")


NS_TILE = 60  # the noise of the north-star field is a (nz, 60, 60) block per level and component, repeated over (y, x)


def ns_field(nx=4320, ny=2160, nz=50, nt=3, seed=4, device=None, threads=None):
    """north-star target field (BASELINE.json north_star: "1e7 particles on a 1/12 deg 3D rectilinear field"): the config-2
    modes at 4320 x 2160 x 50, T=3 -- 5.6 GB per component, 16.8 GB in all.

    Built from 1-D float32 factors (made once on the host with NumPy) by single float32 multiplications / additions in a fixed
    order, plus a seeded noise block tiled over (y, x): IEEE arithmetic without contraction, so the field generated IN HBM
    (``device`` = a CUDA index: torch elementwise kernels, handed to the engine without a copy) and the field generated on the
    HOST (``device=None``: torch CPU threads; for the oracle / the reference arm) are the same bits -- bench checks a plane."""
    import torch

    assert ny % NS_TILE == 0 and nx % NS_TILE == 0, "ny and nx must be multiples of the noise tile"
    dev = torch.device("cpu") if device is None else torch.device(f"cuda:{device}")
    if device is None and threads:
        torch.set_num_threads(int(threads))
    rng = np.random.default_rng(seed)
    lon = np.linspace(-180.0, 180.0, nx)
    lat = np.linspace(-80.0, 80.0, ny)
    depth = 5500.0 * (np.linspace(0.0, 1.0, nz) ** 1.8)
    times = np.arange(nt) * 86400.0
    X, Y, Z = 2 * np.pi * np.linspace(0, 1, nx), 2 * np.pi * np.linspace(0, 1, ny), np.linspace(0, 1, nz)

    def t32(a):
        return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)

    U, V, W = (torch.empty((nt, nz, ny, nx), dtype=torch.float32, device=dev) for _ in range(3))
    for k in range(nt):
        T = float(k)
        # component = (fx[x] * fy[y]) * fz[z] * amp + gy[y] (or gx[x]) + tile          -- every step ONE float32 operation
        spec = {
            "U": (np.sin(3 * X + 0.3 * T), np.cos(2 * Y), 1 - 0.5 * Z, 0.6, ("y", np.cos(5 * Y + T) * 0.3), 1.0),
            "V": (np.cos(2 * X + 0.2 * T), np.sin(4 * Y), 1 - 0.3 * Z, 0.6, ("x", np.sin(3 * X) * 0.25), 1.0),
            "W": (np.sin(2 * X), np.sin(3 * Y), np.sin(np.pi * Z) * np.cos(0.5 * T), 0.9, None, 1e-3),
        }
        for name, out in (("U", U), ("V", V), ("W", W)):
            fx, fy, fz, amp, add, scale = spec[name]
            tile = t32(rng.random((nz, NS_TILE, NS_TILE), dtype=np.float32) * np.float32(0.1) - np.float32(0.05))
            plane = t32(fx)[None, :] * t32(fy)[:, None]                       # (ny, nx)
            lvl = out[k]
            torch.mul(plane[None, :, :], t32(fz)[:, None, None], out=lvl)      # (nz, ny, nx)
            lvl.mul_(float(np.float32(amp)))
            if add is not None:
                lvl.add_(t32(add[1])[None, :, None] if add[0] == "y" else t32(add[1])[None, None, :])
            lvl.add_(tile.repeat(1, ny // NS_TILE, nx // NS_TILE))
            if scale != 1.0:
                lvl.mul_(float(np.float32(scale)))
    if device is not None:
        torch.cuda.synchronize(dev)
        return dict(lon=lon, lat=lat, depth=depth, times=times, U=U, V=V, W=W, mesh="spherical")
    return dict(lon=lon, lat=lat, depth=depth, times=times, U=U.numpy(), V=V.numpy(), W=W.numpy(), mesh="spherical")


def c2_particles(field, n, seed):
    rng = np.random.default_rng(seed)
    return dict(x=rng.uniform(-170, 170, n), y=rng.uniform(-70, 70, n), z=rng.uniform(5, 5000, n), t=np.zeros(n))


def dense_particles(field, n, seed):
    """a dense release (the common Parcels use: a cloud in a patch): 4 deg x 4 deg x the upper 200 m -- on the 1/12 deg grid
    48 x 48 x ~12 cells, hundreds of particles per cell, so the lanes of a warp share cells and cache lines"""
    rng = np.random.default_rng(seed)
    return dict(x=rng.uniform(-32, -28, n), y=rng.uniform(38, 42, n), z=rng.uniform(5, 200, n), t=np.zeros(n))


def c3_field(nx=1442, ny=1021, nt=3, seed=2, nz=1):
    """config 3: curvilinear C-grid of ORCA025 shape (ny, nx) = (1021, 1442): rotated-pole mesh with a
    tanh-stretched latitude, f32 node coordinates (NEMO style), NEMO staggering (offsets X=1, Y=1); 2-D, or with nz > 1
    depth levels and a W component (SURVEY.md 8 row f-4: the 3-D curvilinear path at ORCA size)."""
    rng = np.random.default_rng(seed)
    lam = np.deg2rad(np.linspace(-70.0, 70.0, nx))[None, :]          # rotated longitude
    s = np.linspace(-1.0, 1.0, ny)[:, None]
    phi = np.deg2rad(42.0 * np.tanh(1.2 * s) / np.tanh(1.2))         # rotated latitude, finer near the "equator"
    pole = np.deg2rad(25.0)                                          # tilt of the rotated pole
    xr, yr, zr = np.cos(phi) * np.cos(lam), np.cos(phi) * np.sin(lam), np.sin(phi) * np.ones_like(lam)
    xg = np.cos(pole) * xr - np.sin(pole) * zr
    zg = np.sin(pole) * xr + np.cos(pole) * zr
    lon = np.rad2deg(np.arctan2(yr, xg)).astype(np.float32)
    lat = np.rad2deg(np.arcsin(np.clip(zg, -1, 1))).astype(np.float32)
    times = np.arange(nt) * 86400.0
    I = np.linspace(0, 2 * np.pi, nx, dtype=np.float32)[None, None, None, :]
    J = np.linspace(0, 2 * np.pi, ny, dtype=np.float32)[None, None, :, None]
    T = np.arange(nt, dtype=np.float32)[:, None, None, None]
    shape = (nt, nz, ny, nx)
    K = (np.float32(1.0) - np.float32(0.6) * np.linspace(0, 1, nz, dtype=np.float32))[None, :, None, None]  # weaker flow at depth

    def noise():
        return rng.random(shape, dtype=np.float32) * np.float32(0.1) - np.float32(0.05)

    U = ((np.float32(0.5) * np.sin(3 * I + 0.4 * T) * np.cos(2 * J) + np.float32(0.2) * np.cos(4 * J)) * K + noise()).astype(np.float32)
    V = ((np.float32(0.5) * np.cos(2 * I) * np.sin(3 * J + 0.3 * T) + np.float32(0.2) * np.sin(5 * I)) * K + noise()).astype(np.float32)
    depth = W = None
    if nz > 1:
        depth = (5000.0 * np.linspace(0.0, 1.0, nz) ** 1.7).astype(np.float32)
        W = ((np.float32(2e-3) * np.sin(2 * I) * np.sin(3 * J) * np.cos(np.float32(0.5) * T)) * K + np.float32(1e-2) * noise()).astype(np.float32)
    return dict(lon=lon, lat=lat, depth=depth, times=times, U=U, V=V, W=W, mesh="spherical", interp="cgrid_velocity",
                padding=("low", "low", "high"))  # fmt: skip


def c3_particles(field, n, seed):
    """uniform over the interior of the mesh: random cell + bilinear blend of its corners"""
    rng = np.random.default_rng(seed)
    lon, lat = field["lon"].astype(np.float64), field["lat"].astype(np.float64)
    ny, nx = lon.shape
    jj, ii = rng.uniform(8, ny - 9, n), rng.uniform(8, nx - 9, n)
    j0, i0 = jj.astype(np.int64), ii.astype(np.int64)
    fj, fi = jj - j0, ii - i0

    def bl(a):
        return ((1 - fj) * (1 - fi) * a[j0, i0] + (1 - fj) * fi * a[j0, i0 + 1] + fj * fi * a[j0 + 1, i0 + 1]
                + fj * (1 - fi) * a[j0 + 1, i0])  # fmt: skip

    depth = field.get("depth")
    z = np.zeros(n) if depth is None else rng.uniform(float(depth[1]), float(depth[-2]), n)
    return dict(x=bl(lon), y=bl(lat), z=z, t=np.zeros(n))


def _hash_noise(t, z, y, x, salt):
    """deterministic noise in [-0.05, 0.05) from GLOBAL indices (so neighbouring slabs agree on halo columns)"""
    h = np.sin(t * 12.9898 + z * 78.233 + y * 37.719 + x * 4.1414 + salt) * 43758.5453
    return ((h - np.floor(h)) * 0.1 - 0.05).astype(np.float32)


def c5_slab(rank, world, halo, nx=4320, ny=2160, nz=50, nt=2):
    """config 5: rectilinear 1/12 deg x 50 levels field, THIS RANK'S X-slab only (columns lo..hi of the global
    axis incl. halo); analytic modes + index-hashed noise, so every rank can build its slab independently."""
    from parcels_b200.distributed import slab_plan

    lon = np.linspace(-180.0, 180.0, nx)
    lat = np.linspace(-80.0, 80.0, ny)
    depth = 5500.0 * (np.linspace(0.0, 1.0, nz) ** 1.8)
    times = np.arange(nt) * 86400.0
    plan = slab_plan(lon, world, halo)[rank]
    lo, hi = plan["lo"], plan["hi"]
    xi = np.arange(lo, hi + 1, dtype=np.float64)[None, None, None, :]
    yi = np.arange(ny, dtype=np.float64)[None, None, :, None]
    zi = np.arange(nz, dtype=np.float64)[None, :, None, None]
    ti = np.arange(nt, dtype=np.float64)[:, None, None, None]
    X, Y, Z = 2 * np.pi * xi / (nx - 1), 2 * np.pi * yi / (ny - 1), zi / (nz - 1)
    U = (np.sin(3 * X + 0.3 * ti) * np.cos(2 * Y) * (1 - 0.5 * Z) * 0.6 + np.cos(5 * Y + ti) * 0.3).astype(np.float32)
    U = U + _hash_noise(ti, zi, yi, xi, 0.1)
    V = (np.cos(2 * X + 0.2 * ti) * np.sin(4 * Y) * (1 - 0.3 * Z) * 0.6 + np.sin(3 * X) * 0.25).astype(np.float32)
    V = V + _hash_noise(ti, zi, yi, xi, 1.7) + np.zeros_like(U)
    W = ((np.sin(2 * X) * np.sin(3 * Y) * np.sin(np.pi * Z) * np.cos(0.5 * ti) * 0.9).astype(np.float32)
         + _hash_noise(ti, zi, yi, xi, 2.9)) * np.float32(1e-3)  # fmt: skip
    return dict(lon=lon, lat=lat, depth=depth, times=times, U=np.ascontiguousarray(U), V=np.ascontiguousarray(V),
                W=np.ascontiguousarray(W.astype(np.float32)), lo=lo, hi=hi, plan=plan)


# name -> spec.  bytes: algorithmic bytes per particle-step (SURVEY.md 8d / BASELINE.md 4)
NOTE_AGRID = ("no-reuse byte model: the per-lane corner cache serves most samples on chip, real DRAM traffic is `traffic`; the kernel "
              "is fp64-issue- and refill-latency-bound, not HBM-bound (profiles/README.md)")
WORKLOADS = {
    "ns": dict(field=ns_field, fkw=dict(nx=4320, ny=2160, nz=50, nt=3), particles=c2_particles, n=10_000_000, dt=600.0,
               nsteps=144, kernels=["AdvectionRK4_3D"], bytes=832, device_field=True, ulp=8, roofline_note=NOTE_AGRID,
               desc="BASELINE.json north_star target -- AdvectionRK4_3D, 1e7 particles on a 1/12 deg rectilinear A-grid "
                    "4320x2160x50 T=3 f32 U,V,W (16.8 GB), f64 axes, spherical"),
    "ns_dense": dict(field=ns_field, fkw=dict(nx=4320, ny=2160, nz=50, nt=3), particles=dense_particles, n=10_000_000, dt=600.0,
                     nsteps=144, kernels=["AdvectionRK4_3D"], bytes=832, device_field=True, ulp=8, roofline_note=NOTE_AGRID,
                     desc="dense release on the north-star field: 1e7 particles in a 4 deg x 4 deg x 200 m patch of the 1/12 deg "
                          "rectilinear A-grid (hundreds of particles per cell), AdvectionRK4_3D"),
    "ns_small": dict(field=ns_field, fkw=dict(nx=480, ny=240, nz=20, nt=3), particles=c2_particles, n=200_000, dt=600.0,
                     nsteps=144, kernels=["AdvectionRK4_3D"], bytes=832, device_field=True, ulp=2,
                     desc="small functional variant of ns (480x240x20)"),
    "c2": dict(field=c2_field, fkw=dict(nx=1440, ny=720, nz=50, nt=3), particles=c2_particles, n=1_000_000, dt=600.0,
               nsteps=144, kernels=["AdvectionRK4_3D"], bytes=832, ulp=2, roofline_note=NOTE_AGRID,
               desc="BASELINE.json configs[1] -- AdvectionRK4_3D, 1e6 particles, rectilinear A-grid 1440x720x50 T=3 f32 U,V,W, "
                    "f64 axes, spherical"),
    "c2_small": dict(field=c2_field, fkw=dict(nx=360, ny=180, nz=20, nt=3), particles=c2_particles, n=100_000, dt=600.0,
                     nsteps=144, kernels=["AdvectionRK4_3D"], bytes=832, ulp=2, desc="small functional variant of c2"),
    "c3": dict(field=c3_field, fkw=dict(nx=1442, ny=1021, nt=3), particles=c3_particles, n=10_000_000, dt=3600.0,
               nsteps=48, kernels=["AdvectionRK4"], bytes=320, ulp=8, ulp_quantile=0.999,
               roofline_note="not HBM-bound: 9 double-precision sin/cos + 5 sqrt + ~8 divisions per sample are the reference's own "
                             "arithmetic (profiles/README.md: DRAM < 1 % of peak, cos+sin a quarter of the executed instructions)",
               desc="BASELINE.json configs[2] -- AdvectionRK4, 1e7 particles, curvilinear C-grid ORCA025 shape 1442x1021 T=3, "
                    "f32 lon/lat, CGrid_Velocity + hint/spatial-hash search, spherical"),
    "c3_3d": dict(field=c3_field, fkw=dict(nx=1442, ny=1021, nt=2, nz=31), particles=c3_particles, n=10_000_000, dt=3600.0,
                  nsteps=24, kernels=["AdvectionRK4_3D"], bytes=384, ulp=8, ulp_quantile=0.999,
                  desc="SURVEY 8 row f-4 -- AdvectionRK4_3D on the curvilinear C-grid of ORCA025 shape with 31 depth levels "
                       "(1442x1021x31 T=2 f32 U,V,W, 1.1 GB), 1e7 particles, CGrid_Velocity + W linear between the Z faces"),
    "c3_orca12": dict(field=c3_field, fkw=dict(nx=4322, ny=3059, nt=2), particles=c3_particles, n=10_000_000, dt=1200.0,
                      nsteps=48, kernels=["AdvectionRK4"], bytes=320, ulp=8, ulp_quantile=0.999,
                      desc="SURVEY 8 row f-4 -- AdvectionRK4 on a curvilinear C-grid of ORCA12 shape 4322x3059 (13.2 M faces in the "
                           "spatial hash) T=2, 1e7 particles"),
    "c3_small": dict(field=c3_field, fkw=dict(nx=362, ny=292, nt=3), particles=c3_particles, n=200_000, dt=3600.0,
                     nsteps=48, kernels=["AdvectionRK4"], bytes=320, ulp=8, desc="small functional variant of c3"),
    "c4": dict(field=c2_field, fkw=dict(nx=1440, ny=720, nz=50, nt=3), particles=c2_particles, n=10_000_000, dt=600.0,
               nsteps=144, kernels=["AdvectionRK4_3D", "DiffusionUniformKh"], bytes=832, kh=(100.0, 50.0), ulp=16,
               roofline_note=NOTE_AGRID,
               desc="BASELINE.json configs[3] -- fused AdvectionRK4_3D + DiffusionUniformKh (Kh 100/50 m2/s), 1e7 particles on the "
                    "config-2 field"),
    "c4_small": dict(field=c2_field, fkw=dict(nx=360, ny=180, nz=20, nt=3), particles=c2_particles, n=100_000, dt=600.0,
                     nsteps=144, kernels=["AdvectionRK4_3D", "DiffusionUniformKh"], bytes=832, kh=(100.0, 50.0), ulp=4,
                     desc="small functional variant of c4"),
}  # fmt: skip
C5 = {"c5": dict(dims=dict(nx=4320, ny=2160, nz=50, nt=2), n=12_500_000), "c5_small": dict(dims=dict(nx=432, ny=216, nz=20, nt=2), n=200_000)}


def config_block(name, w, n_per_gpu):
    """`config` of the JSON line: what BOTH arms run (the reference arm prints the same dict)."""
    fbytes = {"ns": 16.8, "ns_dense": 16.8, "c2": 1.87, "c4": 1.87, "c3": 0.035, "c3_3d": 1.1, "c3_orca12": 0.21}.get(name)
    return {
        "workload": f"{name}: {w['desc']}; dt={w['dt']:g} s x {w['nsteps']} dt-steps per pass",
        "kernels": w["kernels"] + ["DeleteParticle"],
        "particles_per_gpu": n_per_gpu, "dt_steps_per_pass": w["nsteps"],
        "l2_policy": "inputs larger than L2" + (f" ({fbytes} GB field" if fbytes else " (field") + f", {52 * n_per_gpu / 1e6:.0f} MB particle SoA; "
                     "particles re-seeded every pass)",
    }  # fmt: skip


class ClockSampler:
    """nvidia-smi SM clock + throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")  # fmt: skip

    def __init__(self, index=0):
        self.index, self.samples, self._stop = index, [], threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()  # fmt: skip
                if out:
                    self.samples.append([s.strip() for s in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.05)

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.samples)}  # fmt: skip


def dump_outputs(out_dir, name, d, input_ids, max_bytes):
    """Write the particle set ``d`` as ParticleSet.execute hands it back (deleted particles dropped, order kept) to
    ``out_dir/<name>_<variable>.npy``.  Integer variables are stored as float64 (exact below 2**53).  If the set is larger than
    ``max_bytes``, only the survivors of a fixed seeded sample of the released particles (``input_ids``) are written, so that two
    builds write the same rows wherever they agree on which particles survive."""
    from parcels_b200.statuscodes import StatusCode

    rows = np.flatnonzero(d["state"] != StatusCode.Delete)
    m = max_bytes // (8 * sum(int(np.prod(v.shape[1:])) for v in d.values()))  # (at most 8 bytes a value)
    if len(rows) > m:
        sample = input_ids[np.random.default_rng(0).choice(len(input_ids), size=min(m, len(input_ids)), replace=False)]
        rows = rows[np.isin(d["particle_id"][rows], sample)]
    os.makedirs(out_dir, exist_ok=True)
    for k, v in d.items():
        v = v[rows]
        np.save(os.path.join(out_dir, f"{name}_{k}.npy"), v if v.dtype.kind == "f" else v.astype(np.float64))


def measured_peak():
    try:
        m = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(m["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def dram_traffic_per_launch(workload):
    """dram__bytes_read+write per launch from the committed ncu capture (profiles/roofline_traffic.json), or None."""
    try:
        j = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
        return j.get(workload)
    except Exception:
        return None


def ncu_limiter(workload):
    """Issue-slot / FP64-pipe utilisation of the workload's kernel from the committed ncu capture (same file), or None: the
    byte model of `roofline` assumes no reuse, these say what the kernel is actually bound by."""
    try:
        j = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
        return (j.get("limiter") or {}).get(workload)
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------
# CPU legs (oracle port of the reference path): cpu_baseline / parity_sample and the reference arm
# ------------------------------------------------------------------------------------------------
def _oracle_fieldset(name, w, field):
    """Oracle-side field description, built once per workload and process (the curvilinear spatial hash is one-time
    grid setup in the reference too, _core/basegrid.py:192-216, and is kept out of the timed passes)."""
    from oracle import parcels_oracle as po

    key = ("ofs", name)
    if key not in _G:
        pad = field.get("padding", ("low", "low", "high"))
        g = po.OGrid(field["lon"], field["lat"], field["depth"], mesh=field["mesh"], offsets=tuple(int(p == "low") for p in pad))
        consts = {"Kh_zonal": w["kh"][0], "Kh_meridional": w["kh"][1]} if "kh" in w else None
        _G[key] = po.OFieldSet(g, field["U"], field["V"], field["W"], time=field["times"], interp=field.get("interp", "linear"),
                               constants=consts)  # fmt: skip
        if g.curvilinear:
            from oracle import curvilinear_oracle as co

            co.get_hash(g)
    return _G[key]


def _oracle_pass(name, w, field, parts, nsteps=None, normal=None):
    """One oracle pass over ``parts``: returns (particle dict after the pass, particle-steps, seconds)."""
    from oracle import parcels_oracle as po

    fs = _oracle_fieldset(name, w, field)
    pd = po.create_particle_data(parts["x"], parts["y"], parts["z"], parts["t"], ngrids=fs.ngrids)
    kmap = {"AdvectionRK4_3D": po.AdvectionRK4_3D, "AdvectionRK4": po.AdvectionRK4}
    kern = [po.DiffusionUniformKh(normal) if k == "DiffusionUniformKh" else kmap[k] for k in w["kernels"]] + [po.DeleteOnError]
    t0 = time.perf_counter()
    steps = po.pset_execute(pd, fs, kern, w["dt"], runtime=w["dt"] * (nsteps or w["nsteps"]))
    return pd, steps, time.perf_counter() - t0


def _c_port_pass(w, field, parts):
    """strong CPU baseline: the C + OpenMP restatement (oracle/advect_rk4_3d.c) on all host cores"""
    from oracle import c_port
    from oracle import parcels_oracle as po

    pd = po.create_particle_data(parts["x"], parts["y"], parts["z"], parts["t"])
    g = po.OGrid(field["lon"], field["lat"], field["depth"], mesh=field["mesh"])
    c_port.advect_rk4_3d(lon=field["lon"], lat=field["lat"], depth=field["depth"], time=field["times"], U=field["U"], V=field["V"],
                         W=field["W"], spherical=g.spherical, deg2m=g.deg2m, pdata=dict(pd), dt=w["dt"], endtime=w["dt"])  # warm-up: 1 step
    pd = po.create_particle_data(parts["x"], parts["y"], parts["z"], parts["t"])
    t0 = time.perf_counter()
    steps = c_port.advect_rk4_3d(lon=field["lon"], lat=field["lat"], depth=field["depth"], time=field["times"], U=field["U"],
                                 V=field["V"], W=field["W"], spherical=g.spherical, deg2m=g.deg2m, pdata=pd, dt=w["dt"],
                                 endtime=w["dt"] * w["nsteps"])  # fmt: skip
    return steps, time.perf_counter() - t0


def parity_and_cpu_baseline(name, w, field, fs, device, n_sample, seed_gpu=1234):
    """The GPU (public API) and the oracle advect the SAME ``n_sample`` particles of the workload for one pass; the oracle's
    time is the cpu_baseline.  Bit-exact: surviving ids, states, times, cell indices; positions within ``w['ulp']`` float32 ulp."""
    import parcels_b200 as pb
    from engine_run import ulp_diff_f32

    parts = w["particles"](field, n_sample, 1)
    normal = None
    if "DiffusionUniformKh" in w["kernels"]:
        from philox_ref import device_normals  # the engine's own Wiener increments (pb_debug_normals) for the oracle

        st = {"it": 0}

        def normal(view):
            zx, zy = device_normals(seed_gpu, 1, st["it"], view.particle_id, device=device)  # (seed; call 1 of a fresh ParticleSet, iteration, id)
            st["it"] += 1
            return zx, zy

    pd, steps, secs = _oracle_pass(name, w, field, parts, normal=normal)
    ps = pb.ParticleSet(fs, x=parts["x"], y=parts["y"], z=parts["z"], t=parts["t"], device=device, seed=seed_gpu)
    kernels = [getattr(pb, k) for k in w["kernels"]] + [pb.DeleteParticle]
    ps.execute(kernels, dt=w["dt"], runtime=w["dt"] * w["nsteps"])
    d = ps._data
    same_ids = d["particle_id"].shape == pd["particle_id"].shape and bool(np.array_equal(d["particle_id"], pd["particle_id"]))
    out = {"n": int(n_sample), "dt_steps": w["nsteps"], "ids_equal": same_ids, "survivors_gpu": int(len(d["x"])),
           "survivors_oracle": int(len(pd["x"])), "deleted_gpu": int(n_sample - len(d["x"])), "deleted_oracle": int(n_sample - len(pd["x"])),
           "tolerance_ulp": w["ulp"],
           "tolerance_note": "float32 ulp of max(|coordinate|, 0.05) after the whole pass; last-place differences of CUDA's vs libm's cos / sin "
                             "flip float32 roundings of single steps and grow along the trajectories"}  # fmt: skip
    if same_ids:
        out["state_mismatch"] = int(np.count_nonzero(d["state"] != pd["state"]))
        out["t_mismatch"] = int(np.count_nonzero(d["t"] != pd["t"]))
        out["ei_mismatch"] = int(np.count_nonzero(d["ei"] != pd["ei"]))
        # ulp of coordinates that cross zero: measured at the size of one step's displacement (tests/engine_run.py)
        ulps = {k: float(ulp_diff_f32(d[k], pd[k], floor=0.05).max()) if len(d[k]) else 0.0 for k in "xyz"}
        out["max_ulp"] = max(ulps.values())
        out["max_ulp_xyz"] = [ulps["x"], ulps["y"], ulps["z"]]
        worst = np.maximum.reduce([ulp_diff_f32(d[k], pd[k], floor=0.05) for k in "xyz"]) if len(d["x"]) else np.zeros(0)
        out["bit_identical"] = int(np.count_nonzero(worst == 0))
        out["outside_tolerance"] = int(np.count_nonzero(worst > w["ulp"]))
        exact = out["state_mismatch"] == 0 and out["t_mismatch"] == 0 and out["ei_mismatch"] == 0
        if w.get("ulp_quantile"):
            # C-grid velocities are DISCONTINUOUS across cell faces (tangential component): a stage sample within one ulp of a face
            # turns a last-place difference (CUDA vs libm sin / cos) into a metre-scale one.  The position bound therefore holds for
            # all but a stated fraction of the sample (DESIGN.md 2, measured: 11 of 20 000 after 48 steps, largest 27 ulp)
            out["ok"] = bool(exact and out["outside_tolerance"] <= (1 - w["ulp_quantile"]) * len(worst))
            out["tolerance_quantile"] = w["ulp_quantile"]
        else:
            out["ok"] = bool(exact and out["max_ulp"] <= w["ulp"])
    else:
        a, b = set(d["particle_id"].tolist()), set(pd["particle_id"].tolist())
        out["only_gpu"], out["only_oracle"] = len(a - b), len(b - a)
        out["ok"] = False
    cpu = {"value": steps / secs, "unit": "particle-steps/s", "cores": 1, "kind": "port",
           "sample": f"{n_sample} particles of the same workload, {w['nsteps']} dt-steps, NumPy oracle port of the reference path ({secs:.1f} s)"}  # fmt: skip
    return out, cpu


def _worker(args):
    seed, n, m = args
    name, w, field = _G["name"], _G["w"], _G["field"]
    _, steps, _ = _oracle_pass(name, w, field, w["particles"](field, n, seed), nsteps=m)
    return steps


def run_reference_arm(a, name, w, field):
    """Reference arm: the reference's algorithm (oracle port) on all host cores (rank 0 only).  Every process advects a FIXED
    ``--ref-particles-per-core`` particles (flat-rate regime of the NumPy port: >= 1e4 per batch); the number of dt-steps of one
    bench step is what is scaled to the time budget (``--ref-step-seconds``), calibrated on a probe AFTER the pool is warm."""
    import multiprocessing as mp

    cores = len(os.sched_getaffinity(0))
    per = max(int(a.ref_particles_per_core), 1)
    _G["name"], _G["w"], _G["field"] = name, w, field
    _oracle_fieldset(name, w, field)  # incl. the spatial hash: built once, before forking
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        def one_pass(k, m):
            t0 = time.perf_counter()
            steps = sum(pool.map(_worker, [(1000 * k + c, per, m) for c in range(cores)]))
            return steps, time.perf_counter() - t0

        one_pass(998, 1)  # pool start-up, imports, first-touch of the shared field pages
        s0, t0_ = one_pass(999, 2)
        m = int(np.clip(round(a.ref_step_seconds * (s0 / t0_) / (cores * per)), 2, w["nsteps"]))
        for k in range(a.warmup):
            one_pass(k, m)
        tot_steps, tot_t = 0, 0.0
        for k in range(a.steps):
            s, t = one_pass(100 + k, m)
            tot_steps += s
            tot_t += t
    v = tot_steps / tot_t
    sample = (f"{cores} processes x {per} particles x {m} dt-steps per bench step (of the workload's {w['nsteps']}; same field, dt, "
              "kernels; NumPy oracle port of the reference path, one process per host core)")
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "particle-steps/s", "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * tot_t / max(a.steps, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_block(name, w, a.particles or w["n"]),
        "cpu_baseline": {"value": v, "unit": "particle-steps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "particle-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }  # fmt: skip
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def build_field(name, w, *, device=None, host=False, threads=None):
    if w.get("device_field"):
        return w["field"](device=None if host else device, threads=threads, **w["fkw"])
    return w["field"](**w["fkw"])


def run_gpu_workload(a, name, *, rank, local_rank, world, dist, steps, warmup, with_e2e=True, with_cpu=True, field_cache=None):
    """Measure one workload on this rank's GPU: device-resident arm, end-to-end arm, and (rank 0, N = 1) the parity sample.
    Returns the dict of the JSON line's workload-specific keys (rank 0) or None."""
    import torch

    import parcels_b200 as pb
    from parcels_b200.kernels import SCHEMES

    w = WORKLOADS[name]
    n_per_gpu = a.particles or w["n"]
    dt, nsteps = w["dt"], w["nsteps"]
    torch.cuda.set_device(local_rank)
    cores = len(os.sched_getaffinity(0))
    field_cache = {} if field_cache is None else field_cache
    fkey = (w["field"].__name__, tuple(sorted(w["fkw"].items())))
    if fkey in field_cache:
        field = field_cache[fkey]
    else:
        field = build_field(name, w, device=local_rank)
        field_cache.clear()  # one field at a time in memory
        field_cache[fkey] = field
    fs = pb.FieldSet.from_arrays(lon=field["lon"], lat=field["lat"], depth=field["depth"], time=field["times"],
                                 U=field["U"], V=field["V"], W=field["W"], mesh=field["mesh"],
                                 interp_method=field.get("interp", "linear"),
                                 padding=field.get("padding", ("low", "low", "high")))  # fmt: skip
    diffusion = "DiffusionUniformKh" in w["kernels"]
    if diffusion:
        fs.add_constant_field("Kh_zonal", w["kh"][0], mesh=field["mesh"])
        fs.add_constant_field("Kh_meridional", w["kh"][1], mesh=field["mesh"])
    parts = w["particles"](field, n_per_gpu, 1 + rank)  # weak scaling: every rank owns its own shard
    if a.sorted and np.ndim(field["lon"]) == 1:
        cell = np.searchsorted(field["lon"], parts["x"]).astype(np.int64)
        cell += len(field["lon"]) * np.searchsorted(field["lat"], parts["y"])
        if field["depth"] is not None:
            cell += len(field["lon"]) * len(field["lat"]) * np.searchsorted(field["depth"], parts["z"])
        order = np.argsort(cell, kind="stable")
        parts = {k: v[order] for k, v in parts.items()}
    ps = pb.ParticleSet(fs, x=parts["x"], y=parts["y"], z=parts["z"], t=parts["t"], device=local_rank, seed=1234)
    init = {k: v.copy() for k, v in ps._data.items()}
    eng = fs.engine(local_rank)
    runtime = dt * nsteps
    kernels = [getattr(pb, k) for k in w["kernels"]] + [pb.DeleteParticle]

    def barrier():
        eng.synchronize()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    def reduce(x, op):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(t, op=getattr(dist.ReduceOp, op))
        return float(t.item())

    # ---- device-resident arm: particles + fields in HBM; per step: restore snapshot + ONE kernel ----
    ei_last = np.ascontiguousarray(init["ei"][:, -1])
    eng.upload_particles(init, ei_last)
    eng.snapshot()
    plan = pb.particleset.KernelPlan(kernels, fs)
    args = eng.make_args(SCHEMES[w["kernels"][0]], dt, runtime, diffusion=diffusion, delete_on_error=True, kh=plan.kh,
                         kh_spherical=plan.kh_spherical, kh_deg2m=plan.kh_deg2m, seed=1234, rng_call=1,
                         hint_all_zero=fs.grid.curvilinear)  # fmt: skip

    def resident_step():
        eng.restore()
        eng.advect_async(args)

    for _ in range(warmup):
        resident_step()
    barrier()
    ksum, psteps = 0.0, 0
    with ClockSampler(local_rank) as clk:
        eng.timer_begin()
        t0 = time.perf_counter()
        for _ in range(steps):
            resident_step()
            rep = eng.last_report()  # waits for this step's kernel (the report is read back every step)
            ksum += rep["kernel_ms"]
            psteps += rep["particle_steps"]
        dev_ms = eng.timer_end_ms()
        barrier()
        wall_ms = 1e3 * (time.perf_counter() - t0)
    dev_ms = reduce(dev_ms, "MAX")
    total_steps = reduce(psteps, "SUM")
    value = total_steps / (dev_ms * 1e-3)
    kernel_ms = ksum / steps
    steps_per_launch = psteps / steps
    if a.dump_outputs and rank == 0:
        last = eng.download_all(ngrids=len(fs.gridset))
        last["dt"][:] = dt
        dump_outputs(a.dump_outputs, name, last, init["particle_id"], a.dump_bytes)
        del last

    # ---- end-to-end arm: public API with host arrays; H2D + D2H of the particle SoA every step ----
    e2e = None
    if with_e2e:
        k_e2e = steps
        # one page-locked host input batch (inputs come from pinned host memory), refilled from `init` before every pass, outside
        # the timed region
        batch = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory().numpy() for k, v in init.items()}

        def e2e_pass():
            for k, v in init.items():
                np.copyto(batch[k], v)
            ps._data = dict(batch)  # (execute leaves shortened views of these arrays in ps._data when particles are deleted)
            barrier()
            t0 = time.perf_counter()
            ps.execute(kernels, dt=dt, runtime=runtime)
            result = ps._data  # device -> host read of the step's result (the particle SoA after the pass)
            assert not ps._host_stale and len(result["x"]) > 0
            barrier()
            return time.perf_counter() - t0

        if a.pipeline >= 0:
            ps.pipeline_chunks = a.pipeline
        ps.eager_host = True  # this arm reads the result on the host after every pass: the download belongs to the (pipelined) call
        for _ in range(warmup):
            e2e_pass()
        e2e_steps, e2e_s = 0, 0.0
        for _ in range(k_e2e):
            e2e_s += e2e_pass()
            e2e_steps += ps.last_report["particle_steps"]
        e2e_s = reduce(e2e_s, "MAX")
        n = n_per_gpu
        e2e = {"value": reduce(e2e_steps, "SUM") / e2e_s, "unit": "particle-steps/s", "h2d_bytes_per_step": n * (6 * 4 + 8 + 4 + 4 + 8),
               "d2h_bytes_per_step": n * (6 * 4 + 8 + 4 + 4), "steps": k_e2e, "pipeline_chunks": ps.pipeline_chunks, "eager_host": True,
               "api": f"parcels_b200.ParticleSet.execute([{', '.join(w['kernels'])}, DeleteParticle], dt={dt:g}, runtime={runtime:g})"}  # fmt: skip
        del batch

    out = None
    if rank == 0:
        peak, peak_src = measured_peak()
        achieved = w["bytes"] * steps_per_launch / (kernel_ms * 1e-3) / 1e9
        out = {
            "value": value, "ms_per_step": dev_ms / steps, "e2e": e2e, "gpu_launches": steps,
            "measured": {"wall_ms_per_step": wall_ms / steps, "kernel_ms_per_launch": kernel_ms,
                         "corner_cache_refills_per_launch": rep["cache_refills"], "deleted_per_launch": rep["n_deleted"],
                         "kernel_variant": rep.get("kernel_variant"), "particles_per_gpu": n_per_gpu},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": dram_traffic_per_launch(name), "peak_source": peak_src,
                         "algorithmic_bytes_per_particle_step": w["bytes"], "particle_steps_per_launch": steps_per_launch,
                         **({"note": w["roofline_note"]} if "roofline_note" in w else {}),
                         **({"limiter_from_ncu": ncu_limiter(name)} if ncu_limiter(name) else {})},
            "clocks": clk.summary(),
        }  # fmt: skip
        if with_cpu and world == 1:
            hfield = field
            if w.get("device_field"):
                # the oracle needs the field on the host: generated there by the same float32 operations -- one plane of each is
                # compared with the field in HBM (the whole point: both sides advect the SAME field)
                hfield = build_field(name, w, host=True, threads=cores)
                for comp in "UVW":
                    lvl, z = field[comp].shape[0] - 1, field[comp].shape[1] // 2
                    same = bool(np.array_equal(field[comp][lvl, z].cpu().numpy(), hfield[comp][lvl, z]))
                    out.setdefault("field_check", {})[comp] = same
            par, cpu = parity_and_cpu_baseline(name, w, hfield, fs, local_rank, a.cpu_sample)
            if "field_check" in out:
                par["field_planes_equal"] = all(out.pop("field_check").values())
                par["ok"] = bool(par["ok"] and par["field_planes_equal"])
            out["parity_sample"], out["cpu_baseline"] = par, cpu
            if w["kernels"] == ["AdvectionRK4_3D"] and field.get("interp", "linear") == "linear":
                nt_omp = os.environ.get("OMP_NUM_THREADS")
                os.environ["OMP_NUM_THREADS"] = str(cores)  # (torchrun exports 1; the C leg is an OpenMP loop over particles)
                big = w["particles"](hfield, min(n_per_gpu, 400_000), 1)
                s2, t2 = _c_port_pass(w, hfield, big)
                if nt_omp is None:
                    os.environ.pop("OMP_NUM_THREADS", None)
                else:
                    os.environ["OMP_NUM_THREADS"] = nt_omp
                out["cpu_baseline_strong"] = {"value": s2 / t2, "unit": "particle-steps/s", "cores": cores, "kind": "port",
                                              "sample": f"{len(big['x'])} particles, {nsteps} dt-steps, C + OpenMP restatement "
                                                        f"(oracle/advect_rk4_3d.c, same arithmetic, {cores} threads; {t2:.1f} s)"}  # fmt: skip
            _G.pop(("ofs", name), None)
            del hfield
    fs.release()
    del ps, init, fs
    torch.cuda.empty_cache()
    return out


def run_decomposed_bench(a, rank, local_rank, world, dist, workload="c5"):
    """Mode D bench (config 5): field cut into X-slabs, particles migrate over NCCL.  One bench step = one
    Kernel.execute over the decomposed field (advect kernels + migration rounds + all-to-all-v).  Returns the `mode_d` block."""
    import torch

    import parcels_b200 as pb
    from parcels_b200 import distributed as D
    from parcels_b200.particle import create_particle_data

    dims = C5[workload]["dims"]
    n_per_gpu = a.particles_d or C5[workload]["n"]
    dt, nsteps, halo = 600.0, 48, 3
    f = c5_slab(rank, world, halo, **dims)
    fs = pb.FieldSet.from_arrays(lon=f["lon"][f["lo"] : f["hi"] + 1].copy(), lat=f["lat"], depth=f["depth"], time=f["times"],
                                 U=f["U"], V=f["V"], W=f["W"], mesh="spherical", xdim=f["lon"].size - 1)  # fmt: skip
    dfs = D.DecomposedFieldSet.from_slab(fs, f["plan"], rank=rank, world=world, device=local_rank)
    p2p_error = ""
    if a.mode_d_transport == "p2p":  # in-kernel migration over peer memory: the advection kernel delivers the leavers itself
        if not D.connect_p2p(dfs, dist, max(n_per_gpu // 8, 4096)):
            p2p_error = dfs.p2p_error  # every rank agreed to stay on the collectives
    rng = np.random.default_rng(100 + rank)
    b = f["plan"]["bounds"]
    # every rank seeds its particles inside its own slab (as a domain-decomposed application would); whatever
    # leaves the slab during the pass migrates over NCCL
    n = n_per_gpu
    x = rng.uniform(max(b[rank], -175.0), min(b[rank + 1], 175.0), n)
    y, z = rng.uniform(-70, 70, n), rng.uniform(5, 5000, n)
    pid = np.arange(n, dtype=np.int64) + rank * n
    runtime = dt * nsteps
    kernels = [pb.AdvectionRK4_3D, pb.DeleteParticle]
    dev = f"cuda:{local_rank}"
    steps, warmup = a.steps, a.warmup

    eng = dfs.engine
    plan = D.decomposed_plan(dfs, kernels)

    def fresh():
        return create_particle_data(nparticles=n, ngrids=1, initial=dict(x=x, y=y, z=z, t=np.zeros(n), particle_id=pid))  # input batch

    def sync_all():
        eng.synchronize()
        torch.cuda.synchronize()
        dist.barrier()

    # ---- device-resident arm: the shard is in HBM (snapshot); per pass: restore + advect kernels + migration rounds ----
    D.upload_decomposed(dfs, fresh(), dt)
    eng.snapshot()

    def resident_pass():
        eng.restore()
        sync_all()
        t0 = time.perf_counter()
        stats = D.run_decomposed_resident(dfs, plan, dt, runtime, dist)
        sync_all()
        return time.perf_counter() - t0, stats

    for _ in range(warmup):
        resident_pass()
    tot_t, tot_steps, tot_mig, rounds, kms, xms = 0.0, 0, 0, 0, 0.0, 0.0
    for _ in range(steps):
        t, st = resident_pass()
        tot_t += D.allreduce_max(t, dist, dev)
        tot_steps += D.allreduce_sum(st["particle_steps"], dist, dev)
        tot_mig += D.allreduce_sum(st["migrated"], dist, dev)
        rounds = max(rounds, st["rounds"])
        kms += D.allreduce_max(st["kernel_ms"], dist, dev)
        xms += D.allreduce_max(st["exchange_ms"], dist, dev)
    n_after = D.allreduce_sum(eng.particle_count(), dist, dev)

    # ---- end-to-end arm: host particle arrays in, host arrays out (upload + rounds + download inside the timed region) ----
    k_e2e = steps
    e_t, e_steps = 0.0, 0
    for i in range(warmup + k_e2e):
        pdata = fresh()
        sync_all()
        t0 = time.perf_counter()
        out, stats = D.execute_decomposed(dfs, pdata, kernels, dt, runtime, dist)
        sync_all()
        if i >= warmup:
            e_t += D.allreduce_max(time.perf_counter() - t0, dist, dev)
            e_steps += D.allreduce_sum(stats["particle_steps"], dist, dev)
    fs.release()
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    peak, _ = measured_peak()
    value = tot_steps / tot_t
    kernel_rate = tot_steps / world / (kms * 1e-3)
    return {
        "value": value, "unit": "particle-steps/s", "ms_per_step": 1e3 * tot_t / steps, "steps": steps, "warmup": warmup,
        "workload": f"{workload}: BASELINE.json configs[4] -- AdvectionRK4_3D, rectilinear {dims['nx']}x{dims['ny']}x{dims['nz']} "
                    f"T={dims['nt']} f32 field DOMAIN-DECOMPOSED into {world} X-slabs (+{halo} halo columns), {n_per_gpu} "
                    f"particles/GPU seeded in the rank's own slab, migration "
                    f"{'inside the advection kernel over peer memory (CUDA IPC + NVLink)' if a.mode_d_transport == 'p2p' else 'by NCCL all-to-all-v'}"
                    f"; dt={dt:g} s x {nsteps} steps",
        "transport": st.get("transport"), **({"p2p_unavailable": p2p_error} if p2p_error else {}),
        "timed_region": "particles resident in HBM (restored from a snapshot every pass): advect kernels + migration rounds (p2p: records "
                        "stored into the new owner's inbox by the advection kernel over NVLink, one 2-value all-reduce + compact/append "
                        "per round; collective: classify / count all-gather / pack / all-to-all-v / unpack), wall clock between "
                        "barrier + synchronize, max over ranks",
        "e2e": {"value": e_steps / e_t, "unit": "particle-steps/s", "steps": k_e2e, "h2d_bytes_per_step": n * 48 * world,
                "d2h_bytes_per_step": n * 48 * world, "timed_region": "host particle arrays in, host arrays out"},
        "migrations_per_pass": tot_mig / steps, "advect_rounds_per_pass": rounds, "particles_after_pass": n_after,
        "kernel_ms_per_pass_max_rank": kms / steps, "collective_ms_per_pass_max_rank": xms / steps,
        "per_gpu_kernel_rate": kernel_rate, "kernel_frac_of_hbm_roofline": 832 * kernel_rate / 1e9 / peak,
    }  # fmt: skip


def decomposed_bitexact_check(rank, local_rank, world, dist, n=200_000, transport="p2p"):
    """Mode D over NCCL against ONE GPU, bit for bit (scripts/decomposed_check.py inside the bench, so that the driver's
    multi-GPU box exercises it): a small field cut into `world` slabs, many slab crossings."""
    import parcels_b200 as pb
    from parcels_b200 import distributed as D
    from parcels_b200.particle import create_particle_data

    f = c2_field(nx=240, ny=60, nz=12, nt=3)
    f["U"] *= np.float32(40.0)
    f["V"] *= np.float32(40.0)
    rng = np.random.default_rng(7)
    x, y, z = rng.uniform(-175, 175, n), rng.uniform(-70, 70, n), rng.uniform(5, 5000, n)
    dt, runtime = 600.0, 86400.0
    full = create_particle_data(nparticles=n, ngrids=1, initial=dict(x=x, y=y, z=z, t=np.zeros(n), particle_id=np.arange(n)))
    dfs = D.DecomposedFieldSet(lon=f["lon"], lat=f["lat"], depth=f["depth"], time=f["times"], U=f["U"], V=f["V"], W=f["W"],
                               mesh="spherical", rank=rank, world=world, halo_cells=3, device=local_rank)
    if transport == "p2p":
        D.connect_p2p(dfs, dist, n // 4)
    out, stats = D.execute_decomposed(dfs, D.shard_particles(full, rank, world), [pb.AdvectionRK4_3D, pb.DeleteParticle], dt, runtime, dist)
    tot = D.allreduce_sum(stats["migrated"], dist, device=f"cuda:{local_rank}")
    merged = D.gather_particles(out, dist, dst=0)
    dfs.fs.release()
    if rank != 0:
        return None
    order = np.argsort(merged["particle_id"], kind="stable")
    merged = {k: v[order] for k, v in merged.items()}
    fs = pb.FieldSet.from_arrays(lon=f["lon"], lat=f["lat"], depth=f["depth"], time=f["times"], U=f["U"], V=f["V"], W=f["W"], mesh="spherical")
    ps = pb.ParticleSet(fs, x=x, y=y, z=z, t=np.zeros(n), device=local_rank)
    ps.execute([pb.AdvectionRK4_3D, pb.DeleteParticle], dt=dt, runtime=runtime)
    ref = ps._data
    bad = [k for k in ("particle_id", "state", "t", "ei", "x", "y", "z") if not (merged[k].shape == ref[k].shape and np.array_equal(merged[k], ref[k]))]
    fs.release()
    return {"particles": n, "survivors": int(len(ref["x"])), "migrations": int(tot), "rounds": stats["rounds"], "backend": dist.get_backend(), "transport": stats["transport"],
            "bit_exact_vs_one_gpu": not bad, "mismatching_columns": bad}  # fmt: skip


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="ns", choices=list(WORKLOADS) + list(C5))
    ap.add_argument("--extras", default=None, help="comma-separated workloads measured as compact blocks under `extra` "
                                                   "(default: c2,c3,c4 with the default workload at N=1, none otherwise)")
    ap.add_argument("--particles", type=int, default=None, help="particles per GPU (default: the workload's)")
    ap.add_argument("--particles-d", type=int, default=None, help="particles per GPU of the mode-D block")
    ap.add_argument("--cpu-sample", type=int, default=20000, help="particles of the parity / cpu_baseline sample")
    ap.add_argument("--ref-particles-per-core", type=int, default=10000, help="reference arm: particles per process (fixed)")
    ap.add_argument("--ref-step-seconds", type=float, default=4.0, help="reference arm: target seconds per bench step")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip parity_sample / cpu_baseline (the oracle legs)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-mode-d", action="store_true", help="N > 1: skip the domain-decomposed block")
    ap.add_argument("--mode-d-timeout", type=float, default=0.0, help="N > 1: seconds the domain-decomposed block may take before the "
                    "mode R line is printed without it (default: max(900, 3 x the time the mode R part took))")
    ap.add_argument("--mode-d-transport", default="p2p", choices=["p2p", "collective"],
                    help="mode D: p2p = in-kernel migration over peer memory (CUDA IPC + NVLink), collective = NCCL all-to-all-v")
    ap.add_argument("--pipeline", type=int, default=-1,
                    help="chunks of the pipelined host-array path of the end-to-end arm (ParticleSet.pipeline_chunks; -1: the library default)")
    ap.add_argument("--sorted", action="store_true",
                    help="experiment: release the particles ordered by grid cell (z, y, x) instead of randomly -- measures what "
                         "spatial coherence between the lanes of a warp is worth (DESIGN.md 4, 'why not Morton-sort')")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the particle arrays the last device-resident pass of every workload of the line "
                         "left (rank 0) as DIR/<workload>_<variable>.npy, float32 / float64, a fixed sample of particles where the "
                         f"whole set would exceed {DUMP_BYTES >> 20} MB in all")
    a = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    name = a.workload

    if a.impl == "reference":
        if rank == 0:
            if name in C5:
                print(json.dumps({"impl": "reference", "unavailable": "config 5 (domain-decomposed) has no single-process CPU equivalent; "
                                                                       "its kernels and field are the ns workload's"}))  # fmt: skip
            else:
                w = WORKLOADS[name]
                run_reference_arm(a, name, w, build_field(name, w, host=True, threads=len(os.sched_getaffinity(0))))
        return

    import torch

    from oracle import c_port
    from parcels_b200 import _lib, build

    # the tree may be read-only: a library older than its sources is compiled into a temporary directory, never into the tree
    tmp = None
    if build.needs_build():
        tmp = tempfile.mkdtemp(prefix="parcels_b200_bench_")
        _lib.LIB_PATH = build.build(out=os.path.join(tmp, "libparcels_b200.so"))
    if c_port.needs_build():
        c_port.LIB = os.path.join(tmp or tempfile.mkdtemp(prefix="parcels_b200_bench_"), "liboracle_c.so")
    dist = None
    if world > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))

    if name in C5:
        if world < 2:
            raise SystemExit("workload c5 is the domain-decomposed mode: launch with torchrun on >= 2 GPUs")
        with ClockSampler(local_rank) as clk:
            md = run_decomposed_bench(a, rank, local_rank, world, dist, name)
        chk = decomposed_bitexact_check(rank, local_rank, world, dist, transport=a.mode_d_transport)
        dist.barrier()
        dist.destroy_process_group()
        if rank == 0:
            md["bitexact_check"] = chk
            line = {"metric": METRIC, "value": md["value"], "unit": "particle-steps/s", "n_gpus": world, "steps": md["steps"],
                    "warmup": md["warmup"], "ms_per_step": md["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                    "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": {"workload": md["workload"]},
                    "e2e": md["e2e"],
                    "gpu_launches": int(md["steps"] * md["advect_rounds_per_pass"] * 4), "mode_d": md, "clocks": clk.summary()}  # fmt: skip
            print(json.dumps(line))
        return

    w = WORKLOADS[name]
    extras = a.extras.split(",") if a.extras else (["c2", "c3", "c4"] if (name == "ns" and world == 1 and a.extras is None) else [])
    extras = [e for e in extras if e and e != name]
    if a.dump_outputs:
        a.dump_bytes = DUMP_BYTES // (1 + len(extras))  # an equal share of the budget for every workload of the line
    cache = {}
    t_main = time.perf_counter()
    main_out = run_gpu_workload(a, name, rank=rank, local_rank=local_rank, world=world, dist=dist, steps=a.steps, warmup=a.warmup,
                                with_e2e=not a.no_e2e, with_cpu=not a.no_cpu_baseline, field_cache=cache)  # fmt: skip
    extra_out = {}
    for e in extras:
        r = run_gpu_workload(a, e, rank=rank, local_rank=local_rank, world=world, dist=dist, steps=a.steps, warmup=a.warmup,
                             with_e2e=not a.no_e2e, with_cpu=not a.no_cpu_baseline, field_cache=cache)  # fmt: skip
        if r is not None:
            r["config"] = config_block(e, WORKLOADS[e], a.particles or WORKLOADS[e]["n"])
            extra_out[e] = r
    cache.clear()
    line = None
    if rank == 0:
        n_per_gpu = a.particles or w["n"]
        line = {
            "metric": METRIC, "value": main_out["value"], "unit": "particle-steps/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": main_out["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": config_block(name, w, n_per_gpu),
        }  # fmt: skip
        for k in ("e2e", "gpu_launches", "roofline", "measured", "parity_sample", "cpu_baseline", "cpu_baseline_strong", "clocks"):
            if k in main_out:
                line[k] = main_out[k]
        if a.sorted:
            line["measured"]["sorted_release"] = True
        if extra_out:
            line["extra"] = extra_out
    mode_d, watchdog = None, None
    if world > 1 and not a.no_mode_d:
        torch.cuda.empty_cache()
        # The mode R line is printed whatever happens in this block.  An exception is reported in the line; a rank that dies or
        # hangs would leave the others inside a collective for good, so a watchdog bounds the block: past the limit rank 0 prints
        # the mode R line with the reason and every rank leaves (the limit is generous: the block normally takes well under a
        # minute, and scales with what the mode R part -- full-field generation included -- took on this box).
        limit = a.mode_d_timeout or max(900.0, 3.0 * (time.perf_counter() - t_main))
        watchdog = threading.Timer(limit, _leave_mode_d, args=(line, limit))
        watchdog.daemon = True
        watchdog.start()
        try:
            mode_d = run_decomposed_bench(a, rank, local_rank, world, dist, "c5" if name == "ns" else "c5_small")
            chk = decomposed_bitexact_check(rank, local_rank, world, dist, transport=a.mode_d_transport)
            if mode_d is not None:
                mode_d["bitexact_check"] = chk
        except Exception as ex:  # noqa: BLE001 -- reported in the line
            mode_d = {"error": f"{type(ex).__name__}: {ex}"[:400]} if rank == 0 else None
    if dist is not None:
        dist.barrier()
        if watchdog is not None:
            watchdog.cancel()
        dist.destroy_process_group()
    if rank != 0:
        return
    if mode_d is not None:
        line["mode_d"] = mode_d
    print(json.dumps(line))


def _leave_mode_d(line, limit):
    """Watchdog of the mode D block of a multi-GPU run (see main): the block did not finish within ``limit`` seconds."""
    if line is not None:
        line["mode_d"] = {"error": f"the domain-decomposed block did not finish within {limit:.0f} s (a rank failed or hangs in a collective); "
                                   "the mode R numbers of this line are complete"}  # fmt: skip
        print(json.dumps(line), flush=True)
    os._exit(0)


if __name__ == "__main__":
    main()
