#!/usr/bin/env python3
"""tests/golden/test_full.npz: the data sets and parameters of the reference's own integration tests
(splashsurf_lib/tests/integration_tests/test_full.rs:144-157) with the REFERENCE's results (pysplashsurf 0.14.0 wheel in oracle/_ref):
particle densities, vertex / triangle counts, the outcome of its check_mesh_consistency.  Run in the build container (reads
/root/reference/data through this package's particle readers); the fixture is what travels to the GPU box.

The reference's tests reconstruct with enable_multi_threading = false and enable_simd = false (test_full.rs:30-42), compact support
4 r (= smoothing length 2.0) and auto_disable = false for the subdomain grid; they assert a triangle-count window and a closed,
manifold mesh.  tests/test_zzzz_reference_datasets.py holds the GPU path to the same windows AND to the reference's exact counts and
densities, and compares the whole mesh with the pinned oracle."""
import io
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402
from splashsurf_b200 import particle_formats as pf  # noqa: E402

DATA = "/root/reference/data"
# (test name, file, particle radius, cube size (relative), threshold, subdomain grid, particle AABB, triangle window) -- test_full.rs:144-157
CASES = [
    ("bunny_global", "bunny_frame_14_7705_particles.vtk", 0.025, 0.75, 0.6, False, None, (60000, 80000)),
    ("bunny_grid", "bunny_frame_14_7705_particles.vtk", 0.025, 0.75, 0.6, True, None, (60000, 80000)),
    ("hexecontahedron_grid", "pentagonal_hexecontahedron_32286_particles.bgeo", 0.025, 0.75, 0.6, True, None, (550000, 650000)),
    ("hilbert_grid", "hilbert_46843_particles.bgeo", 0.025, 0.75, 0.6, True, None, (360000, 400000)),
    ("hilbert2_grid", "hilbert2_7954_particles.vtk", 0.025, 1.1, 0.6, True, None, (90000, 100000)),
    ("octocat_grid", "octocat_32614_particles.bgeo", 0.025, 0.75, 0.6, True, None, (140000, 180000)),
    ("knot_global", "sailors_knot_19539_particles.vtk", 0.025, 1.1, 0.6, False, None, (40000, 70000)),
    ("knot_grid", "sailors_knot_19539_particles.vtk", 0.025, 1.1, 0.6, True, None, (40000, 70000)),
    ("free_particles_01", "free_particles_1000_particles.vtk", 0.5, 1.5, 0.45, False, None, (21000, 25000)),
    ("free_particles_02", "free_particles_125_particles.vtk", 0.5, 1.5, 0.45, False, ([-10.0] * 3, [210.0] * 3), (1500, 1600)),
]


def kwargs_of(case):
    _, _, r, c, t, grid, aabb, _ = case
    kw = dict(particle_radius=r, smoothing_length=2.0, cube_size=c, iso_surface_threshold=t, multi_threading=False, simd=False,
              subdomain_grid=grid, subdomain_grid_auto_disable=False)
    if aabb is not None:
        kw.update(aabb_min=aabb[0], aabb_max=aabb[1])
    return kw


def main():
    ps = oracle.reference()
    out, files, meta = {}, {}, {}
    for case in CASES:
        name, fname, *_rest, window = case
        if fname not in files:
            files[fname] = pf.particles_from_file(os.path.join(DATA, fname))
            out["particles:" + fname] = files[fname]
        p = files[fname]
        kw = kwargs_of(case)
        r = ps.reconstruct_surface(p, **kw)
        nv, nt = len(r.mesh.vertices), len(r.mesh.triangles)
        assert window[0] < nt < window[1], (name, nt)
        check = ps.check_mesh_consistency(r.mesh, r.grid, check_closed=True, check_manifold=True, debug=False)
        out["densities:" + name] = np.asarray(r.particle_densities, dtype=np.float32)
        meta[name] = {"file": fname, "kwargs": kw, "window": list(window), "nv": nv, "nt": nt, "consistent": check is None,
                      "grid_min": [float(v) for v in r.grid.aabb.min], "grid_ncells": [int(v) for v in r.grid.ncells_per_dim]}
        print(name, len(p), "particles ->", nv, "vertices", nt, "triangles", "consistent" if check is None else "INCONSISTENT")
    out["meta"] = json.dumps(meta)
    # no fixture file above 1 MB: the arrays go to test_full.npz, test_full_1.npz, ... (tests/conftest.py load_npz_parts)
    parts = [{}]
    for key in ["meta"] + sorted((k for k in out if k != "meta"), key=lambda k: -out[k].nbytes):
        buf = io.BytesIO()
        np.savez_compressed(buf, **parts[-1], **{key: out[key]})
        if parts[-1] and len(buf.getvalue()) > 950_000:
            parts.append({})
        parts[-1][key] = out[key]
    for i, part in enumerate(parts):
        path = os.path.join(ROOT, "tests", "golden", "test_full.npz" if i == 0 else f"test_full_{i}.npz")
        np.savez_compressed(path, **part)
        print(path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
