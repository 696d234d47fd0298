#!/usr/bin/env python3
"""Generates tests/golden/meshproc_ref.npz from the REFERENCE ITSELF (pysplashsurf 0.14.0 wheel in oracle/_ref): a marching-cubes
mesh of the reference plus what its marching_cubes_cleanup (postprocessing.rs:99-242; with and without a snap distance, with and
without keep_vertices) and its barnacle_decimation (:244-686) make of it.  SURVEY 8(f.4) parity fixture: both algorithms are
sequential and deterministic for a given vertex / triangle order, so the library's host implementation must reproduce these
arrays bit for bit."""
import os, sys
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402
from splashsurf_b200 import synthetic as syn  # noqa: E402

ps = oracle.reference()
p = syn.splash((9, 9, 9), 3, 0.025, 411)
kw = dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.75, iso_surface_threshold=0.6, subdomain_grid=True)
rec = ps.reconstruct_surface(p, **kw)
out = dict(vertices=np.asarray(rec.mesh.vertices, np.float32), triangles=np.asarray(rec.mesh.triangles).astype(np.uint32),
           grid_min=np.asarray(rec.grid.aabb.min, np.float32), grid_max=np.asarray(rec.grid.aabb.max, np.float32),
           cell_size=np.float32(rec.grid.cell_size), npoints=np.asarray(rec.grid.npoints_per_dim, np.int64),
           ncells=np.asarray(rec.grid.ncells_per_dim, np.int64))
for tag, snap, keep in [("cleanup", None, False), ("cleanup_snap03", 0.3, False), ("cleanup_keep", None, True)]:
    m = rec.mesh.copy()
    ps.marching_cubes_cleanup(m, rec.grid, max_rel_snap_dist=snap, max_iter=5, keep_vertices=keep)
    out[tag + "_v"], out[tag + "_t"] = np.asarray(m.vertices, np.float32), np.asarray(m.triangles).astype(np.uint32)
    if tag == "cleanup_snap03":
        m2 = m.copy()
        c = ps.barnacle_decimation(m2, keep_vertices=False)
        out["cleanup_snap03_decimated_v"], out["cleanup_snap03_decimated_t"] = np.asarray(m2.vertices, np.float32), np.asarray(m2.triangles).astype(np.uint32)
m = rec.mesh.copy()
c = ps.barnacle_decimation(m, keep_vertices=False)
out["decimated_v"], out["decimated_t"] = np.asarray(m.vertices, np.float32), np.asarray(m.triangles).astype(np.uint32)
conn = c.copy_connectivity()
out["decimated_conn_offsets"] = np.concatenate([[0], np.cumsum([len(l) for l in conn])]).astype(np.uint64)
out["decimated_conn_sorted"] = np.concatenate([sorted(l) for l in conn]).astype(np.uint32)
out["decimated_conn"] = np.concatenate([list(l) for l in conn]).astype(np.uint32)      # in the reference's half-edge order
for tag, src, qkw in [("quads", rec.mesh, {}), ("quads_strict", rec.mesh, dict(non_squareness_limit=1.3, normal_angle_limit=4.0, max_interior_angle=110.0))]:
    q = ps.convert_tris_to_quads(src, **qkw)                    # postprocessing.rs:689-910 (cells in the reference's order)
    out[tag + "_t"], out[tag + "_q"] = np.asarray(q.get_triangles()).astype(np.uint32), np.asarray(q.get_quads()).astype(np.uint32)
# two files below 1 MB each (tests/conftest.py load_npz_parts): the decimation and quad results go to meshproc_ref_1.npz
second = ("decimated", "quads")
for name, part in (("meshproc_ref", {k: v for k, v in out.items() if not k.startswith(second)}),
                   ("meshproc_ref_1", {k: v for k, v in out.items() if k.startswith(second)})):
    path = os.path.join(ROOT, "tests", "golden", name + ".npz")
    np.savez_compressed(path, **part)
    print({k: v.shape for k, v in part.items()}, os.path.getsize(path) // 1024, "KiB")
