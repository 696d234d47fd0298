"""SURVEY 8(f.4): marching-cubes clean-up and barnacle decimation (host code of the library, csrc/ss_meshproc.inc) against the
reference's own outputs -- committed fixtures generated from the reference wheel (tools/make_golden_meshproc.py, the mesh-AABB clamp's
tests/golden/clamp_ref.npz) and, where the wheel is present, live runs on further meshes.  Both algorithms are sequential and deterministic
for a given vertex / triangle order, so parity is bit-exact: vertex positions, triangle indices and their order.  These tests need
no GPU: the entries take host arrays and no context."""
import os

import numpy as np
import pytest

from conftest import load_golden


def _grid(ss, g):
    return ss.UniformGrid(ss.Aabb3d(g["grid_min"], g["grid_max"]), float(g["cell_size"]), [int(v) for v in g["npoints"]], [int(v) for v in g["ncells"]])


def _same(mesh, v, t):
    return mesh.vertices.shape == v.shape and np.array_equal(mesh.vertices.view(np.uint32), v.view(np.uint32)) and \
        mesh.triangles.shape == t.shape and np.array_equal(mesh.triangles, t.astype(np.uint64))


@pytest.mark.parametrize("tag,snap,keep", [("cleanup", None, False), ("cleanup_snap03", 0.3, False), ("cleanup_keep", None, True)])
def test_marching_cubes_cleanup_matches_reference_fixture(ss, tag, snap, keep):
    g = load_golden("meshproc_ref")
    m = ss.TriMesh3d(g["vertices"].copy(), g["triangles"].astype(np.uint64))
    conn = ss.marching_cubes_cleanup(m, _grid(ss, g), max_rel_snap_dist=snap, max_iter=5, keep_vertices=keep)
    assert _same(m, g[tag + "_v"], g[tag + "_t"])
    # the connectivity it returns is the one of the new mesh (halfedge_mesh.rs:92-100)
    lists = conn.copy_connectivity()
    assert len(lists) == m.nvertices
    want = [set() for _ in range(m.nvertices)]
    for a, b, c in m.triangles.astype(np.int64):
        want[a] |= {b, c}; want[b] |= {a, c}; want[c] |= {a, b}
    assert all(set(l) == w and len(l) == len(w) for l, w in zip(lists, want))
    if keep:
        assert m.nvertices == len(g["vertices"]) and sum(1 for l in lists if not l) == len(g["vertices"]) - len(g["cleanup_v"])


def test_barnacle_decimation_matches_reference_fixture(ss):
    g = load_golden("meshproc_ref")
    m = ss.TriMesh3d(g["vertices"].copy(), g["triangles"].astype(np.uint64))
    conn = ss.barnacle_decimation(m)
    assert _same(m, g["decimated_v"], g["decimated_t"])
    assert len(g["decimated_v"]) < len(g["vertices"])                      # the fixture does contain barnacle configurations
    # connectivity: same neighbour sets as the reference reports
    assert np.array_equal(conn.offsets, g["decimated_conn_offsets"])
    mine = np.concatenate([sorted(l) for l in conn.copy_connectivity()]).astype(np.uint32)
    assert np.array_equal(mine, g["decimated_conn_sorted"])
    # ... and in the same order inside every list: the collapses happened in the reference's sequence (its hash maps' iteration order)
    assert np.array_equal(conn.indices, g["decimated_conn"])
    # chained like the pipeline does (reconstruct.rs:1058-1092): clean-up, then decimation
    m2 = ss.TriMesh3d(g["cleanup_snap03_v"].copy(), g["cleanup_snap03_t"].astype(np.uint64))
    ss.barnacle_decimation(m2)
    assert _same(m2, g["cleanup_snap03_decimated_v"], g["cleanup_snap03_decimated_t"])


@pytest.mark.parametrize("tag,qkw", [("quads", {}), ("quads_strict", dict(non_squareness_limit=1.3, normal_angle_limit=4.0, max_interior_angle=110.0))])
def test_convert_tris_to_quads_matches_reference_fixture(ss, tag, qkw):
    """postprocessing.rs:689-910: remaining triangles and quads, in the reference's cell order (its hash-set iteration order)."""
    g = load_golden("meshproc_ref")
    q = ss.convert_tris_to_quads(ss.TriMesh3d(g["vertices"].copy(), g["triangles"].astype(np.uint64)), **qkw)
    assert np.array_equal(q.get_triangles(), g[tag + "_t"].astype(np.uint64)) and np.array_equal(q.get_quads(), g[tag + "_q"].astype(np.uint64))
    assert len(q.get_quads()) > 100 and len(q.get_triangles()) + 2 * len(q.get_quads()) == len(g["triangles"])
    assert np.array_equal(q.vertices, g["vertices"])
    empty = ss.convert_tris_to_quads(ss.TriMesh3d(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.uint64)))
    assert len(empty.get_triangles()) == 0 and len(empty.get_quads()) == 0


def test_meshproc_edge_cases(ss):
    g = load_golden("meshproc_ref")
    grid = _grid(ss, g)
    empty = ss.TriMesh3d(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.uint64))
    assert ss.marching_cubes_cleanup(empty, grid).copy_connectivity() == [] and empty.nvertices == 0
    assert ss.barnacle_decimation(empty).copy_connectivity() == []
    # a single triangle (every edge is a boundary edge: nothing can collapse, halfedge_mesh.rs:204-256)
    one = ss.TriMesh3d(np.array([[0.1, 0.1, 0.1], [0.12, 0.1, 0.1], [0.1, 0.12, 0.1]], np.float32) + g["grid_min"], np.array([[0, 1, 2]], np.uint64))
    ss.marching_cubes_cleanup(one, grid)
    assert one.nvertices == 3 and one.ncells == 1
    # a vertex outside of the grid: the reference panics (unwrap); here an error code
    bad = ss.TriMesh3d(np.array([[1e6, 0, 0], [0, 0, 0], [0, 1, 0]], np.float32), np.array([[0, 1, 2]], np.uint64))
    with pytest.raises(ss.SplashsurfError) as e:
        ss.marching_cubes_cleanup(bad, grid)
    assert e.value.code == 6                                               # SS_ERR_INVALID_PARAMETER
    with pytest.raises(ss.SplashsurfError):
        ss.barnacle_decimation(ss.TriMesh3d(np.zeros((2, 3), np.float32), np.array([[0, 1, 5]], np.uint64)))      # index out of range


def _mesh_digest(vertices, triangles):
    from conftest import digest
    return digest(np.asarray(vertices, np.float32), np.asarray(triangles).astype(np.uint64))


def _wheel_meshproc_digests(ps, rec, snap, keep):
    """The wheel's clean-up of its raw mesh, quad conversion of the raw and the cleaned mesh, barnacle decimation from both."""
    ref = rec.mesh.copy()
    ps.marching_cubes_cleanup(ref, rec.grid, max_rel_snap_dist=snap, max_iter=5, keep_vertices=keep)
    out = {"cleanup": _mesh_digest(ref.vertices, ref.triangles)}
    for name, src in (("raw", rec.mesh), ("cleanup", ref)):
        q = ps.convert_tris_to_quads(src)
        out["quads_" + name] = _mesh_digest(q.get_triangles(), q.get_quads())
    for name, start in (("raw", rec.mesh.copy()), ("cleanup", ref)):
        ps.barnacle_decimation(start, keep_vertices=keep)
        out["decimated_" + name] = _mesh_digest(start.vertices, start.triangles)
    return out


def _library_meshproc_digests(ss, v0, t0, grid, snap, keep):
    """The same steps with this package's functions, from the same raw mesh."""
    mine = ss.TriMesh3d(v0.copy(), t0.copy())
    ss.marching_cubes_cleanup(mine, grid, max_rel_snap_dist=snap, max_iter=5, keep_vertices=keep)
    out = {"cleanup": _mesh_digest(mine.vertices, mine.triangles)}
    for name, (v, t) in (("raw", (v0, t0)), ("cleanup", (mine.vertices, mine.triangles))):
        q = ss.convert_tris_to_quads(ss.TriMesh3d(np.array(v, np.float32), np.array(t, np.uint64)))
        out["quads_" + name] = _mesh_digest(q.get_triangles(), q.get_quads())
        m = ss.TriMesh3d(np.array(v, np.float32), np.array(t, np.uint64))
        ss.barnacle_decimation(m, keep_vertices=keep)
        out["decimated_" + name] = _mesh_digest(m.vertices, m.triangles)
    return out


@pytest.mark.parametrize("case", ["cube_c05", "dam_snap05_keep"])
def test_meshproc_matches_reference_live(ss, oracle_mod, case, reference_output):
    """Against the wheel on other meshes (larger, other cell sizes), bit for bit.  The cube's raw mesh is stored
    (tests/golden/meshproc_cube_c05_ref.npz) with the digests of the wheel's results (tests/golden/reference_outputs.json); the
    148k-vertex dam-break mesh (1.9 MB) is compared where the wheel is present."""
    from conftest import GOLDEN
    from splashsurf_b200 import synthetic as syn
    if case == "cube_c05":
        p, kw, snap, keep = syn.jittered_cube(14, 0.025, 5), dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.5), None, False
    else:
        p, kw, snap, keep = syn.dam_break_scaled(30000, 0.01, 9), dict(particle_radius=0.01, smoothing_length=2.0, cube_size=0.6), 0.5, True
        if not oracle_mod.reference_available():
            pytest.skip("reference wheel not unpacked (oracle/_ref)")

    def run_reference(save):
        ps = oracle_mod.reference()
        rec = ps.reconstruct_surface(p, iso_surface_threshold=0.6, subdomain_grid=True, **kw)
        rg = rec.grid
        raw = dict(vertices=np.asarray(rec.mesh.vertices, np.float32), triangles=np.asarray(rec.mesh.triangles).astype(np.uint32),
                   grid_min=np.asarray(rg.aabb.min, np.float32), grid_max=np.asarray(rg.aabb.max, np.float32), cell_size=np.float32(rg.cell_size),
                   npoints=np.asarray(rg.npoints_per_dim, np.int64), ncells=np.asarray(rg.ncells_per_dim, np.int64))
        if save:
            np.savez_compressed(os.path.join(GOLDEN, f"meshproc_{case}_ref.npz"), **raw)
        return _wheel_meshproc_digests(ps, rec, snap, keep), raw
    if case == "cube_c05":
        want = reference_output(f"meshproc_live.{case}", lambda: run_reference(True)[0])
        g = load_golden(f"meshproc_{case}_ref")
    else:
        want, g = run_reference(False)
    assert _library_meshproc_digests(ss, g["vertices"], g["triangles"].astype(np.uint64), _grid(ss, g), snap, keep) == want


def _tetra(offset, base):
    v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1]], np.float32) + np.asarray(offset, np.float32)
    t = np.array([[0, 2, 1], [0, 1, 3], [1, 2, 3], [0, 3, 2]], np.uint64) + base
    return v, t


def _flat_sheet(n=6):
    """n x n quads of the z = 0 plane, two triangles each, all oriented +z."""
    g = np.stack(np.meshgrid(np.arange(n + 1), np.arange(n + 1), indexing="ij"), -1).reshape(-1, 2)
    v = np.concatenate([g, np.zeros((len(g), 1))], axis=1).astype(np.float32)
    idx = lambda i, j: i * (n + 1) + j          # noqa: E731
    t = []
    for i in range(n):
        for j in range(n):
            t += [(idx(i, j), idx(i + 1, j), idx(i + 1, j + 1)), (idx(i, j), idx(i + 1, j + 1), idx(i, j + 1))]
    return v, np.array(t, np.uint64)


def test_check_mesh_consistency_and_clamp_unit_cases(ss):
    """marching_cubes.rs:129-213 / mesh.rs:334-371, :1007-1090 on hand-made meshes: a closed tetrahedron, an open one, two tetrahedra
    glued at one vertex (non-manifold vertex) and at one edge (non-manifold edge: four incident faces)."""
    grid = ss.UniformGrid(ss.Aabb3d(np.zeros(3, np.float32), np.full(3, 4, np.float32)), 1.0, [5, 5, 5], [4, 4, 4])
    v, t = _tetra([0, 0, 0], 0)
    closed = ss.TriMesh3d(v, t)
    assert ss.check_mesh_consistency(closed, grid) is None and len(ss.find_non_manifold_vertices(closed)) == 0
    opened = ss.TriMesh3d(v, t[:3])
    msg = ss.check_mesh_consistency(opened, grid)
    assert msg.startswith("Mesh is not closed. It has 3 boundary edges") and ss.check_mesh_consistency(opened, grid, check_closed=False) is None
    # two tetrahedra sharing vertex 0 only
    v2, t2 = _tetra([-2, -2, -2], 4)
    vv = np.concatenate([v, v2[1:]]); t2 = np.where(t2 == 4, 0, t2 - 1)
    glued = ss.TriMesh3d(vv, np.concatenate([t, t2]))
    assert ss.find_non_manifold_vertices(glued).tolist() == [0]
    msg = ss.check_mesh_consistency(glued, grid, debug=True)
    assert "1 non-manifold vertices" in msg and "Non-manifold vertices: [0]" in msg and ss.check_mesh_consistency(glued, grid, check_manifold=False) is None
    # two tetrahedra sharing the edge (0, 1): that edge has four incident faces
    w = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [0, -1, 0], [0, 0, -1]], np.float32)
    ta = np.array([[0, 2, 1], [0, 1, 3], [1, 2, 3], [0, 3, 2]], np.uint64)
    tb = np.array([[0, 1, 4], [0, 5, 1], [1, 5, 4], [0, 4, 5]], np.uint64)
    msg = ss.check_mesh_consistency(ss.TriMesh3d(w, np.concatenate([ta, tb])), grid)
    assert "1 non-manifold edges" in msg
    # orientation: a consistently oriented mesh has no flipped face; a reversed triangle of a flat sheet is anti-parallel to the normals of its vertices
    assert len(ss.find_flipped_faces(closed)) == 0
    sheet_v, sheet_t = _flat_sheet()
    assert len(ss.find_flipped_faces(ss.TriMesh3d(sheet_v, sheet_t))) == 0
    bad_t = sheet_t.copy(); bad_t[31] = bad_t[31][[0, 2, 1]]                                  # an interior triangle, reversed
    assert ss.find_flipped_faces(ss.TriMesh3d(sheet_v, bad_t)).tolist() == [31]
    # clamp: triangles with a vertex inside [min, max) stay, unused vertices go, the rest is clamped into the box
    m, attrs = ss.clamp_mesh_with_aabb(closed, [-0.5, -0.5, 0.5], [2, 2, 2], point_attributes={"a": np.arange(4.0)})
    assert m.ncells == 3 and m.nvertices == 4 and float(m.vertices[:, 2].min()) == 0.5 and attrs["a"].tolist() == [0.0, 1.0, 2.0, 3.0]
    m, attrs = ss.clamp_mesh_with_aabb(closed, [0.5, -0.5, -0.5], [2, 2, 2], clamp_vertices=False, point_attributes={"a": np.arange(4.0)})
    assert m.ncells == 3 and np.array_equal(m.vertices, closed.vertices)            # every vertex is still used by a kept triangle
    m, _ = ss.clamp_mesh_with_aabb(closed, [5, 5, 5], [6, 6, 6])
    assert m.ncells == 0 and m.nvertices == 0
    m, _ = ss.clamp_mesh_with_aabb(closed, [5, 5, 5], [6, 6, 6], keep_vertices=True, clamp_vertices=False)
    assert m.ncells == 0 and m.nvertices == 4


def test_clamp_and_checks_match_reference_live(ss, oracle_mod, reference_output):
    """The reference pipeline's mesh-AABB clamp (same input mesh: its own raw mesh) and check_mesh_consistency, on random boxes.  Its raw
    mesh and grid are stored in tests/golden/clamp_ref.npz, its results by digests in tests/golden/reference_outputs.json."""
    import re
    from conftest import GOLDEN, digest
    from splashsurf_b200 import synthetic as syn
    p = syn.splash((12, 12, 12), 4, 0.025, 91)
    kw = dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.75, iso_surface_threshold=0.6, subdomain_grid=True)
    rng = np.random.default_rng(5)
    head = lambda s_: [l for l in (s_ or "None").split("\n") if not l.startswith("\t")]       # noqa: E731

    def run_reference():
        ps = oracle_mod.reference()
        rec = ps.reconstruct_surface(p, **kw)
        g = rec.grid
        v, t = np.array(rec.mesh.vertices, np.float32), np.array(rec.mesh.triangles, np.uint64)
        np.savez_compressed(os.path.join(GOLDEN, "clamp_ref.npz"), vertices=v, triangles=t.astype(np.uint32),
                            grid_min=np.asarray(g.aabb.min, np.float32), grid_max=np.asarray(g.aabb.max, np.float32), cell_size=np.float32(g.cell_size),
                            npoints=np.asarray(g.npoints_per_dim, np.int64), ncells=np.asarray(g.ncells_per_dim, np.int64))
        out = {"consistent": ps.check_mesh_consistency(rec.mesh, g) is None, "trials": []}
        lo, hi = v.min(0), v.max(0)
        for trial in range(12):
            c = lo + rng.random(3) * (hi - lo); e = rng.uniform(0.05, 0.3, 3) * (hi - lo)
            a, b = (c - e).tolist(), (c + e).tolist()
            keep, clampv = bool(rng.integers(0, 2)), bool(rng.integers(0, 2))
            mw, _ = ps.reconstruction_pipeline(p, mesh_aabb_min=a, mesh_aabb_max=b, mesh_aabb_clamp_vertices=clampv, keep_vertices=keep, mesh_smoothing_weights=False, **kw)
            r = ps.check_mesh_consistency(mw.mesh, g, debug=True)
            nm = sorted(int(x) for x in re.findall(r"\d+", r.split("Non-manifold vertices:")[1])) if r and "Non-manifold vertices" in r else None
            out["trials"].append({"box": [a, b], "keep": keep, "clamp": clampv, "mesh": digest(np.asarray(mw.mesh.vertices, np.float32), np.asarray(mw.mesh.triangles, np.uint64)),
                                  "check": head(r), "non_manifold": nm})
        return out
    want = reference_output("clamp_and_checks", run_reference)
    g = load_golden("clamp_ref")
    v, t = g["vertices"], g["triangles"].astype(np.uint64)
    grid = ss.UniformGrid(ss.Aabb3d(g["grid_min"], g["grid_max"]), float(g["cell_size"]), [int(x) for x in g["npoints"]], [int(x) for x in g["ncells"]])
    assert want["consistent"] and ss.check_mesh_consistency(ss.TriMesh3d(v, t), grid) is None
    for w in want["trials"]:
        (a, b), keep, clampv = w["box"], w["keep"], w["clamp"]
        cm, _ = ss.clamp_mesh_with_aabb(ss.TriMesh3d(v, t), a, b, clamp_vertices=clampv, keep_vertices=keep)
        assert digest(np.asarray(cm.vertices, np.float32), np.asarray(cm.triangles, np.uint64)) == w["mesh"]
        assert head(ss.check_mesh_consistency(cm, grid, debug=True)) == w["check"]
        if w["non_manifold"] is not None:
            assert w["non_manifold"] == ss.find_non_manifold_vertices(cm).tolist()


def test_half_edge_connectivity_kat(ss):
    """halfedge_mesh.rs:564-590 (test_half_edge_mesh): the vertex connectivity a half-edge mesh reports for two triangles sharing an
    edge equals TriMesh3d::vertex_vertex_connectivity up to order."""
    v = np.array([[0, 1, 0], [1, 0, 0], [1, 2, 0], [2, 1, 0]], np.float32)
    t = np.array([[0, 1, 2], [1, 3, 2]], np.uint64)
    m = ss.TriMesh3d(v, t)
    conn = ss.barnacle_decimation(m, keep_vertices=True).copy_connectivity()        # no barnacles: the mesh comes back unchanged
    assert np.array_equal(m.triangles, t) and [sorted(c) for c in conn] == [[1, 2], [0, 2, 3], [0, 1, 3], [1, 2]]


def test_mesh_containers_mirror_the_reference_bindings(ss, oracle_mod, tmp_path, reference_output):
    """pysplashsurf's mesh containers (pysplashsurf/src/mesh.rs, aabb.rs): MeshWithData(mesh), add_*_attribute with its type / shape / length
    checks, copy / copy_mesh / mesh_type / dtype, Aabb3d helpers -- same results as the wheel (stored in tests/golden/reference_outputs.json)."""
    v = np.random.default_rng(0).normal(size=(6, 3)).astype(np.float32)
    t = np.array([[0, 1, 2], [3, 4, 5]], np.uint64)
    m = ss.MeshWithData(ss.TriMesh3d(v, t))
    assert m.dtype == np.float32 and m.mesh.dtype == np.float32 and m.mesh_type == ss.MeshType.Tri3d and m.point_attributes == {} == m.cell_attributes
    m.add_point_attribute("w", np.zeros(6, np.float32))
    m.add_point_attribute("v", np.zeros((6, 3), np.float32))
    m.add_point_attribute("i", np.arange(6, dtype=np.uint64))
    m.add_point_attribute("w", np.ones(6, np.float32))                     # replaces, keeps its place
    m.add_cell_attribute("c", np.zeros(2, np.float32))
    assert list(m.point_attributes) == ["w", "v", "i"] and m.point_attributes["w"].max() == 1.0 and list(m.cell_attributes) == ["c"]
    with pytest.raises(TypeError, match="unsupported attribute data type"):
        m.add_point_attribute("d", np.zeros(6, np.float64))
    with pytest.raises(TypeError, match="unsupported attribute data type"):
        m.add_point_attribute("d", np.zeros(6, np.int32))
    with pytest.raises(ValueError, match="expected Nx1 or Nx3 array"):
        m.add_point_attribute("d", np.zeros((6, 2), np.float32))
    with pytest.raises(ValueError, match="must match number of vertices"):
        m.add_point_attribute("d", np.zeros(3, np.float32))
    with pytest.raises(ValueError, match="must match number of cells"):
        m.add_cell_attribute("d", np.zeros(3, np.float32))
    with pytest.raises(TypeError, match="unsupported mesh type"):
        ss.MeshWithData(m)
    c = m.copy()
    c.point_attributes["w"][:] = 5
    c.mesh.vertices[:] = 0
    assert m.point_attributes["w"].max() == 1.0 and np.array_equal(m.mesh.vertices, v) and type(m.copy_mesh()) is ss.TriMesh3d
    q = ss.MeshWithData(ss.MixedTriQuadMesh3d(v, t[:1], np.array([[0, 1, 2, 3]], np.uint64)))
    assert q.mesh_type == ss.MeshType.MixedTriQuad3d and q.ncells == 2 and type(q.copy_mesh()) is ss.MixedTriQuadMesh3d
    m.mesh.write_to_file(str(tmp_path / "t.obj"))
    m.write_to_file(str(tmp_path / "m.ply"))
    q.mesh.write_to_file(str(tmp_path / "q.vtk"))
    from splashsurf_b200 import io
    assert len(io.read_obj(str(tmp_path / "t.obj"))[0]) == 6 and list(io.read_ply_mesh(str(tmp_path / "m.ply"))[3]) == ["w", "v", "i"]
    assert len(io.read_vtk_mesh(str(tmp_path / "q.vtk"))[2]) == 1
    a = ss.Aabb3d.from_min_max([0, 0, 0], [1, 2, 3])
    b = ss.Aabb3d.from_points(np.array([[0, 1, 2], [3, -1, 5]], np.float32))
    assert a.min.dtype == np.float64 and not a.contains_point([1, 1, 1]) and a.contains_point([0, 0, 0]) and not a.contains_point([0.5, 2, 1])
    assert np.array_equal(b.min, [0, -1, 2]) and np.array_equal(b.max, [3, 1, 5])
    points = ([1, 1, 1], [0, 0, 0], [0.5, 2, 1], [0.999, 1.999, 2.999], [-1e-9, 0, 0])

    def run_reference():                    # the wheel's answers, stored in tests/golden/reference_outputs.json
        ps = oracle_mod.reference()
        ra = ps.Aabb3d.from_min_max([0, 0, 0], [1, 2, 3])
        rb = ps.Aabb3d.from_points(np.array([[0, 1, 2], [3, -1, 5]], np.float32))
        return {"min": np.asarray(ra.min).tolist(), "min_dtype": str(np.asarray(ra.min).dtype), "from_points_max": np.asarray(rb.max).tolist(),
                "contains": [bool(ra.contains_point(pt)) for pt in points], "mesh_types": [str(ps.MeshType.Tri3d), str(ps.MeshType.MixedTriQuad3d)]}
    want = reference_output("mesh_containers.aabb_and_mesh_type", run_reference)
    assert a.min.tolist() == want["min"] and str(a.min.dtype) == want["min_dtype"] and b.max.tolist() == want["from_points_max"]
    assert [a.contains_point(pt) for pt in points] == want["contains"]
    assert [str(ss.MeshType.Tri3d), str(ss.MeshType.MixedTriQuad3d)] == want["mesh_types"]


def test_mesh_rs_manifold_known_answers(ss):
    """The reference's unit tests of its mesh checks (mesh.rs:1120-1221: test_tri_mesh_edge_info, test_tri_mesh_non_manifold_vertex_info,
    test_tri_mesh_manifold_info) on the helpers behind check_mesh_consistency, and aabb.rs:277-291 (half-open contains_point)."""
    v5 = np.float32([[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0], [0, 0, 1]])
    nm_edge = ss.TriMesh3d(v5, np.uint64([[0, 1, 2], [1, 3, 2], [1, 2, 4]]))
    nm_edge2 = ss.TriMesh3d(v5, np.uint64([[0, 1, 2], [1, 3, 2], [1, 2, 4], [4, 2, 1]]))
    nm_vert = ss.TriMesh3d(np.float32([[1, 0, 0], [0, 1, 0], [1, 1, 0], [2, 1, 1], [1, 2, 1]]), np.uint64([[0, 2, 1], [2, 3, 4]]))
    one = ss.TriMesh3d(np.random.default_rng(0).random((3, 3)).astype(np.float32), np.uint64([[0, 1, 2]]))
    uniq, cnt, _ = ss._edge_table(nm_edge.triangles)                           # test_tri_mesh_edge_info
    for e, c in zip(uniq.tolist(), cnt.tolist()):
        assert c == (3 if sorted(e) == [1, 2] else 1)
    assert int((cnt == 1).sum()) == 6 and int((cnt > 2).sum()) == 1
    assert ss.find_non_manifold_vertices(nm_vert).tolist() == [2]              # test_tri_mesh_non_manifold_vertex_info

    def info(mesh):
        _, c, _ = ss._edge_table(mesh.triangles)
        nb, ne, nv = int((c == 1).sum()), int((c > 2).sum()), len(ss.find_non_manifold_vertices(mesh))
        return nb == 0, ne == 0 and nv == 0, ne, nv                            # closed, manifold, #non-manifold edges, #non-manifold vertices
    assert info(one) == (False, True, 0, 0)                                    # test_tri_mesh_manifold_info
    assert info(nm_edge) == (False, False, 1, 0)
    assert info(nm_edge2) == (False, False, 1, 0)
    assert info(nm_vert) == (False, False, 0, 1)
    for mesh, closed_msg, manifold_msg in ((nm_edge, "not closed", "non-manifold edges"), (nm_vert, "not closed", "non-manifold vertices")):
        text = ss.check_mesh_consistency(mesh, None, check_closed=True, check_manifold=True)
        assert text is not None and closed_msg in text and manifold_msg in text
        assert ss.check_mesh_consistency(mesh, None, check_closed=False, check_manifold=False) is None
    box = ss.Aabb3d.from_min_max([0.0, 0.0, 0.0], [1.0, 1.0, 1.0])             # aabb.rs:277-291
    for q, inside in (([.5, .5, .5], True), ([0, .5, .5], True), ([.5, 0, .5], True), ([.5, .5, 0], True), ([0, 0, 0], True), ([1, 0, 0], False),
                      ([0, 1, 0], False), ([0, 0, 1], False), ([1, 1, 1], False)):
        assert box.contains_point(q) == inside
