"""GPU tests of the device post-processing entries (SURVEY §8f) through the C ABI / the pipeline mirror, against
oracle/postprocess.py (pinned against the reference pipeline, tests/test_oracle_postprocess.py).  The kernels themselves are
also stepped on the CPU by tests/test_post_emulation.py.  Tolerance: 2e-5 relative (f32 sums in a different order)."""
import ctypes as C

import numpy as np
import pytest

REL = 2e-5


def _key_order(keys):
    k = np.asarray(keys).reshape(len(keys), -1)
    return np.lexsort(tuple(k[:, c] for c in range(k.shape[1] - 1, -1, -1)))


def compare_point_fields(fields_a, keys_a, fields_b, keys_b, tol=REL):
    """Compares per-vertex arrays of two meshes with the same vertex set in different orders (matched by MC edge key)."""
    oa, ob = _key_order(keys_a), _key_order(keys_b)
    assert np.array_equal(np.asarray(keys_a)[oa], np.asarray(keys_b)[ob])
    worst = {}
    for name in fields_b:
        a = np.asarray(fields_a[name], dtype=np.float64)[oa]
        b = np.asarray(fields_b[name], dtype=np.float64)[ob]
        assert a.shape == b.shape, name
        assert not np.isnan(a).any() and not np.isnan(b).any(), name
        err = float(np.abs(a - b).max()) / max(float(np.abs(b).max()), 1.0)
        worst[name] = err
        assert err <= tol, (name, err)
    return worst


def test_compare_helper_matches_permuted_copy():
    """CPU self-test of the matching helper used by the GPU tests below."""
    rng = np.random.default_rng(0)
    keys = rng.permutation(40 * 4).reshape(40, 4).astype(np.int64)
    f = {"a": rng.normal(size=40).astype(np.float32), "v": rng.normal(size=(40, 3)).astype(np.float32)}
    perm = rng.permutation(40)
    compare_point_fields({k: v[perm] for k, v in f.items()}, keys[perm], f, keys)
    bad = {k: v[perm].copy() for k, v in f.items()}
    bad["a"][3] += 1.0
    with pytest.raises(AssertionError):
        compare_point_fields(bad, keys[perm], f, keys)


def _oracle_pipeline(oracle_mod, x, kw, post, attributes=None):
    from oracle import postprocess as pp
    o = oracle_mod.reconstruct(x, **kw)
    assert o["rc"] == 0
    inside = o.get("particle_inside_aabb")
    xf = x[inside] if inside is not None else x
    attrs = {k: (v[inside] if inside is not None else v) for k, v in (attributes or {}).items()}
    _, h, _ = oracle_mod.absolute_params(kw["particle_radius"], kw["smoothing_length"], kw["cube_size"])
    out = pp.pipeline(xf, o["particle_densities"], o["vertices"], o["triangles"], particle_radius=kw["particle_radius"], rest_density=1000.0,
                      compact_support_radius=float(h), attributes=attrs, sph_normals_fn=oracle_mod.sph_normals, **post)
    return o, out


CASES = [
    ("weights_smoothing_sphnormals", dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.75, subdomain_num_cubes_per_dim=32,
                                          subdomain_grid_auto_disable=False),
     dict(mesh_smoothing_weights=True, mesh_smoothing_weights_normalization=13.0, mesh_smoothing_iters=5, compute_normals=True,
          sph_normals=True, normals_smoothing_iters=3)),
    ("unweighted_even_iterations_area_normals", dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.6),
     dict(mesh_smoothing_weights=False, mesh_smoothing_iters=4, compute_normals=True, sph_normals=False, normals_smoothing_iters=None)),
    ("weights_only_no_smoothing", dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.9),
     dict(mesh_smoothing_weights=True, mesh_smoothing_weights_normalization=9.0, mesh_smoothing_iters=None, compute_normals=True,
          sph_normals=True, normals_smoothing_iters=None)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,kw,post", CASES, ids=[c[0] for c in CASES])
def test_pipeline_postprocessing_matches_oracle(ss, oracle_mod, name, kw, post):
    from splashsurf_b200 import synthetic
    x = synthetic.splash((14, 12, 13), 4, 0.025, 201)
    rng = np.random.default_rng(202)
    attributes = {"vel": rng.normal(size=x.shape).astype(np.float32), "temp": (x[:, 1] * 3 + 1).astype(np.float32)}
    o, ref = _oracle_pipeline(oracle_mod, x, kw, post, attributes)
    m, rec = ss.reconstruction_pipeline(x, attributes_to_interpolate=attributes, **kw, **post, output_mesh_smoothing_weights=True,
                                        output_raw_normals=True, with_debug=True)
    got = dict(m.point_attributes)
    got["vertices"] = m.mesh.vertices
    want = {k: v for k, v in ref.items() if k in got}
    assert set(want) >= {"vertices", "vel", "temp", "normals"}
    if post.get("compute_normals") and not post.get("sph_normals") and post.get("mesh_smoothing_iters"):
        # Area-weighted normals of a smoothed mesh amplify the 1-ulp differences of the smoothed vertices by
        # 1 / (edge length) on sliver triangles, so they are checked on the device's own vertices instead.
        from oracle import postprocess as pp
        want.pop("normals")
        mine = pp.vertex_normals(m.mesh.vertices, m.mesh.triangles)
        assert np.abs(got["normals"].astype(np.float64) - mine).max() <= REL
    compare_point_fields(got, rec.vertex_edge_keys, want, o["vertex_keys"], 5e-5 if post.get("sph_normals") else REL)
    # the raw mesh stays available in the reconstruction object and the smoothing really moved the vertices
    assert np.array_equal(rec.mesh.triangles, m.mesh.triangles)
    if post.get("mesh_smoothing_iters"):
        assert np.abs(rec.mesh.vertices - m.mesh.vertices).max() > 1e-4
    else:
        assert np.array_equal(rec.mesh.vertices, m.mesh.vertices)


@pytest.mark.gpu
def test_pipeline_with_particle_aabb_filters_attributes(ss, oracle_mod):
    from splashsurf_b200 import synthetic
    x = synthetic.splash((16, 12, 12), 3, 0.025, 211)
    kw = dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.75, aabb_min=[-0.05, -0.05, -0.05], aabb_max=[0.55, 1.5, 0.7])
    post = dict(mesh_smoothing_weights=True, mesh_smoothing_iters=2, compute_normals=False)
    attributes = {"temp": (x[:, 0] - x[:, 2]).astype(np.float32)}
    o, ref = _oracle_pipeline(oracle_mod, x, kw, post, attributes)
    assert o.get("particle_inside_aabb") is not None and not o["particle_inside_aabb"].all()
    m, rec = ss.reconstruction_pipeline(x, attributes_to_interpolate=attributes, **kw, **post, with_debug=True)
    compare_point_fields({"vertices": m.mesh.vertices, "temp": m.point_attributes["temp"]}, rec.vertex_edge_keys,
                         {"vertices": ref["vertices"], "temp": ref["temp"]}, o["vertex_keys"])


@pytest.mark.gpu
def test_c_abi_smoothing_with_explicit_weights_and_connectivity(ss, oracle_mod):
    """ss_surface_laplacian_smoothing_f32 with caller weights / beta, ss_surface_vertex_connectivity, and the stale-surface error."""
    from oracle import postprocess as pp
    from splashsurf_b200 import synthetic
    x = synthetic.splash((12, 12, 12), 2, 0.025, 221)
    kw = dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.75)
    ctx = ss.Context()
    L = ctx._L
    p = ss.make_params(**kw)
    s = ctx.reconstruct_raw(x.ctypes.data, len(x), p)
    try:
        nv, nt = L.ss_surface_num_vertices(s), L.ss_surface_num_triangles(s)
        v0 = np.empty((nv, 3), np.float32); t = np.empty((nt, 3), np.uint64)
        assert L.ss_surface_copy_vertices(s, v0.ctypes.data) == 0 and L.ss_surface_copy_triangles_u64(s, t.ctypes.data) == 0
        # connectivity: same sets as the reference's, ascending per vertex
        n_idx = C.c_uint64()
        off = np.empty(nv + 1, np.uint64)
        assert L.ss_surface_vertex_connectivity(s, off.ctypes.data, None, C.byref(n_idx)) == 0
        idx = np.empty(n_idx.value, np.uint32)
        assert L.ss_surface_vertex_connectivity(s, off.ctypes.data, idx.ctypes.data, C.byref(n_idx)) == 0
        roff, radj = pp.vertex_vertex_connectivity(t, nv)
        assert np.array_equal(off.astype(np.int64), roff)
        for i in range(0, nv, 11):
            assert np.array_equal(idx[int(off[i]):int(off[i + 1])], np.sort(radj[roff[i]:roff[i + 1]]))
        # smoothing with explicit weights, beta = 0.8, odd and even iteration counts applied one after the other
        w = np.random.default_rng(3).uniform(0, 1, nv).astype(np.float32)
        want = v0
        for iters in (3, 2):
            assert L.ss_surface_laplacian_smoothing_f32(s, iters, C.c_float(0.8), w.ctypes.data) == 0
            want = pp.laplacian_smoothing(want, roff, radj, iters, 0.8, w)
            got = np.empty((nv, 3), np.float32)
            assert L.ss_surface_copy_vertices(s, got.ctypes.data) == 0
            assert np.abs(got.astype(np.float64) - want).max() <= REL
        # a second reconstruction on the context retires the first surface's particle bins
        s2 = ctx.reconstruct_raw(x.ctypes.data, len(x), p)
        try:
            assert L.ss_surface_compute_smoothing_weights_f32(s, C.c_float(13.0), None, None) == 6      # SS_ERR_INVALID_PARAMETER
            assert b"bins" in L.ss_last_error()
            assert L.ss_surface_compute_smoothing_weights_f32(s2, C.c_float(13.0), None, None) == 0
            assert L.ss_surface_compute_normals_f32(s, 0) == 0                                          # mesh-only steps still work
        finally:
            ctx.free_surface(s2)
    finally:
        ctx.free_surface(s)
        ctx.close()


@pytest.mark.gpu
def test_standalone_mesh_functions(ss, oracle_mod):
    """The mirrors of pysplashsurf's free mesh functions (laplacian_smoothing_parallel, laplacian_smoothing_normals_parallel,
    TriMesh3d.vertex_normals_parallel / vertex_vertex_connectivity) on a mesh that does not come from a device reconstruction."""
    from oracle import postprocess as pp
    from splashsurf_b200 import synthetic
    x = synthetic.splash((9, 9, 9), 2, 0.025, 231)
    o = oracle_mod.reconstruct(x, particle_radius=0.025, smoothing_length=2.0, cube_size=0.75)
    v0, t = np.ascontiguousarray(o["vertices"], np.float32), np.ascontiguousarray(o["triangles"])
    mesh = ss.TriMesh3d(v0.copy(), t.copy())
    conn = mesh.vertex_vertex_connectivity()
    roff, radj = pp.vertex_vertex_connectivity(t, len(v0))
    assert np.array_equal(conn.offsets.astype(np.int64), roff)
    lists = conn.copy_connectivity()
    for i in range(0, len(v0), 13):
        assert lists[i] == sorted(radj[roff[i]:roff[i + 1]].tolist())
    n0 = mesh.vertex_normals_parallel()
    assert np.abs(n0.astype(np.float64) - pp.vertex_normals(v0, t)).max() <= REL
    w = np.random.default_rng(4).uniform(0, 1, len(v0)).astype(np.float32)
    ss.laplacian_smoothing_parallel(mesh, conn, iterations=3, beta=0.7, weights=w)
    assert np.abs(mesh.vertices.astype(np.float64) - pp.laplacian_smoothing(v0, roff, radj, 3, 0.7, w)).max() <= REL
    n = n0.copy()
    ss.laplacian_smoothing_normals_parallel(n, conn, iterations=2)
    assert np.abs(n.astype(np.float64) - pp.laplacian_smoothing_normals(n0, roff, radj, 2)).max() <= REL
    # particle queries are rejected on such a surface (no particles behind it)
    with ss._MeshSurface(v0, t) as m:
        assert m.L.ss_surface_compute_normals_f32(m.s, 1) == 6


@pytest.mark.gpu
def test_pipeline_with_mesh_cleanup_and_decimation(ss, oracle_mod, reference_output):
    """SURVEY 8(f.4) inside the pipeline mirror (reconstruct.rs:1058-1092): clean-up + decimation run first (host), the new mesh
    goes back to the device, and the particle-based steps (weights, smoothing, SPH normals, attribute interpolation) run on it.
    Checked against (a) the same steps composed by hand from the free functions and the oracle's post-processing on the cleaned
    mesh, and (b) the reference pipeline's mesh sizes (stored in tests/golden/reference_outputs.json; its raw mesh has another vertex
    order, so the collapse sequence -- and with it single vertices -- may differ)."""
    from oracle import postprocess as pp
    from splashsurf_b200 import synthetic as syn
    x = syn.splash((12, 12, 12), 3, 0.025, 515)
    kw = dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.75, iso_surface_threshold=0.6)
    rho_attr = np.linspace(0.0, 1.0, len(x), dtype=np.float32)
    post = dict(mesh_smoothing_iters=3, mesh_smoothing_weights=True, compute_normals=True, sph_normals=True, output_mesh_smoothing_weights=True)
    mwd, rec = ss.reconstruction_pipeline(x, attributes_to_interpolate={"a": rho_attr}, mesh_cleanup=True, mesh_cleanup_snap_dist=0.5,
                                          decimate_barnacles=True, **kw, **post)
    # (a) by hand: raw mesh -> free functions -> oracle post-processing of that mesh
    raw = ss.reconstruct_surface(x, **kw)
    m = raw.mesh.copy()
    ss.marching_cubes_cleanup(m, raw.grid, max_rel_snap_dist=0.5, max_iter=5)
    ss.barnacle_decimation(m)
    assert m.nvertices < raw.mesh.nvertices and mwd.mesh.nvertices == m.nvertices and np.array_equal(mwd.mesh.triangles, m.triangles)
    o = oracle_mod.reconstruct(x, **kw)
    _, h, _ = oracle_mod.absolute_params(kw["particle_radius"], kw["smoothing_length"], kw["cube_size"])
    want = pp.pipeline(x, o["particle_densities"], m.vertices, m.triangles.astype(np.int64), particle_radius=0.025, rest_density=1000.0,
                       compact_support_radius=float(h), attributes={"a": rho_attr}, sph_normals_fn=oracle_mod.sph_normals,
                       **{k: v for k, v in post.items() if k != "output_mesh_smoothing_weights"})
    scale = float(np.abs(want["vertices"]).max())
    assert float(np.abs(mwd.mesh.vertices - want["vertices"]).max()) <= REL * scale
    for name in ("wnn", "sw", "a"):
        assert float(np.abs(mwd.point_attributes[name] - want[name]).max()) <= REL * max(float(np.abs(want[name]).max()), 1.0), name
    assert float(np.abs(mwd.point_attributes["normals"] - want["normals"]).max()) <= 5e-5
    # (b) the reference pipeline on the same particles
    def run_reference():
        ps = oracle_mod.reference()
        rm, _ = ps.reconstruction_pipeline(x, mesh_cleanup=True, mesh_cleanup_snap_dist=0.5, decimate_barnacles=True, subdomain_grid=True, **kw, **post)
        return [len(np.asarray(rm.mesh.vertices)), len(np.asarray(rm.mesh.triangles))]
    rv, rt = reference_output("pipeline_with_mesh_cleanup_and_decimation.mesh_size", run_reference)
    assert abs(rv - mwd.mesh.nvertices) <= 0.01 * rv and abs(rt - mwd.mesh.ncells) <= 0.01 * rt, (rv, rt, mwd.mesh.nvertices, mwd.mesh.ncells)


@pytest.mark.gpu
def test_mesh_without_triangles_has_empty_connectivity(ss):
    """Vertices without any triangle (e.g. what `keep_vertices` leaves behind): empty adjacency lists like the reference's
    vertex_vertex_connectivity (their normals are 0/0 = NaN there as well: mesh.rs:879-906 normalises unconditionally)."""
    m = ss.TriMesh3d(np.random.default_rng(3).random((7, 3)).astype(np.float32), np.zeros((0, 3), np.uint64))
    assert m.vertex_vertex_connectivity().copy_connectivity() == [[] for _ in range(7)]
    assert np.isnan(m.vertex_normals_parallel()).all()


@pytest.mark.gpu
def test_pipeline_quads_mesh_aabb_and_checks(ss, oracle_mod):
    """The remaining switches of the pipeline mirror: generate_quads (reconstruct.rs:1410-1441), mesh_aabb_min / max (+ clamp,
    :1394-1408) and check_mesh_closed / check_mesh_manifold (:1445-1470) -- composed exactly like the free functions on the raw mesh."""
    from splashsurf_b200 import synthetic as syn
    x = syn.splash((10, 10, 10), 2, 0.025, 616)
    kw = dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.75, iso_surface_threshold=0.6)
    raw = ss.reconstruct_surface(x, **kw)
    # quads
    mwd, _ = ss.reconstruction_pipeline(x, generate_quads=True, quad_max_normal_angle=15.0, mesh_smoothing_weights=False, **kw)
    want = ss.convert_tris_to_quads(raw.mesh, normal_angle_limit=15.0)
    assert np.array_equal(mwd.mesh.get_quads(), want.get_quads()) and np.array_equal(mwd.mesh.get_triangles(), want.get_triangles())
    assert len(want.get_quads()) > 0
    # a closed, manifold mesh passes the checks; clamping it to a box opens it, and the closedness check then fails like the reference's
    ss.reconstruction_pipeline(x, check_mesh_closed=True, check_mesh_manifold=True, mesh_smoothing_weights=False, **kw)
    lo, hi = raw.mesh.vertices.min(0), raw.mesh.vertices.max(0)
    a, b = (lo + 0.2 * (hi - lo)).tolist(), (lo + 0.7 * (hi - lo)).tolist()
    mwd, _ = ss.reconstruction_pipeline(x, mesh_aabb_min=a, mesh_aabb_max=b, mesh_smoothing_weights=False, compute_normals=True, **kw)
    cm, _ = ss.clamp_mesh_with_aabb(raw.mesh, a, b)
    assert np.array_equal(mwd.mesh.vertices, cm.vertices) and np.array_equal(mwd.mesh.triangles, cm.triangles)
    assert mwd.point_attributes["normals"].shape == cm.vertices.shape and 0 < cm.ncells < raw.mesh.ncells
    with pytest.raises(ss.SplashsurfError) as e:
        ss.reconstruction_pipeline(x, mesh_aabb_min=a, mesh_aabb_max=b, check_mesh_closed=True, mesh_smoothing_weights=False, **kw)
    assert e.value.code == ss.SS_ERR_MESH_CHECK and "Mesh is not closed" in e.value.message
    ss.reconstruction_pipeline(x, check_mesh_orientation=True, mesh_smoothing_weights=False, **kw)       # a marching-cubes mesh is consistently oriented


@pytest.mark.gpu
def test_reference_python_tests_check_consistency_and_quads(ss):
    """pysplashsurf/tests/test_basic.py:193-268 (check_consistency_test, tris_to_quads_test) and test_calling.py:35 on the same anchor file
    with this package in the place of pysplashsurf."""
    import os
    from conftest import GOLDEN
    particles = np.load(os.path.join(GOLDEN, "cfg1_particles.npy"))
    rec = ss.reconstruct_surface(particles, particle_radius=0.025, rest_density=1000.0, smoothing_length=2.0, cube_size=1.0, iso_surface_threshold=0.6)
    assert ss.check_mesh_consistency(rec.mesh, rec.grid) is None
    mwd, rec2 = ss.reconstruction_pipeline(particles, particle_radius=0.025, rest_density=1000.0, smoothing_length=2.0, cube_size=1.0,
                                           iso_surface_threshold=0.6, mesh_smoothing_iters=5, output_mesh_smoothing_weights=True)
    assert ss.check_mesh_consistency(mwd, rec2.grid) is None
    q = ss.convert_tris_to_quads(mwd)
    assert type(q.mesh) is ss.MixedTriQuadMesh3d and q.nvertices == mwd.nvertices and q.ncells < mwd.ncells
    tris, quads = q.mesh.get_triangles(), q.mesh.get_quads()
    assert tris.dtype in (np.uint32, np.uint64) and quads.dtype in (np.uint32, np.uint64)
    assert tris.shape[1] == 3 and quads.shape[1] == 4 and len(tris) + 2 * len(quads) == mwd.ncells
    assert set(q.point_attributes) == set(mwd.point_attributes)
    ss.marching_cubes_cleanup(mwd, rec2.grid)                       # test_calling.py:35: accepts a MeshWithData
    assert mwd.mesh.nvertices < rec2.mesh.nvertices
