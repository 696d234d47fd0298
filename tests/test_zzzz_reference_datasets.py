"""The reference's own integration tests (splashsurf_lib/tests/integration_tests/test_full.rs:144-157): ten reconstructions of its eight
particle data sets with the parameters of those tests (no SIMD, sequential, compact support 4 r, auto_disable off; global and
subdomain-grid strategies, one with a particle AABB).  The reference asserts a triangle-count window and a closed, manifold mesh.
Here, on top of that: the reference's EXACT vertex / triangle counts, grid and particle densities (tests/golden/test_full.npz, generated
from the reference wheel by tools/make_golden_full.py) and the whole mesh bit for bit against the pinned oracle."""
import json
import os

import numpy as np
import pytest

from conftest import load_npz_parts

Z = load_npz_parts("test_full")
META = json.loads(str(Z["meta"]))
CASES = list(META)


def _case(name):
    m = META[name]
    return Z["particles:" + m["file"]], m["kwargs"], Z["densities:" + name], m


def _check_against_reference(name, particles, densities, nv, nt, grid_min, grid_ncells):
    _, _, ref_rho, m = _case(name)
    assert m["window"][0] < nt < m["window"][1]                                # test_full.rs:119-130
    assert (nv, nt) == (m["nv"], m["nt"])                                      # the reference's exact counts
    assert list(grid_ncells) == m["grid_ncells"] and [float(v) for v in grid_min] == m["grid_min"]
    assert np.array_equal(np.asarray(densities).view(np.uint32), ref_rho.view(np.uint32))       # bit for bit


@pytest.mark.parametrize("name", CASES)
def test_oracle_reproduces_the_reference_on_its_integration_data_sets(oracle_mod, name):
    p, kw, _, m = _case(name)
    o = oracle_mod.reconstruct(p, **kw)
    assert o["rc"] == 0 and o["used_decomposition"] == kw["subdomain_grid"]
    _check_against_reference(name, p, o["particle_densities"], len(o["vertices"]), len(o["triangles"]), o["grid"]["aabb_min"], o["grid"]["ncells"])
    if "aabb_min" in kw:
        assert o["particle_inside_aabb"].sum() == len(o["particle_densities"]) <= len(p)
    # closed + manifold like the reference's check_mesh_consistency (test_full.rs:132-139); the wheel's verdict is in the fixture
    import splashsurf_b200 as ss
    mesh = ss.TriMesh3d(o["vertices"], o["triangles"])
    assert m["consistent"] and ss.check_mesh_consistency(mesh, None, check_closed=True, check_manifold=True) is None


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_cuda_reference_integration_data_sets(ss, oracle_mod, name):
    """Through the C ABI on the GPU: the reference's counts, grid and densities (fixture) and the oracle's mesh, bit for bit."""
    p, kw, _, m = _case(name)
    g = ss.reconstruct_surface(p, with_debug=True, **kw)
    _check_against_reference(name, p, g.particle_densities, g.mesh.nvertices, g.mesh.ncells, g.grid.aabb.min, g.grid.ncells_per_dim)
    assert (g.subdomain_grid is not None) == kw["subdomain_grid"]
    o = oracle_mod.reconstruct(p, **kw)
    par = oracle_mod.mesh_parity(g.mesh.vertices, g.mesh.triangles, g.vertex_edge_keys, o["vertices"], o["triangles"], o["vertex_keys"], 64)
    assert par["keys_equal"] and par["triangles_equal"] and par["n_not_bitexact"] == 0, par
    assert ss.check_mesh_consistency(g.mesh, g.grid, check_closed=True, check_manifold=True) is None


# ---- hand-made neighbourhood cases of the reference (tests/integration_tests/test_neighborhood_search.rs:11-86), search radius 0.3 = the
# compact support radius of the reconstruction (h = 2 * smoothing_length * particle_radius = 2 * 2.0 * 0.075, exact in f32)
def _ns_cases(sr):
    return [
        ([[1, 1, 1], [1 + sr, 1 + sr, 1 + sr]], [[], []]),
        ([[1, 1, 1], [1 + 0.9999 * sr, 1, 1]], [[1], [0]]),
        ([[1, 1, 1], [1 + sr, 1, 1]], [[1], [0]]),                            # f32: (1 + 0.3) - 1 < 0.3
        ([[1, 1, 1], [1 + sr * 1.0001, 1, 1]], [[], []]),
        ([[1, 1, 1], [1 + 0.9 * sr, 1, 1], [1 - 0.9 * sr, 1, 1], [1, 1 + 0.2 * sr, 1]], [[1, 2, 3], [0, 3], [0, 3], [0, 1, 2]]),
        ([[1, 1, 1], [1 + 0.9 * sr, 1, 1], [1 - 0.9 * sr, 1, 1], [1 - 0.8 * sr, 1, -0.2 * sr], [1, 1 + 0.2 * sr, 1], [1, 1 - 0.2 * sr, 1],
          [1, 1 + 0.2 * sr, 1 + 0.2 * sr], [1, 1 - 0.2 * sr, 1 - 0.2 * sr]],
         [[1, 2, 4, 5, 6, 7], [0, 4, 5, 6, 7], [0, 4, 5, 6, 7], [], [0, 1, 2, 5, 6, 7], [0, 1, 2, 4, 6, 7], [0, 1, 2, 4, 5, 7], [0, 1, 2, 4, 5, 6]]),
    ]


def _ns_particles(rows, sr):
    # the reference builds every coordinate in f32 arithmetic (Vector3<f32>::new(1.0 + 0.9 * search_radius, ...))
    f = np.float32
    one, s = f(1.0), f(sr)
    table = {1: one, 1 + sr: one + s, 1 + 0.9999 * sr: one + f(0.9999) * s, 1 + sr * 1.0001: one + s * f(1.0001), 1 + 0.9 * sr: one + f(0.9) * s,
             1 - 0.9 * sr: one - f(0.9) * s, 1 + 0.2 * sr: one + f(0.2) * s, 1 - 0.2 * sr: one - f(0.2) * s, 1 - 0.8 * sr: one - f(0.8) * s,
             -0.2 * sr: f(-0.2) * s}
    return np.array([[table[v] for v in row] for row in rows], dtype=np.float32)


NS_KW = dict(particle_radius=0.075, smoothing_length=2.0, cube_size=1.0)


def _check_ns(reconstruct, neighbors_of):
    for rows, expect in _ns_cases(0.3):
        p = _ns_particles(rows, 0.3)
        for extra in (dict(subdomain_grid_auto_disable=False), dict(subdomain_grid=False)):     # per-subdomain search and global search
            got = neighbors_of(reconstruct(p, **NS_KW, **extra), len(p))
            assert [sorted(g) for g in got] == expect, (rows, extra, got)


def test_oracle_neighborhood_hand_cases(oracle_mod):
    def nbrs(o, n):
        off, idx = o["neighbors"]
        return [idx[off[i]:off[i + 1]].tolist() for i in range(n)]
    _check_ns(lambda p, **kw: oracle_mod.reconstruct(p, want_neighbors=True, **kw), nbrs)


@pytest.mark.gpu
def test_cuda_neighborhood_hand_cases(ss):
    _check_ns(lambda p, **kw: ss.reconstruct_surface(p, global_neighborhood_list=True, **kw), lambda g, n: [g.particle_neighbors[i] for i in range(n)])


# ---- SphInterpolator at arbitrary points (sph_interpolation.rs:22-258; pysplashsurf.SphInterpolator): the oracle's restatements (pinned to
# the wheel, tests/test_oracle_postprocess.py) and the wheel's own class (its results in tests/golden/sph_interpolator_ref.npz); tolerance 2e-5
# (f32 sums in another order)
def check_sph_interpolator(ss, oracle_mod, reference_output):
    from conftest import GOLDEN, digest, load_golden
    from oracle import postprocess as opp
    from splashsurf_b200 import synthetic as syn
    p = syn.splash((12, 12, 12), 3, 0.025, 77)
    rho = oracle_mod.reconstruct(p, particle_radius=0.025, smoothing_length=2.0, cube_size=0.75)["particle_densities"]
    h, m = np.float32(0.1), float(oracle_mod.sph_rest_mass(0.025))
    rng = np.random.default_rng(1)
    near = p[::7] + rng.normal(scale=0.02, size=(len(p[::7]), 3)).astype(np.float32)
    x = np.concatenate([near, np.float32([[50, 50, 50], [-3, 0, 0]])]).astype(np.float32)        # the last two see no particle
    sc, ve = rng.normal(size=len(p)).astype(np.float32), rng.normal(size=(len(p), 3)).astype(np.float32)

    def run_reference():                    # the wheel's results are stored in tests/golden/sph_interpolator_ref.npz
        it_ref = oracle_mod.reference().SphInterpolator(p, rho, m, float(h))
        arrays = {f"quantity_{int(corr)}_{q.ndim}": np.asarray(it_ref.interpolate_quantity(q, x, first_order_correction=corr))
                  for corr in (False, True) for q in (sc, ve)}
        arrays["normals"] = np.asarray(it_ref.interpolate_normals(x))
        np.savez_compressed(os.path.join(GOLDEN, "sph_interpolator_ref.npz"), **arrays)
        return digest(*[arrays[k] for k in sorted(arrays)])
    want = reference_output("sph_interpolator", run_reference)
    ref = load_golden("sph_interpolator_ref")
    assert digest(*[ref[k] for k in sorted(ref)]) == want
    it = ss.SphInterpolator(p, rho, m, float(h))
    for corr in (False, True):
        for q in (sc, ve):
            g = it.interpolate_quantity(q, x, first_order_correction=corr)
            o = opp.interpolate_quantity(p, rho, m, h, q, x, first_order_correction=corr)
            assert g.shape == o.shape and g.dtype == np.float32
            assert np.isnan(g[-2:]).all() and np.isfinite(g[:-2]).all()              # 0 * inf + ... = NaN without neighbours (:252-254)
            assert np.abs(g[:-2] - o[:-2]).max() <= 2e-5 * max(1.0, float(np.abs(o[:-2]).max()))
            r = ref[f"quantity_{int(corr)}_{q.ndim}"]
            assert np.array_equal(np.isnan(r), np.isnan(g)) and np.abs(g[:-2] - r[:-2]).max() <= 2e-5 * max(1.0, float(np.abs(r[:-2]).max()))
    g = it.interpolate_normals(x)
    o = oracle_mod.sph_normals(p, rho, x[:-2], compact_support_radius=h, particle_rest_mass=m)
    assert np.isnan(g[-2:]).all() and np.abs(np.linalg.norm(g[:-2], axis=1) - 1.0).max() < 1e-5 and np.abs(g[:-2] - o).max() <= 2e-5
    assert np.abs(g[:-2] - ref["normals"][:-2]).max() <= 2e-5
    # no particles at all; argument checks; sharing a context: the bins are gone after the next reconstruction on it
    e = ss.SphInterpolator(np.zeros((0, 3), np.float32), np.zeros(0, np.float32), m, float(h))
    assert np.isnan(e.interpolate_quantity(np.zeros(0, np.float32), x[:3])).all() and np.isnan(e.interpolate_normals(x[:3])).all()
    assert it.interpolate_normals(np.zeros((0, 3), np.float32)).shape == (0, 3)
    with pytest.raises(ValueError):
        it.interpolate_quantity(sc[:-1], x)
    with pytest.raises(TypeError):
        it.interpolate_normals(x.astype(np.float64))
    ctx = ss.Context()
    shared = ss.SphInterpolator(p, rho, m, float(h), context=ctx)
    assert np.array_equal(shared.interpolate_normals(x[:5]), g[:5])
    ss.reconstruct_surface(p[:200], particle_radius=0.025, smoothing_length=2.0, cube_size=1.0, context=ctx)
    with pytest.raises(ss.SplashsurfError, match="particle bins of this interpolator are gone"):
        shared.interpolate_normals(x[:5])
    assert np.array_equal(it.interpolate_normals(x[:5]), g[:5])                        # its own context: still valid
    for o_ in (shared, it, e):
        o_.close()
    ctx.close()


# ---- stand-alone neighbourhood search (neighborhood_search.rs:444-588; pysplashsurf/tests/test_basic.py:150-182): the reference's hand
# cases, a random cloud against a k-d tree and against the wheel's function, the lists of the reconstruction itself
def _lists_digest(lists):
    from conftest import digest
    return digest(np.array([len(l) for l in lists], np.int64), np.array([i for l in lists for i in l], np.int64))


def check_neighborhood_search(ss, oracle_mod, reference_output):
    from scipy.spatial import cKDTree
    from splashsurf_b200 import synthetic as syn
    def grown(points, r):                                             # Aabb3d::from_points + grow_uniformly (test_neighborhood_search.rs:104-106)
        return ss.Aabb3d((points.min(axis=0) - np.float32(r)).astype(np.float32), (points.max(axis=0) + np.float32(r)).astype(np.float32))

    def naive(points, r):                                             # neighborhood_search_naive: |dx|^2 < r^2 in f32
        pairs = cKDTree(points.astype(np.float64)).query_pairs(float(r) * 1.001, output_type="ndarray")
        dx = points[pairs[:, 0]] - points[pairs[:, 1]]
        keep = (dx[:, 0] * dx[:, 0] + dx[:, 1] * dx[:, 1] + dx[:, 2] * dx[:, 2]).astype(np.float32) < np.float32(r) * np.float32(r)
        out = [[] for _ in range(len(points))]
        for a, b in pairs[keep]:
            out[a].append(int(b)); out[b].append(int(a))
        return [sorted(l) for l in out]
    for rows, expect in _ns_cases(0.3):                               # test_neighborhood_search_spatial_hashing_parallel_simple (:152-176)
        p = _ns_particles(rows, 0.3)
        nl = ss.neighborhood_search_spatial_hashing_parallel(p, grown(p, 0.3), float(np.float32(0.3)))
        assert type(nl) is ss.NeighborhoodLists and [sorted(l) for l in nl.get_neighborhood_lists()] == expect
    # test_compare_free_particles_125 / _1000 (:184-300): the naive search against the spatial hashing on the reference's data sets
    for name, r in (("free_particles_125_particles.vtk", 1.0), ("free_particles_1000_particles.vtk", 1.0), ("bunny_frame_14_7705_particles.vtk", 0.1)):
        q = Z["particles:" + name]
        nl = ss.neighborhood_search_spatial_hashing_parallel(q, grown(q, r), r)
        assert [sorted(l) for l in nl.get_neighborhood_lists()] == naive(q, r), name
    p = syn.splash((14, 14, 14), 3, 0.025, 91)
    sr = float(np.float32(0.1))
    rec = ss.reconstruct_surface(p, particle_radius=0.025, smoothing_length=2.0, cube_size=1.0, global_neighborhood_list=True)
    nl = ss.neighborhood_search_spatial_hashing_parallel(p, rec.grid.aabb, sr)
    got = [sorted(l) for l in nl.get_neighborhood_lists()]
    assert len(got) == len(p) and got == [sorted(l) for l in rec.particle_neighbors.get_neighborhood_lists()]     # test_basic.py:150-182
    d = p.astype(np.float64)
    pairs = cKDTree(d).query_pairs(sr * 1.001, output_type="ndarray")
    dx = p[pairs[:, 0]] - p[pairs[:, 1]]                                       # the reference's f32 test: |dx|^2 < r^2
    keep = (dx[:, 0] * dx[:, 0] + dx[:, 1] * dx[:, 1] + dx[:, 2] * dx[:, 2]).astype(np.float32) < np.float32(sr) * np.float32(sr)
    brute = [[] for _ in range(len(p))]
    for a, b in pairs[keep]:
        brute[a].append(int(b)); brute[b].append(int(a))
    mism = [i for i in range(len(p)) if sorted(brute[i]) != got[i]]
    # pairs whose squared distance rounds differently in another summation order sit exactly on the radius: none are expected in this cloud
    assert not mism, mism[:5]

    def run_reference():                    # the wheel's lists, stored by their digest
        ps = oracle_mod.reference()
        ref = ps.neighborhood_search_spatial_hashing_parallel(p, domain=ps.Aabb3d.from_min_max(rec.grid.aabb.min, rec.grid.aabb.max), search_radius=sr)
        return _lists_digest([sorted(l) for l in ref.get_neighborhood_lists()])
    assert reference_output("neighborhood_search.splash14", run_reference) == _lists_digest(got)
    assert len(ss.neighborhood_search_spatial_hashing_parallel(np.zeros((0, 3), np.float32), rec.grid.aabb, sr)) == 0
    with pytest.raises(ss.SplashsurfError, match="outside of the domain"):
        ss.neighborhood_search_spatial_hashing_parallel(p, ss.Aabb3d(np.float32([0, 0, 0]), np.float32([0.2, 0.2, 0.2])), sr)
    with pytest.raises(ss.SplashsurfError, match="search radius must be positive"):
        ss.neighborhood_search_spatial_hashing_parallel(p, rec.grid.aabb, 0.0)


# ---- marching cubes on a dense array (pysplashsurf.marching_cubes = marching_cubes::triangulate_density_map): the reference's one-cell
# known-answer test (marching_cubes.rs:325-396), its sphere-SDF test (pysplashsurf/tests/test_sdf.py) and random fields of awkward shapes
# (borders with values on both sides of the threshold, arrays that do not fill whole tiles) against the wheel's function
def _canonical_mesh(v, t):
    """Vertices sorted by position; triangles in terms of the sorted positions (coincident vertices -- an interpolation weight that rounds to
    0 puts two vertices of neighbouring edges on the same grid point -- share one number, so their order cannot matter), rotated to their
    smallest number and sorted."""
    o = np.lexsort(v.T[::-1])
    rank = np.empty(len(v), np.int64)
    vs = v[o].view(np.uint32).reshape(-1, 3) if len(v) else np.zeros((0, 3), np.uint32)
    group = np.cumsum(np.r_[True, (vs[1:] != vs[:-1]).any(axis=1)]) - 1 if len(v) else np.zeros(0, np.int64)
    rank[o] = group
    t = rank[np.asarray(t).astype(np.int64)]
    if len(t):
        t = np.stack([np.roll(row, -s) for row, s in zip(t, np.argmin(t, axis=1))])
        t = t[np.lexsort(t.T[::-1])]
    return v[o], t


def _mesh_digest(v, t):
    from conftest import digest
    cv, ct = _canonical_mesh(np.asarray(v, np.float32), np.asarray(t))
    return digest(cv.view(np.uint32), ct)


def check_marching_cubes(ss, oracle_mod, reference_output):
    # one cell (marching_cubes.rs:325-396): threshold 0.25, six vertices on the local edges 0, 3, 5, 6, 9, 11
    vals = np.zeros((2, 2, 2), np.float32)
    for (i, j, k), val in (((0, 0, 0), 0.0), ((1, 0, 0), 0.75), ((1, 1, 0), 1.0), ((0, 1, 0), 0.5), ((0, 0, 1), 0.0), ((1, 0, 1), 0.0), ((1, 1, 1), 1.0),
                           ((0, 1, 1), 0.0)):
        vals[i, j, k] = val
    mesh, grid = ss.marching_cubes(vals, iso_surface_threshold=0.25, cube_size=1.0, return_grid=True)
    assert np.array_equal(grid.aabb.max, np.float32([1, 1, 1])) and grid.ncells_per_dim == [1, 1, 1] and grid.npoints_per_dim == [2, 2, 2]
    expect = np.float32([[1 / 3, 0, 0], [0, 0.5, 0], [1, 0.25, 1], [0.25, 1, 1], [1, 0, 2 / 3], [0, 1, 0.5]])
    assert mesh.vertices.shape == (6, 3) and mesh.triangles.dtype == np.uint64
    assert np.abs(_canonical_mesh(mesh.vertices, mesh.triangles)[0] - expect[np.lexsort(expect.T[::-1])]).max() < 1e-6
    assert len(mesh.triangles) == 4                                    # a hexagon: corners 1, 2, 3, 6 are inside
    empty = ss.marching_cubes(np.zeros((3, 4, 5), np.float32), iso_surface_threshold=0.25, cube_size=1.0)
    assert empty.vertices.shape == (0, 3) and empty.triangles.shape == (0, 3)
    # sphere SDF (pysplashsurf/tests/test_sdf.py): values grow towards the outside, so the surface is seen "inside out" -- still one closed sphere
    n, radius = 100, 1.0
    dx = radius * 2.2 / (n - 1)
    tr = -0.5 * radius * 2.2
    c = np.arange(n, dtype=np.float32) * np.float32(dx) + np.float32(tr)
    x, y, z = np.meshgrid(c, c, c, indexing="ij")
    sdf = (np.sqrt(x**2 + y**2 + z**2) - radius).astype(np.float32)
    mesh, grid = ss.marching_cubes(sdf, iso_surface_threshold=0.0, cube_size=dx, translation=[tr] * 3, return_grid=True)
    norms = np.linalg.norm(mesh.vertices, axis=1)
    assert len(mesh.vertices) > 0 and norms.min() > radius - 1e-4 and norms.max() < radius + 1e-4
    assert ss.check_mesh_consistency(mesh, grid) is None
    cases = [(sdf, 0.0, dx, [tr] * 3)]
    rng = np.random.default_rng(3)
    from scipy.ndimage import gaussian_filter
    for shape in ((5, 9, 3), (66, 65, 70), (130, 20, 67)):
        cases.append((gaussian_filter(rng.normal(size=shape), 1.5).astype(np.float32), 0.01, 0.3, [0.5, -2.0, 7.0]))
    for ci, (f, thr, cs, t) in enumerate(cases):
        m = ss.marching_cubes(f, iso_surface_threshold=thr, cube_size=cs, translation=t)
        # every vertex lies on a grid edge inside the array; every triangle is a valid one
        q = (m.vertices.astype(np.float64) - np.asarray(t)) / cs
        assert q.min() > -1e-4 and (q.max(axis=0) < np.asarray(f.shape) - 1 + 1e-4).all() and int(m.triangles.max()) < len(m.vertices)

        def run_reference():
            r = oracle_mod.reference().marching_cubes(f, iso_surface_threshold=thr, cube_size=cs, translation=t)
            return _mesh_digest(r.vertices, r.triangles)
        assert _mesh_digest(m.vertices, m.triangles) == reference_output(f"marching_cubes.field{ci}", run_reference)      # bit for bit
    # values exactly ON the threshold: inside for the vertex pass, for the case index only next to a value below (narrow_band_extraction.rs:
    # 79-126, :179-184).  Consistent arrays give the reference's mesh; where the table would ask for a vertex nobody created the reference
    # stops with "Missing iso surface vertex" and so does this front end (it never returns a mesh the reference would not)
    f = np.zeros((3, 3, 3), np.float32)
    f[1, 1, 1], f[0, 1, 1] = 1.0, 0.5
    m = ss.marching_cubes(f, iso_surface_threshold=0.5, cube_size=1.0)
    assert (len(m.vertices), len(m.triangles)) == (9, 12)
    f[:] = 1.0
    f[1, 1, 1] = 0.5                                                   # on the threshold, every neighbour above it
    with pytest.raises(ss.SplashsurfError, match="Missing iso surface vertex"):
        ss.marching_cubes(f, iso_surface_threshold=0.5, cube_size=1.0)
    agree = refused = 0
    for seed in range(40):
        rs = np.random.default_rng(seed)
        g = rs.normal(size=(6, 5, 7)).astype(np.float32)
        g.reshape(-1)[rs.integers(0, g.size, size=3)] = 1.0            # three values exactly on the threshold
        try:
            m = ss.marching_cubes(g, iso_surface_threshold=1.0, cube_size=0.5)
        except ss.SplashsurfError:
            refused += 1
            continue
        assert int(m.triangles.max(initial=0)) < max(len(m.vertices), 1)

        def run_reference():
            r = oracle_mod.reference().marching_cubes(g, iso_surface_threshold=1.0, cube_size=0.5)
            return _mesh_digest(r.vertices, r.triangles)
        assert _mesh_digest(m.vertices, m.triangles) == reference_output(f"marching_cubes.on_threshold{seed}", run_reference)
        agree += 1
    assert refused > 0 and agree > 0
    with pytest.raises(ValueError):
        ss.marching_cubes(np.zeros((4, 4), np.float32), iso_surface_threshold=0.0, cube_size=1.0)
    with pytest.raises(TypeError):
        ss.marching_cubes(np.zeros((4, 4, 4)), iso_surface_threshold=0.0, cube_size=1.0)
    with pytest.raises(ss.SplashsurfError):
        ss.marching_cubes(np.zeros((4, 4, 4), np.float32), iso_surface_threshold=0.0, cube_size=0.0)


# ---- the command line on the device: a frame sequence on one context (pooled buffers reused from frame to frame), files equal to what the
# library calls give frame by frame
def check_cli_sequence(ss, tmp_path):
    from splashsurf_b200 import io, synthetic as syn, __main__ as cli
    frames = tmp_path / "frames"
    frames.mkdir()
    clouds = {i: syn.splash((7 + i, 7, 7), 2, 0.025, 800 + i) for i in (1, 2, 3)}            # growing clouds: the pooled buffers have to grow
    for i, p in clouds.items():
        io.write_particles(str(frames / f"f_{i}.bgeo"), p)
    out = tmp_path / "out"
    assert cli.main(["reconstruct", str(frames / "f_{}.bgeo"), "-r=0.025", "-l=2.0", "-c=0.75", "--normals=on", "--sph-normals=on", "--output-dir", str(out),
                     "-o", "m_{}.ply", "-q"]) == 0
    assert sorted(os.listdir(out)) == ["m_1.ply", "m_2.ply", "m_3.ply"]
    for i, p in clouds.items():
        v, t, _, attrs = io.read_ply_mesh(str(out / f"m_{i}.ply"))
        mesh, _ = ss.reconstruction_pipeline(p, particle_radius=0.025, smoothing_length=2.0, cube_size=0.75, compute_normals=True, sph_normals=True,
                                             subdomain_grid_auto_disable=False)
        assert np.array_equal(v, mesh.mesh.vertices) and np.array_equal(t.astype(np.uint64), mesh.mesh.triangles.astype(np.uint64))
        assert np.array_equal(attrs["normals"], mesh.point_attributes["normals"])


# ---- tests/integration_tests/test_simple.rs:68-126: one particle whose only surface-crossing edges run from a point above the threshold to a
# point outside of the compact support -- 6 vertices, 8 triangles, closed and manifold, with the global and the subdomain-grid strategy
def check_test_simple(reconstruct, ss):
    p = np.array([[0.01, 0.0, 0.0]], np.float32)
    for grid in (False, True):
        r = reconstruct(p, particle_radius=1.0, smoothing_length=0.5, cube_size=1.0, iso_surface_threshold=0.1, multi_threading=False, simd=False,
                        subdomain_grid=grid, subdomain_grid_auto_disable=False)
        v, t = (r["vertices"], r["triangles"]) if isinstance(r, dict) else (r.mesh.vertices, r.mesh.triangles)
        assert (len(v), len(t)) == (6, 8), (grid, len(v), len(t))
        assert ss.check_mesh_consistency(ss.TriMesh3d(v, t), None, check_closed=True, check_manifold=True) is None


def test_oracle_test_simple(oracle_mod):
    import splashsurf_b200 as ss
    check_test_simple(oracle_mod.reconstruct, ss)


@pytest.mark.gpu
def test_cuda_test_simple(ss):
    check_test_simple(ss.reconstruct_surface, ss)


# ---- GPU-marked wrappers of the entries added after the last GPU session: last in the file (the suite runs with -x)
@pytest.mark.gpu
def test_cuda_sph_interpolator_at_arbitrary_points(ss, oracle_mod, reference_output):
    check_sph_interpolator(ss, oracle_mod, reference_output)


@pytest.mark.gpu
def test_cuda_neighborhood_search_stand_alone(ss, oracle_mod, reference_output):
    check_neighborhood_search(ss, oracle_mod, reference_output)


@pytest.mark.gpu
def test_cuda_marching_cubes_on_a_dense_array(ss, oracle_mod, reference_output):
    check_marching_cubes(ss, oracle_mod, reference_output)


@pytest.mark.gpu
def test_cuda_cli_frame_sequence(ss, tmp_path):
    check_cli_sequence(ss, tmp_path)
