"""CPU tests: the C oracle against the reference's golden vectors (fixtures generated from the reference binary by
tools/make_golden.py) and against the reference's own known-answer tests."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, MESH_CASES, load_golden


@pytest.mark.parametrize("case", MESH_CASES)
def test_oracle_matches_reference_fixture(oracle_mod, case):
    g = load_golden(case)
    o = oracle_mod.reconstruct(g["particles"], **g["kwargs"])
    assert o["rc"] == 0
    # grid (lib.rs:476-516 + dense_subdomains.rs:168-188)
    assert np.array_equal(o["grid"]["aabb_min"], g["grid_min"])
    assert np.array_equal(o["grid"]["ncells"], g["grid_ncells"])
    # densities: bit-exact (density_map.rs:150-186 in the reference's summation order)
    assert np.array_equal(o["particle_densities"], g["densities"])
    # mesh: identical connectivity after canonical ordering; positions bit-exact away from subdomain faces
    m = oracle_mod.mesh_parity(o["vertices"], o["triangles"], o["vertex_keys"], g["vertices"], g["triangles"], g["keys"],
                               g["kwargs"].get("subdomain_num_cubes_per_dim", 64))
    assert m["keys_equal"] and m["triangles_equal"], m
    assert m["n_interior_not_bitexact"] == 0, m
    assert m["max_abs"] <= 2e-6, m     # boundary copies differ by ulps (which subdomain's copy the stitch keeps)


def test_oracle_single_particle_cases(oracle_mod):
    """tests/integration_tests/test_subdomains.rs:80-105 and test_simple.rs:99-126."""
    exp = json.load(open(os.path.join(GOLDEN, "single_particle.json")))
    for c in ("0.5", "0.1"):
        o = oracle_mod.reconstruct(np.zeros((1, 3), np.float32), particle_radius=0.025, smoothing_length=2.0, cube_size=float(c),
                                   subdomain_grid_auto_disable=False)
        assert (len(o["vertices"]), len(o["triangles"])) == (exp[c]["nv"], exp[c]["nt"])
        assert float(o["particle_densities"][0]) == exp[c]["rho"]
    # c = 0.025 r: the reference test's windows (the released wheel asserts on this input, see DESIGN.md)
    o = oracle_mod.reconstruct(np.zeros((1, 3), np.float32), particle_radius=0.025, smoothing_length=2.0, cube_size=0.025,
                               subdomain_grid_auto_disable=False)
    assert 90000 <= len(o["triangles"]) < 100000 and 45000 <= len(o["vertices"]) < 48000
    assert 330 <= int(np.prod(o["subdomain_grid"]["ncells"])) <= 350
    o = oracle_mod.reconstruct(np.array([[0.01, 0, 0]], np.float32), particle_radius=1.0, smoothing_length=0.5, cube_size=1.0,
                               iso_surface_threshold=0.1, subdomain_grid_auto_disable=False)
    assert (len(o["vertices"]), len(o["triangles"])) == (exp["simple"]["nv"], exp["simple"]["nt"]) == (6, 8)


def test_mc_lut_known_answers():
    """marching_cubes_lut.rs:427-451 KATs against the table the kernels and the oracle share."""
    cases = json.load(open(os.path.join(GOLDEN, "mc_lut_cases.json")))["emitted_triplets"]
    assert len(cases) == 256
    assert cases[0b00000001] == [[3, 8, 0]]
    assert cases[0b00010100] == [[10, 2, 1], [7, 4, 8]]
    assert cases[0] == [] and cases[255] == []
    inc = open(os.path.join(os.path.dirname(GOLDEN), "..", "splashsurf_b200", "csrc", "mc_lut.inc")).read()
    import re
    words = [int(w, 16) for w in re.findall(r"0x([0-9a-f]{16})ull", inc)]
    assert len(words) == 256
    for idx, (word, tl) in enumerate(zip(words, cases)):
        vals = [(word >> (4 * k)) & 0xF for k in range(16)]
        raw = [e for t in tl for e in (t[2], t[1], t[0])]
        assert vals[:len(raw)] == raw and all(v == 0xF for v in vals[len(raw):]), idx
    # complementary cases use the same edge sets
    for idx in range(256):
        a = sorted({e for t in cases[idx] for e in t}); b = sorted({e for t in cases[255 - idx] for e in t})
        assert a == b


def test_kernel_properties(oracle_mod):
    """kernel.rs:143-180 (compact support, unit integral) and :381-481 (AVX lane vs scalar tolerance)."""
    L = oracle_mod.lib()
    for h in (0.025, 0.1, 2.0):
        assert L.so_kernel_scalar(h, h) == 0.0 and L.so_kernel_scalar(h, 1.5 * h) == 0.0
        rs = np.linspace(0.0, 2.0 * h, 1024, dtype=np.float32)
        for r in rs:
            a, s = L.so_kernel_avx(h, float(r)), L.so_kernel_scalar(h, float(r))
            assert abs(a - s) <= max(1e-6, 1e-5 * abs(s))
    h, n = 1.0, 40
    dr = 2.0 * h / n
    xs = (-h + (np.arange(n) + 0.5) * dr).astype(np.float32)
    X, Y, Z = np.meshgrid(xs, xs, xs, indexing="ij")
    R = np.sqrt(X * X + Y * Y + Z * Z).astype(np.float32).ravel()
    total = sum(L.so_kernel_scalar(h, float(r)) for r in R) * dr ** 3
    assert abs(total - 1.0) < 1e-2


def test_grid_loop_fixture_oracle(oracle_mod):
    """benches/benches/bench_grid_loop.rs:203-262: AVX-semantics tile vs scalar tile on the reference's fixture,
    all |delta| < f32::EPSILON * 100."""
    g = load_golden("grid_loop_subdomain_33")
    kw = dict(global_min=g["global_min"], cube_size=g["cell_size"], subdomain_ijk=g["subdomain_ijk"], subdomain_cubes=64,
              subdomain_min=g["subdomain_min"], h=g["h"], rest_mass=g["rest_mass"])
    a = oracle_mod.levelset_tile(g["particles"], g["densities"], mode=0, **kw)
    s = oracle_mod.levelset_tile(g["particles"], g["densities"], mode=1, **kw)
    assert a.max() > 0.9 and np.abs(a - s).max() < np.finfo(np.float32).eps * 100


def _result_digests(oracle_mod, densities, vertices, triangles, keys, subdomain_cubes):
    """Digests of a reconstruction in canonical order: densities, MC edge keys, triangles and the vertices off the subdomain faces
    (equal digests = the densities bit-exact, connectivity identical, interior vertices bit-exact)."""
    from conftest import digest
    v, t, k = oracle_mod.canonicalize(np.asarray(vertices, np.float32), triangles, keys)
    onface = np.zeros(len(k), dtype=bool)
    for d in range(3):
        onface |= (k[:, 3] != d) & (k[:, d] % int(subdomain_cubes) == 0)
    return {"densities": digest(np.asarray(densities, np.float32)), "keys": digest(k), "triangles": digest(t.astype(np.int64)),
            "interior_vertices": digest(v[~onface]), "nv": len(v)}


def _reference_digests(oracle_mod, p, o, subdomain_cubes, **kw):
    """The reference binary's reconstruction of `p` as `_result_digests`; the oracle's result `o` only resolves the edge keys of
    vertices that sit on a lattice point."""
    r = oracle_mod.reference().reconstruct_surface(p, **kw)
    rv, rt = np.asarray(r.mesh.vertices), np.asarray(r.mesh.triangles)
    keys = oracle_mod.resolve_keys(rv, o["grid"]["aabb_min"], o["grid"]["cell_size"], o["vertex_keys"], rt, o["triangles"]) if len(rv) else np.zeros((0, 4), np.int64)
    return _result_digests(oracle_mod, r.particle_densities, rv, rt, keys, subdomain_cubes)


def test_oracle_vs_reference_binary_live(oracle_mod, reference_output):
    """Pin the restatement against the reference binary on a splash cloud that no other fixture uses (the reference's result is
    stored as digests in tests/golden/reference_outputs.json)."""
    from splashsurf_b200 import synthetic as syn
    p = syn.splash((18, 18, 18), 4, 0.025, seed=31337)
    kw = dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.55)
    o = oracle_mod.reconstruct(p, **kw)
    want = reference_output("oracle_live", lambda: _reference_digests(oracle_mod, p, o, 64, **kw))
    assert _result_digests(oracle_mod, o["particle_densities"], o["vertices"], o["triangles"], o["vertex_keys"], 64) == want


def test_oracle_fuzz_vs_reference_binary(oracle_mod, reference_output):
    """Randomised pin of the restatement against the reference binary: radii, smoothing lengths, cube sizes, subdomain sizes
    (also not multiples of 8), thresholds, rest densities, AVX / scalar loop, translated clouds (different rounding regime),
    subdomain and (auto-disabled) global path.  Densities bit-exact, connectivity identical, interior vertices bit-exact (the
    reference's results are stored as digests in tests/golden/reference_outputs.json)."""
    from splashsurf_b200 import synthetic as syn
    rng = np.random.default_rng(2024)
    checked = 0
    for case in range(14):
        r = float(rng.choice([0.01, 0.025, 0.05, 0.2]))
        kw = dict(particle_radius=r, smoothing_length=float(rng.choice([1.5, 2.0, 2.2, 2.5])), cube_size=float(rng.choice([0.4, 0.5, 0.75, 1.0, 1.3])),
                  iso_surface_threshold=float(rng.choice([0.3, 0.6, 0.8])), rest_density=float(rng.choice([1000.0, 850.0])),
                  simd=bool(rng.integers(0, 2)), subdomain_num_cubes_per_dim=int(rng.choice([16, 20, 24, 32, 50, 64])))
        p = syn.splash((int(rng.integers(6, 14)), int(rng.integers(4, 12)), int(rng.integers(4, 12))), int(rng.integers(0, 4)), r,
                       seed=int(rng.integers(0, 1e6)))
        p = (p.astype(np.float64) + rng.uniform(-50, 50, 3) * r * 20).astype(np.float32)
        o = oracle_mod.reconstruct(p, **kw)
        S = kw["subdomain_num_cubes_per_dim"]
        want = reference_output(f"oracle_fuzz.{case}", lambda: _reference_digests(oracle_mod, p, o, S, multi_threading=False, **kw))
        assert _result_digests(oracle_mod, o["particle_densities"], o["vertices"], o["triangles"], o["vertex_keys"], S) == want, kw
        checked += len(o["vertices"]) > 0
    assert checked >= 10


def test_oracle_sph_normals_fixture(oracle_mod):
    """SPH normals of the reference pipeline (fixture from the reference binary) vs the restatement: 2e-5 absolute on unit
    vectors (the reference sums in R-tree traversal order, the restatement in cell order)."""
    g = load_golden("sph_normals_ref")
    n = oracle_mod.sph_normals(g["particles"], g["densities"], g["vertices"], compact_support_radius=g["h"], particle_rest_mass=g["rest_mass"])
    assert np.abs(n - g["normals"]).max() <= 2e-5


def test_oracle_neighbor_lists_fixture(oracle_mod):
    """Neighbour lists of the reference binary (global_neighborhood_list=True) vs the restatement: identical lists, in order."""
    g = load_golden("neighbors_ref")
    o = oracle_mod.reconstruct(g["particles"], particle_radius=0.025, smoothing_length=2.0, cube_size=0.5, want_neighbors=True)
    off, idx = o["neighbors"]
    assert np.array_equal(off, g["offsets"]) and np.array_equal(idx, g["indices"])
