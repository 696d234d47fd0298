"""Reconstructions on a reused context whose pooled scratch still holds what earlier calls left in it.

Level-set variant 2 (the default) does not zero-fill the tiles and the warp-per-brick marching cubes do not zero-fill the edge
masks: every value a later pass reads has to be written in the same frame (ss_pipeline.cu, ss_certify.cuh: k_zero_untouched).
A fresh context cannot show a break in that rule -- new device memory reads 0, which is the value a missed point should have --
so these tests run many reconstructions on ONE context and fill its tiles with "inside" values first (through the stand-alone
marching cubes, which copy caller values straight into the tiles).  A point a pass forgets to write then becomes extra surface.

Every reconstruction is compared with the pinned oracle bit for bit (densities, subdomain lists, mesh) and with the same call on
a fresh context (raw arrays: vertex and triangle order included).  The checks are `check_*(ss, oracle_mod)` functions, run on
the B200 (GPU-marked) and, reduced, on the CPU executor of the CUDA sources in its non-guard build (the guard build reallocates
every buffer whose size changes, which would drop the poison)."""
import ctypes as C
import importlib.util
import math
import os

import numpy as np
import pytest

from conftest import ROOT

SS_MARKER = np.float32(3.0e38)              # ss_kernels.cuh: "certified inside, exact value not computed"
POISONS = ("marker", "thr_plus_ulp", "plus_1e3", "nan")
TILE = 65                                   # points per dimension of a marching-cubes tile (64 cells)


def _random_case():
    """tools/fuzz_emulated.py:random_case, so that the clouds follow the executor fuzz's distribution."""
    spec = importlib.util.spec_from_file_location("fuzz_emulated", os.path.join(ROOT, "tools", "fuzz_emulated.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.random_case


def pick_seeds(base: int, n_subdomain: int, n_other: int) -> list:
    """The first `n_subdomain` seeds from `base` on whose case forces the subdomain grid (the tiles that are not zero-filled belong
    to it) and the first `n_other` whose case takes the global path or decides by itself, in seed order."""
    random_case = _random_case()
    sub, other, seed = [], [], base
    while len(sub) < n_subdomain or len(other) < n_other:
        _, kw, _ = random_case(np.random.default_rng(seed))
        bucket, n = (sub, n_subdomain) if kw.get("subdomain_grid_auto_disable") is False else (other, n_other)
        if len(bucket) < n:
            bucket.append(seed)
        seed += 1
    return sorted(sub + other)


def switches_for(i: int) -> dict:
    """Context switches of the i-th case: every switch cycles with its own period, so that the combinations vary.  Variant 2 (the
    default, no zero-fill of the tiles) comes up in three cases out of five, exact-everywhere (which zero-fills) in one out of seven."""
    return dict(variant=(2, 2, 1, 2, 0)[i % 5], exact=i % 7 == 6, batch=(0, 1, 3)[i % 3], mc=(i // 3) % 2, density=(i // 4) % 3)


def rejected_variant(i: int, x, kw):
    """A call the oracle refuses, made on the reused context between two cases: no cube size, or a negative particle radius."""
    return x, (dict(kw, cube_size=0.0) if i % 2 else dict(kw, particle_radius=-kw["particle_radius"]))


def apply_switches(ctx, sw: dict) -> None:
    ctx.set_levelset_variant(sw["variant"])
    ctx.set_levelset_exact_everywhere(sw["exact"])
    ctx.set_tile_batch(sw["batch"])             # 0: as many tiles per batch as fit
    ctx.set_mc_variant(sw["mc"])
    ctx.set_density_variant(sw["density"])


def poison_value(kind: str, thr) -> np.float32:
    thr = np.float32(thr)
    return {"marker": SS_MARKER, "thr_plus_ulp": np.nextafter(thr, np.float32(np.inf)), "plus_1e3": np.float32(1e3),
            "nan": np.float32(np.nan)}[kind]


def tiles_used(o: dict, kw: dict, batch: int) -> int:
    """Level-set tiles one batch of the reconstruction holds at most, in units of 65^3-point marching-cubes tiles."""
    if o["used_decomposition"]:
        S, n = int(kw.get("subdomain_num_cubes_per_dim", 64)), len(o["subdomain_flat"])
    else:
        S, n = 64, int(np.prod([(int(c) + 63) // 64 for c in o["grid"]["ncells"]]))
    k = max(1, min(n, batch) if batch else n)
    return max(1, math.ceil(k * (S + 1) ** 3 / TILE ** 3))


def poison_tiles(ss, ctx, ntiles: int, kind: str, thr) -> None:
    """Fills the first `ntiles` 65^3 tiles of the context's tile buffer with `kind` by triangulating a dense array on it; each tile
    keeps one point below the threshold, so that the front end does not skip it as a tile without a sign change."""
    v = np.full((64 * ntiles + 1, TILE, TILE), poison_value(kind, thr), np.float32)
    v[32::64, 32, 32] = np.float32(thr) - np.float32(1.0)
    ss.marching_cubes(v, iso_surface_threshold=float(thr), cube_size=1.0, context=ctx)


def assert_matches_oracle(oracle_mod, g, o, kw, tag):
    assert np.array_equal(g.particle_densities, o["particle_densities"]), f"{tag}: densities differ from the oracle"
    if o["used_decomposition"]:
        assert np.array_equal(g.subdomains["flat"], o["subdomain_flat"]), f"{tag}: subdomain indices differ from the oracle"
        assert np.array_equal(g.subdomains["sparse"], o["subdomain_sparse"]), f"{tag}: sparse flags differ from the oracle"
    if o.get("particle_inside_aabb") is not None:
        assert np.array_equal(g.particle_inside_aabb, o["particle_inside_aabb"]), f"{tag}: AABB filter differs from the oracle"
    m = oracle_mod.mesh_parity(g.mesh.vertices, g.mesh.triangles, g.vertex_edge_keys, o["vertices"], o["triangles"], o["vertex_keys"],
                               kw.get("subdomain_num_cubes_per_dim", 64))
    assert m["keys_equal"] and m["triangles_equal"] and m["n_not_bitexact"] == 0, f"{tag}: mesh differs from the oracle: {m}"


def _raw(g) -> dict:
    d = {"vertices": g.mesh.vertices, "triangles": g.mesh.triangles, "densities": g.particle_densities, "keys": g.vertex_edge_keys}
    if g.subdomains is not None:
        d.update({"sub_" + k: v for k, v in g.subdomains.items()})
    if g.particle_inside_aabb is not None:
        d["inside"] = g.particle_inside_aabb
    return d


def assert_raw_equal(a: dict, b: dict, tag: str):
    assert sorted(a) == sorted(b), tag
    for k in a:
        x, y = np.ascontiguousarray(a[k]), np.ascontiguousarray(b[k])
        assert x.dtype == y.dtype and x.shape == y.shape and x.tobytes() == y.tobytes(), f"{tag}: {k} differs"    # bit for bit, NaNs too


def on_fresh_context(ss, sw, call):
    ctx = ss.Context()
    try:
        if sw is not None:
            apply_switches(ctx, sw)
        return call(ctx)
    finally:
        ctx.close()


# ------------------------------------------------------------------ 1. fuzz cases on one poisoned context ----
def _expect_rejection(ss, oracle_mod, ctx, x, kw, tag):
    o = oracle_mod.reconstruct(x, **kw)
    assert o["rc"] != 0, f"{tag}: the oracle accepted the call"
    with pytest.raises(ss.SplashsurfError) as e:
        ss.reconstruct_surface(x, context=ctx, **kw)
    assert e.value.code == o["rc"], f"{tag}: error code {e.value.code}, the oracle's is {o['rc']}"


def check_poisoned_pool(ss, oracle_mod, seeds, max_points=6e6, reject_every=8):
    """The fuzz cases `seeds` one after another on ONE context, every switch set explicitly before each case and the tiles filled
    with an "inside" value (or NaN) first.  Nothing is reset between cases, so each one also reads what the previous one left in
    the edge masks, vertex ids, brick states and bins.  After every `reject_every`-th case a call the oracle refuses must fail with
    the oracle's error code, and the next case on the context must still pass.  Returns the number of cases compared."""
    random_case = _random_case()
    ctx = ss.Context()
    ran, after_error = 0, None
    try:
        for i, seed in enumerate(seeds):
            x, kw, _ = random_case(np.random.default_rng(seed))
            sw, kind = switches_for(i), POISONS[i % len(POISONS)]
            tag = f"seed={seed} poison={kind} switches={sw} n={len(x)} kw={kw}"
            o = oracle_mod.reconstruct(x, **kw)
            apply_switches(ctx, sw)
            if o["rc"] != 0:
                _expect_rejection(ss, oracle_mod, ctx, x, kw, tag)
                after_error = tag
                continue
            if float(np.prod(o["grid"]["npoints"].astype(np.float64))) > max_points:
                continue
            poison_tiles(ss, ctx, tiles_used(o, kw, sw["batch"]), kind, kw["iso_surface_threshold"])
            apply_switches(ctx, sw)
            try:
                g = ss.reconstruct_surface(x, with_debug=True, context=ctx, **kw)
            except ss.SplashsurfError as e:
                raise AssertionError(f"{tag}: the device path failed ({e.code}: {e}) where the oracle succeeded") from e
            assert_matches_oracle(oracle_mod, g, o, kw, tag)
            fresh = on_fresh_context(ss, sw, lambda c: ss.reconstruct_surface(x, with_debug=True, context=c, **kw))
            assert_raw_equal(_raw(g), _raw(fresh), f"{tag}: reused vs fresh context")
            ran, after_error = ran + 1, None
            if ran % reject_every == 0:
                xr, kwr = rejected_variant(ran // reject_every, x, kw)
                after_error = f"rejected call after {tag}: kw={kwr}"
                _expect_rejection(ss, oracle_mod, ctx, xr, kwr, after_error)
        if after_error is not None:              # the last case was rejected: the context must still work
            x = np.random.default_rng(0).normal(0, 0.05, (300, 3)).astype(np.float32)
            kw = dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.5, subdomain_grid_auto_disable=False)
            assert_matches_oracle(oracle_mod, ss.reconstruct_surface(x, with_debug=True, context=ctx, **kw), oracle_mod.reconstruct(x, **kw),
                                  kw, f"first case after the rejected {after_error}")
    finally:
        ctx.close()
    return ran


# ------------------------------------------------------------------ 2. one scripted history on one context ----
def check_context_history(ss, oracle_mod, big, big_kw):
    """A sequence of frames and stand-alone calls on one context with the default switches (level-set variant 2, warp-per-brick
    marching cubes: the paths without zero-fill).  `big` must give a mesh larger than the 65 536 vertices every context starts with:
    run with one tile per batch, the surface buffers then grow while they hold the earlier batches' vertices."""
    from test_zz_gpu_postprocess import _oracle_pipeline, compare_point_fields
    from splashsurf_b200 import synthetic as syn
    ctx = ss.Context()
    tail_kw = dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.6, subdomain_num_cubes_per_dim=16, subdomain_grid_auto_disable=False)
    tail = syn.splash((9, 8, 9), 3, 0.025, 912)

    def frame(name, x, kw, batch=0):
        ctx.set_tile_batch(batch)
        g = ss.reconstruct_surface(x, with_debug=True, context=ctx, **kw)
        assert_matches_oracle(oracle_mod, g, oracle_mod.reconstruct(x, **kw), kw, f"history frame {name!r}")
        return g

    def stand_alone(name, call, reduce):
        got = reduce(call(ctx))
        want = on_fresh_context(ss, None, lambda c: reduce(call(c)))
        assert_raw_equal(got, want, f"history: {name} on the reused vs a fresh context")
        frame(f"after {name}", tail, tail_kw)

    try:
        frame("tiny first frame", np.float32([[0, 0, 0], [0.01, 0.02, 0.0]]), dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.5))
        first = frame("big, one tile per batch", big, big_kw, batch=1)
        assert first.mesh.nvertices > 1 << 16 and first.mesh.ncells > 1 << 17, (first.mesh.nvertices, first.mesh.ncells)
        frame("big, all tiles in one batch", big, big_kw)
        g = frame("two far-apart particles", np.float32([[0, 0, 0], [3, 3, 3]]), dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.5,
                                                                                   subdomain_grid_auto_disable=False))
        assert g.mesh.nvertices == 252
        g = frame("empty cloud", np.zeros((0, 3), np.float32), dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.5,
                                                                   subdomain_grid_auto_disable=False))
        assert g.mesh.nvertices == 0 and g.mesh.ncells == 0
        frame("global path", syn.splash((9, 9, 9), 2, 0.025, 913), dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.75, subdomain_grid=False))
        g = frame("particle AABB", syn.splash((10, 10, 10), 2, 0.025, 914), dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.6,
                                                                                 aabb_min=[-0.05, -0.05, -0.05], aabb_max=[0.4, 1.2, 0.45]))
        assert not g.particle_inside_aabb.all()
        frame("tiny frame (small capacity hints)", np.float32([[0.5, 0.5, 0.5]]), dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.5))
        again = frame("big again, one tile per batch", big, big_kw, batch=1)
        assert_raw_equal(_raw(again), _raw(first), "history: the same frame twice with other frames in between")

        # the pipeline with SPH normals and smoothing weights, against oracle/postprocess.py
        px = syn.splash((12, 10, 11), 3, 0.025, 915)
        pkw = dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.75, subdomain_num_cubes_per_dim=32, subdomain_grid_auto_disable=False)
        post = dict(mesh_smoothing_weights=True, mesh_smoothing_weights_normalization=13.0, mesh_smoothing_iters=3, compute_normals=True,
                    sph_normals=True, normals_smoothing_iters=2)
        o, ref = _oracle_pipeline(oracle_mod, px, pkw, post)
        run = lambda c: ss.reconstruction_pipeline(px, **pkw, **post, output_mesh_smoothing_weights=True, with_debug=True, context=c)  # noqa: E731
        m, rec = run(ctx)
        got = dict(m.point_attributes, vertices=m.mesh.vertices)
        compare_point_fields(got, rec.vertex_edge_keys, {k: v for k, v in ref.items() if k in got}, o["vertex_keys"], 5e-5)
        m2, _ = on_fresh_context(ss, None, run)
        assert_raw_equal(dict(m.point_attributes, vertices=m.mesh.vertices, triangles=m.mesh.triangles),
                         dict(m2.point_attributes, vertices=m2.mesh.vertices, triangles=m2.mesh.triangles), "history: pipeline on the reused vs a fresh context")
        frame("after the pipeline", tail, tail_kw)

        # stand-alone entries on the same context, each followed by a reconstruction
        rng = np.random.default_rng(916)
        sx = syn.splash((8, 8, 8), 2, 0.025, 917)
        rho = rng.uniform(800, 1200, len(sx)).astype(np.float32)
        pts = np.concatenate([sx[::7] + rng.normal(0, 0.02, (len(sx[::7]), 3)).astype(np.float32), np.float32([[9, 9, 9]])])
        q = rng.normal(size=(len(sx), 3)).astype(np.float32)

        def interpolate(c):
            it = ss.SphInterpolator(sx, rho, float(oracle_mod.sph_rest_mass(0.025)), 0.1, context=c)
            try:
                return {"quantity": it.interpolate_quantity(q, pts), "scalar_corrected": it.interpolate_quantity(rho, pts, first_order_correction=True),
                        "normals": it.interpolate_normals(pts)}
            finally:
                it.close()
        stand_alone("SphInterpolator", interpolate, lambda d: d)

        def search(c):
            dom = ss.Aabb3d.from_min_max(sx.min(axis=0) - 0.1, sx.max(axis=0) + 0.1)
            return ss.neighborhood_search_spatial_hashing_parallel(sx, dom, 0.1, context=c)
        stand_alone("neighbourhood search", search, lambda nl: {"offsets": nl.offsets, "indices": nl.indices})

        ii = np.stack(np.meshgrid(*[np.arange(n, dtype=np.float32) for n in (70, 40, 90)], indexing="ij"), -1)
        sdf = np.float32(30.0) - np.linalg.norm(ii - np.float32([35, 20, 45]), axis=-1).astype(np.float32)   # inside is positive
        stand_alone("marching cubes", lambda c: ss.marching_cubes(sdf, iso_surface_threshold=0.25, cube_size=0.1, translation=[1, 2, 3], context=c),
                    lambda mesh: {"vertices": mesh.vertices, "triangles": mesh.triangles})
    finally:
        ctx.close()


# ------------------------------------------------------------------ 3. the slab partition entries on one device ----
def check_slab_partition_one_device(ss, oracle_mod, device):
    """Every per-rank library call of a 2- and 3-rank slab partition, both protocols and a rank that owns nothing, run one after
    another in this process (tests/test_emulated_pipeline.py:_virtual_ranks); the welded mesh equals the single-device oracle's."""
    from splashsurf_b200 import synthetic as syn
    from test_emulated_pipeline import _virtual_ranks
    kw = dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.75, subdomain_num_cubes_per_dim=16, subdomain_grid_auto_disable=False)
    x = syn.dam_break((10, 6, 6), (14, 2, 6), 0.025, 401)
    o = oracle_mod.reconstruct(x, **kw)
    nlayers = (int(o["grid"]["ncells"][0]) + 15) // 16
    for world, cuts in ((2, None), (3, None), (3, [0, nlayers // 2, nlayers // 2, nlayers])):
        for use_callback in (False, True):
            v, t, keys, plan, nrecv = _virtual_ranks(ss, oracle_mod, x, kw, world, use_callback, cuts, device=device)
            assert all(plan.cuts[r] <= plan.cuts[r + 1] for r in range(world)), plan
            if cuts is not None:
                assert nrecv[1] == 0
            m = oracle_mod.mesh_parity(v, t, keys, o["vertices"], o["triangles"], o["vertex_keys"], 16)
            assert m["keys_equal"] and m["triangles_equal"] and m["n_not_bitexact"] == 0, (world, cuts, use_callback, m)


def _big_splash():
    from splashsurf_b200 import synthetic as syn
    x = syn.splash((38, 36, 37), 6, 0.025, 911)
    assert len(x) >= 50_000
    return x


BIG_KW = dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.5)


@pytest.mark.gpu
def test_cuda_poisoned_pool_differential(ss, oracle_mod):
    assert check_poisoned_pool(ss, oracle_mod, pick_seeds(7_000_000, 30, 10)) >= 35


@pytest.mark.gpu
def test_cuda_context_history(ss, oracle_mod):
    check_context_history(ss, oracle_mod, _big_splash(), BIG_KW)


@pytest.mark.gpu
def test_cuda_slab_partition_on_one_device(ss, oracle_mod):
    # SS_TEST_EMULATED (conftest.py): the GPU-marked tests on the CPU executor, whose device memory is host memory
    check_slab_partition_one_device(ss, oracle_mod, "cpu" if os.environ.get("SS_TEST_EMULATED") else "cuda")


# ------------------------------------------------------------------ 4. the same checks on the CPU executor (non-guard build) ----
@pytest.fixture(scope="module")
def emu_pooled():
    """splashsurf_b200 bound to the non-guard executor build for this module (its buffers keep their contents between calls)."""
    import splashsurf_b200 as ss
    from test_emulated_pipeline import build_emulated_library
    guard = os.environ.pop("SS_EMUL_GUARD", None)
    try:
        so = build_emulated_library()
    finally:
        if guard is not None:
            os.environ["SS_EMUL_GUARD"] = guard
    saved_lib, saved_ctx = ss._LIB, dict(ss._DEFAULT_CTX)
    ss._DEFAULT_CTX.clear()
    ss._LIB = ss._bind(C.CDLL(so))
    try:
        yield ss
    finally:
        for ctx in ss._DEFAULT_CTX.values():
            ctx.close()
        ss._DEFAULT_CTX.clear()
        ss._DEFAULT_CTX.update(saved_ctx)
        ss._LIB = saved_lib


def test_emulated_poisoned_pool_differential(emu_pooled, oracle_mod):
    assert check_poisoned_pool(emu_pooled, oracle_mod, pick_seeds(7_000_000, 6, 2), max_points=1.5e6, reject_every=3) >= 6


def test_emulated_context_history(emu_pooled, oracle_mod):
    from splashsurf_b200 import synthetic as syn
    check_context_history(emu_pooled, oracle_mod, syn.jittered_cube(16, 0.025, 918), dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.3))
